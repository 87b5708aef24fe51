"""The reference's learner step (oracle/_ref: the reference's own vtrace / loss_fn / atari_model modules under the restated
learn() statements, what bench.py's reference arm runs) == the oracle's learn_step, whole step: losses, grad norm, post-step
weights.  The reference learner's results are stored in tests/golden/reference_cases.npz (oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import impala_oracle as O
from oracle import make_golden as MG
from oracle import ref_learner as R
from tests.conftest import GOLDEN
from tests.helpers import strided_sample


@pytest.mark.parametrize('T,B,A,clip', MG.LEARNER_CASES)
def test_reference_learner_step_equals_oracle(T, B, A, clip):
    torch.set_num_threads(4)
    g = np.load(os.path.join(GOLDEN, 'reference_cases.npz'))
    params, batch = MG.learner_inputs(T, B, A)
    p0 = {k: v.clone() for k, v in params.items()}
    opt = O.new_opt_state(params)
    for step in range(2):
        p = f'learner_t{T}b{B}a{A}_{clip}_s{step}_'
        st = dict(zip(('pg_loss', 'baseline_loss', 'entropy_loss', 'total_loss', 'grad_norm'), (float(x) for x in g[p + 'stats'])))
        ref = O.learn_step(p0, opt, batch, dict(reward_clipping=clip), use_autograd=True)
        for k in ('pg_loss', 'baseline_loss', 'entropy_loss', 'total_loss'):
            assert abs(st[k] - ref[k]) <= 1e-5 * max(1.0, abs(ref[k])), (step, k)
        assert abs(st['grad_norm'] - ref['grad_norm']) <= 1e-4 * ref['grad_norm']
        for k in O.PARAM_ORDER:
            assert float((torch.from_numpy(g[p + 'param_' + k]) - strided_sample(p0[k].reshape(-1))).abs().max()) <= 2e-6, (step, k)


@pytest.mark.skipif(not R.available(), reason='oracle/_ref not built (python oracle/make_ref.py, needs the reference sources)')
def test_bench_reference_arm_runs_the_reference_modules():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('bench_mod2', os.path.join(root, 'bench.py'))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    cpu = b._CpuLearner(3, 2, 6)
    assert cpu.kind == 'reference'
    st = cpu.step()
    assert 'total_loss' in st
    assert b.workload_config(20, 32, 6, 1) == b.workload_config(20, 32, 6, 1)
