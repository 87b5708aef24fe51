"""Oracle vs the REFERENCE's own modules on randomised inputs: the reference's outputs are stored in
tests/golden/reference_cases.npz, recorded by oracle/make_golden.py from scalerl/algorithms/impala/vtrace.py, loss_fn.py,
scalerl/algorithms/utils/atari_model.py and scalerl/data/segment_tree.py.  The inputs are rebuilt from the same seeds by the
input functions of oracle/make_golden.py."""
import os

import numpy as np
import pytest
import torch

from oracle import impala_oracle as O
from oracle import make_golden as MG
from tests.conftest import GOLDEN


@pytest.fixture(scope='module')
def ref():
    return np.load(os.path.join(GOLDEN, 'reference_cases.npz'))


@pytest.mark.parametrize('seed', range(12))
def test_vtrace_from_logits_random_shapes(ref, seed):
    """vtrace.py:43-172 on random (T, B, A), with terminal steps and every clip-threshold combination incl. None"""
    a = MG.vtrace_random_inputs(seed)
    r = {k: torch.from_numpy(ref[f'vtrace_s{seed}_{k}']) for k in ('vs', 'pg', 'log_rhos', 'balp', 'talp')}
    cr, cp = a['clip_rho_threshold'], a['clip_pg_rho_threshold']
    discounts, rewards, values, boot = a['discounts'], a['rewards'], a['values'], a['bootstrap_value']
    vs, pg, lr, balp, talp = O.vtrace_from_logits(a['behavior_policy_logits'], a['target_policy_logits'], a['actions'], discounts, rewards,
                                                  values, boot, cr, cp)
    assert torch.allclose(vs, r['vs'], rtol=1e-5, atol=1e-5) and torch.allclose(pg, r['pg'], rtol=1e-5, atol=1e-5)
    assert torch.allclose(lr, r['log_rhos'], atol=1e-6) and torch.allclose(balp, r['balp'], atol=1e-6)
    assert torch.allclose(talp, r['talp'], atol=1e-6)
    # the float64 scalar witness agrees with both
    vs64, pg64 = O.vtrace_from_importance_weights_np64(lr.numpy(), discounts.numpy(), rewards.numpy(), values.numpy(), boot.numpy(), cr, cp)
    assert np.allclose(vs64, r['vs'].numpy(), rtol=1e-4, atol=1e-4) and np.allclose(pg64, r['pg'].numpy(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('seed', range(6))
def test_losses_and_head_gradients_random(ref, seed):
    """loss_fn.py:5-23 with the weights of impala_atari.py:320-330; the oracle's closed-form head gradients equal autograd
    through the reference's loss functions"""
    logits, values, actions, vs, adv, bc, ec = MG.loss_random_inputs(seed)
    pg, bl, en = (float(x) for x in ref[f'loss_s{seed}_losses'])
    o_pg, o_bl, o_en = O.impala_losses(logits, actions, values, vs, adv, bc, ec)
    assert abs(float(o_pg) - pg) <= 1e-4 * max(1, abs(pg)) and abs(float(o_bl) - bl) <= 1e-4 * max(1, abs(bl))
    assert abs(float(o_en) - en) <= 1e-5 * max(1, abs(en))
    dl, dv = O.head_grads(logits, actions, values, vs, adv, bc, ec)
    assert torch.allclose(dl, torch.from_numpy(ref[f'loss_s{seed}_dlogits']), rtol=1e-4, atol=1e-6)
    assert torch.allclose(dv, torch.from_numpy(ref[f'loss_s{seed}_dvalues']), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize('A,seed', [(6, 0), (18, 1), (3, 2)])
def test_atarinet_forward_random_weights(ref, A, seed):
    """atari_model.py:77-143 (no LSTM): the oracle's functional forward == AtariNet.forward with the same state_dict,
    greedy actions excluded (the reference samples with torch.multinomial in training mode)"""
    params = O.init_params(A, seed=seed)
    T, B = 3, 2
    batch = O.synthetic_batch(T, B, A, seed=seed)
    lg, bs = O.atari_forward(params, batch['obs'], batch['reward'], batch['action'])
    assert torch.allclose(lg.view(T + 1, B, A), torch.from_numpy(ref[f'atari_a{A}_s{seed}_logits']), rtol=1e-4, atol=1e-5)
    assert torch.allclose(bs.view(T + 1, B), torch.from_numpy(ref[f'atari_a{A}_s{seed}_baseline']), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('seed', range(6))
def test_per_trees_random_against_reference_segment_trees(ref, seed):
    """scalerl/data/segment_tree.py driven by the statements of PrioritizedReplayBuffer (replay_buffer.py:318-381) vs the
    PER oracle: random capacities (incl. wrap-around of the ring pointer), duplicate update indices, several rounds"""
    from oracle.per_oracle import PerOracle
    mem, alpha, beta, rounds = MG.per_random_inputs(seed)
    o = PerOracle(mem, alpha)
    max_p, size = 1.0, 0
    for rnd, (nadd, idx, pr, u) in enumerate(rounds):
        o.add(nadd)
        size = min(size + nadd, mem)
        o.update_priorities(idx, pr)
        max_p = max(max_p, float(pr.max()))
        got, got_w = o.sample(u, beta)
        p = f'per_s{seed}_r{rnd}_'
        assert np.array_equal(got, ref[p + 'idx']), (seed, rnd)
        assert np.array_equal(got_w, ref[p + 'w'])
        assert o.size == size and o.max_priority == max_p
        assert o.sum_tree.operate() == ref[p + 'sum'][0] and o.min_tree.operate() == ref[p + 'min'][0]


@pytest.mark.parametrize('A,seed', [(6, 0), (3, 1)])
def test_atarinet_lstm_forward_random(ref, A, seed):
    """use_lstm=True (atari_model.py:52-55,109-120): the oracle's step-wise 2-layer LSTM with done-resets and a random
    initial state vs the reference module holding the same weights"""
    params, lp, batch, state = MG.lstm_random_inputs(A, seed)
    T, B = batch['reward'].shape[0] - 1, batch['reward'].shape[1]
    with torch.no_grad():
        lg, bs, os_ = O.atari_forward_lstm(params, lp, batch['obs'], batch['reward'], batch['action'], batch['done'], state)
    r = {k: torch.from_numpy(ref[f'lstm_a{A}_s{seed}_{k}']) for k in ('logits', 'baseline', 'h', 'c')}
    assert torch.allclose(lg.view(T + 1, B, A), r['logits'], rtol=1e-4, atol=1e-5)
    assert torch.allclose(bs.view(T + 1, B), r['baseline'], rtol=1e-4, atol=1e-5)
    assert torch.allclose(os_[0], r['h'], rtol=1e-4, atol=1e-5) and torch.allclose(os_[1], r['c'], rtol=1e-4, atol=1e-5)
