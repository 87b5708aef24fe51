"""CPU tests of the host side that mirrors the reference interface: BaseAgent surface, torch.optim-layout optimizer state,
Timings, the ActorNet stand-in vs the reference's AtariNet (its outputs recorded in tests/golden/reference_cases.npz by
oracle/make_golden.py), the reference actor calling convention in ImpalaTrainer.get_action, rnn-state buffers."""
import os
import threading

import numpy as np
import pytest
import torch

from oracle import make_golden as MG
from oracle import ref_learner as R
from scalerl_b200.learner import (B200ImpalaLearner, ImpalaHParams, LSTM_PARAM_NAMES, PARAM_NAMES, from_torch_optimizer_state,
                                  param_shapes, reference_param_order, to_torch_optimizer_state)
from scalerl_b200.algorithms.base import BaseAgent
from scalerl_b200.algorithms.impala.impala_atari import ImpalaArguments, ImpalaTrainer
from scalerl_b200.algorithms.utils.atari_model import ActorNet, SyntheticAtariEnv
from scalerl_b200.utils.profile import Timings
from tests.conftest import GOLDEN


def _golden():
    return np.load(os.path.join(GOLDEN, 'reference_cases.npz'))


def _ref_atarinet():
    """the reference's own AtariNet class (oracle/_ref, built by oracle/make_ref.py where the reference sources are present)"""
    return R._load('atari_model').AtariNet


class _Shaped(torch.nn.Module):
    """parameters with AtariNet's names / shapes / registration order (conv1, conv2, conv3, fc, [rnn_layer], policy, baseline)"""

    def __init__(self, A, use_lstm):
        super().__init__()
        shapes = param_shapes(A, use_lstm)
        for n in reference_param_order(use_lstm):
            self.register_parameter(n.replace('.', '__'), torch.nn.Parameter(torch.randn(shapes[n])))


def test_learner_is_a_base_agent():
    assert issubclass(B200ImpalaLearner, BaseAgent)
    for m in ('get_action', 'predict', 'get_value', 'learn', 'get_weights', 'set_weights', 'save_checkpoint', 'load_checkpoint', 'name'):
        assert callable(getattr(B200ImpalaLearner, m)), m                    # algorithms/base.py:23-124
    for m in ('get_action', 'predict', 'get_value', 'learn', 'get_weights', 'set_weights', 'save_checkpoint', 'load_checkpoint'):
        assert getattr(B200ImpalaLearner, m) is not getattr(BaseAgent, m), f'{m} must be overridden'
    with pytest.raises(RuntimeError):          # no CPU fallback: constructing without CUDA fails loudly
        if torch.cuda.is_available():
            raise RuntimeError('skip')
        B200ImpalaLearner(ImpalaHParams())


@pytest.mark.parametrize('optimizer,use_lstm', [('rmsprop', False), ('adam', False), ('rmsprop', True)])
def test_optimizer_state_is_torch_layout(optimizer, use_lstm):
    """what the learner saves is what torch.optim.<Opt>(AtariNet.parameters()).state_dict() would hold: the installed torch
    loads it, steps with it, and the way back recovers step count and tensors (impala_atari.py:99-105,506-511)"""
    A = 6
    hp = ImpalaHParams(num_actions=A, optimizer=optimizer, use_lstm=use_lstm)
    names = PARAM_NAMES + (LSTM_PARAM_NAMES if use_lstm else ())
    shapes = param_shapes(A, use_lstm)
    g = torch.Generator().manual_seed(1)
    kinds = ('square_avg',) if optimizer == 'rmsprop' else ('exp_avg', 'exp_avg_sq')
    tensors = {k: {n: torch.rand(shapes[n], generator=g) for n in names} for k in kinds}
    sd = to_torch_optimizer_state(hp, tensors, step=7)
    net = _Shaped(A, use_lstm)
    opt = (torch.optim.RMSprop(net.parameters(), lr=hp.learning_rate, momentum=0.0, eps=hp.epsilon, alpha=hp.alpha) if optimizer == 'rmsprop'
           else torch.optim.Adam(net.parameters(), lr=hp.learning_rate))
    opt.load_state_dict(sd)                                   # torch accepts the layout
    order = reference_param_order(use_lstm)
    for i, p in enumerate(net.parameters()):
        st = opt.state[p]
        assert float(st['step']) == 7.0
        for k in kinds:
            assert torch.equal(st[k], tensors[k][order[i]]), (k, order[i])
    for p in net.parameters():
        p.grad = torch.ones_like(p)
    opt.step()                                                # ... and can continue training from it
    step, back = from_torch_optimizer_state(opt.state_dict(), use_lstm)
    assert step == 8 and set(back) == set(kinds) and set(back[kinds[0]]) == set(names)
    # a fresh optimizer has no state: step 0
    assert from_torch_optimizer_state(to_torch_optimizer_state(hp, tensors, step=0), use_lstm) == (0, {})
    # round 1's own layout is still readable; unknown layouts fail loudly
    step, back = from_torch_optimizer_state({'step': 3, 'state': {'square_avg': tensors.get('square_avg', {})}}, use_lstm)
    assert step == 3
    with pytest.raises(ValueError):
        from_torch_optimizer_state({'state': {0: {'step': torch.tensor(1.), 'momentum_buffer': torch.zeros(1)}}, 'param_groups': []}, False)


def test_reference_param_order_is_atarinet_parameters_order():
    g = _golden()
    for use_lstm in (False, True):
        assert list(g[f'param_order_lstm{int(use_lstm)}']) == list(reference_param_order(use_lstm))


def test_timings_matches_reference_statistics():
    tm = Timings()
    xs = {'a': [], 'b': []}
    import time
    for i in range(6):
        tm.reset()
        time.sleep(0.001 * (1 + i % 3)); t0 = tm.last_time; tm.time('a'); xs['a'].append(tm.last_time - t0)
        time.sleep(0.0005); t0 = tm.last_time; tm.time('b'); xs['b'].append(tm.last_time - t0)
    for k, v in xs.items():
        mean = sum(v) / len(v)
        var = sum((x - mean) ** 2 for x in v) / len(v)
        assert abs(tm.means()[k] - mean) < 1e-12 and abs(tm.vars()[k] - var) < 1e-12
        assert abs(tm.stds()[k] - var ** 0.5) < 1e-9
    s = tm.summary('Batch and learn: ')
    assert s.startswith('Batch and learn: ') and 'Total:' in s and 'a:' in s and 'b:' in s
    # same numbers as the reference's own class fed the same samples (scalerl/utils/profile.py, recorded by oracle/make_golden.py)
    mine = Timings()
    import timeit
    real = timeit.default_timer
    try:
        for x in (0.5, 0.25, 1.0, 0.75):
            mine.last_time = 0.0
            timeit.default_timer = lambda x=x: x
            mine.time('k')
    finally:
        timeit.default_timer = real
    ref_mean, ref_var = _golden()['timings_mean_var']
    assert abs(ref_mean - mine.means()['k']) < 1e-12 and abs(ref_var - mine.vars()['k']) < 1e-12


@pytest.mark.parametrize('use_lstm', [False, True])
def test_actornet_equals_reference_atarinet(use_lstm):
    """same state_dict keys/shapes, same outputs and next state as the reference model on the actor's one-step calls"""
    g = _golden()
    p = f'actor_lstm{int(use_lstm)}_'
    A = 6
    mine = ActorNet((4, 84, 84), A, use_lstm=use_lstm)
    sd = mine.state_dict()
    assert list(g[p + 'keys']) == list(sd) and all(tuple(g[p + 'shape_' + k]) == tuple(sd[k].shape) for k in sd)
    mine.load_state_dict(MG.actor_weights(A, use_lstm))
    torch.manual_seed(0)                       # SyntheticAtariEnv mixes torch.initial_seed() into its seed
    env = SyntheticAtariEnv((4, 84, 84), A, seed=3)
    out = env.reset()
    s_mine = mine.initial_hidden_state(1)
    assert [tuple(s.shape) for s in s_mine] == [tuple(s) for s in g[p + 'state_shapes']]
    mine.eval()
    for t in range(4):
        o_mine, s_mine = mine(out, s_mine)
        q = f'{p}t{t}_'
        assert torch.allclose(torch.from_numpy(g[q + 'logits']), o_mine['policy_logits'], atol=1e-5)
        assert torch.allclose(torch.from_numpy(g[q + 'baseline']), o_mine['baseline'], atol=1e-5)
        assert torch.equal(torch.from_numpy(g[q + 'action']), o_mine['action'])
        assert len(s_mine) == len(g[p + 'state_shapes'])
        for i, b in enumerate(s_mine):
            assert torch.allclose(torch.from_numpy(g[f'{q}state{i}']), b, atol=1e-5)
        out = env.step(o_mine['action'])
        if t == 1:
            out['done'] = torch.ones(1, 1, dtype=torch.bool)          # exercise the state reset (atari_model.py:114-116)


@pytest.mark.parametrize('which', ['actornet', 'reference', 'reference_lstm'])
def test_get_action_fills_slots_with_the_reference_actor_convention(which, tmp_path):
    """ImpalaTrainer.get_action drives actor_model(env_output, agent_state) -> (outputs, state) (impala_atari.py:177-197)
    -- with the stand-in ActorNet and with the reference's own AtariNet, unchanged -- and writes rollouts + initial LSTM
    states into the shared slots"""
    if which != 'actornet' and not R.available():
        pytest.skip('oracle/_ref not built (python oracle/make_ref.py, needs the reference sources)')
    use_lstm = which == 'reference_lstm'
    a = ImpalaArguments(num_actors=1, batch_size=2, rollout_length=3, num_buffers=3, use_lstm=use_lstm, output_dir=str(tmp_path))
    fn = None
    if which != 'actornet':
        AtariNet = _ref_atarinet()
        fn = lambda: AtariNet((4, 84, 84), a.num_actions, use_lstm=use_lstm)
    t = ImpalaTrainer(a, actor_model_fn=fn)
    assert len(t.rnn_state_buffers) == 3
    if use_lstm:
        h, c = t.rnn_state_buffers[1]
        assert tuple(h.shape) == (2, 1, 513 + a.num_actions) and h.is_shared() and c.is_shared()   # impala_atari.py:108-120
    else:
        assert t.rnn_state_buffers[0] == tuple()
    import queue
    free_q, full_q = queue.SimpleQueue(), queue.SimpleQueue()
    for m in (2, 0):
        free_q.put(m)
    free_q.put(None)
    th = threading.Thread(target=t.get_action, args=(0, free_q, full_q, t.actor_model, t.buffers, t.rnn_state_buffers))
    th.start(); th.join(timeout=120)
    assert not th.is_alive()
    assert [full_q.get(), full_q.get()] == [2, 0]
    for m in (2, 0):
        assert int(t.buffers['obs'][m].sum()) > 0 and torch.isfinite(t.buffers['policy_logits'][m]).all()
        assert int(t.buffers['episode_step'][m][-1]) > 0
    assert int(t.buffers['obs'][1].sum()) == 0                       # untouched slot
    if use_lstm:                                                     # second rollout starts from a non-zero carried state
        assert float(t.rnn_state_buffers[0][0].abs().sum()) > 0


def test_trainer_validation_and_lstm_accepted(tmp_path):
    t = ImpalaTrainer(ImpalaArguments(use_lstm=True, num_actors=1, batch_size=2, output_dir=str(tmp_path)))
    assert t.hparams().use_lstm and t._rnn_block is not None and tuple(t._rnn_block.shape) == (2, 2, 2, 1, 519)
    assert int(t.weights_version[0]) == 0 and t.weights_version.is_shared()


@pytest.mark.parametrize('use_lstm', [False, True])
def test_get_action_batched_matches_the_slot_protocol(use_lstm, tmp_path):
    """one actor process, N environments, one model call per step: every environment fills its own slot (same rows / keys /
    initial LSTM state as get_action writes for a single environment)"""
    a = ImpalaArguments(num_actors=1, batch_size=2, rollout_length=3, num_buffers=4, use_lstm=use_lstm, output_dir=str(tmp_path))
    seeds = iter(range(100))
    t = ImpalaTrainer(a, env_fn=lambda: SyntheticAtariEnv((4, 84, 84), a.num_actions, seed=next(seeds)))
    import queue
    free_q, full_q = queue.SimpleQueue(), queue.SimpleQueue()
    for m in (3, 1, 0):
        free_q.put(m)
    for _ in range(3):
        free_q.put(None)
    th = threading.Thread(target=t.get_action_batched, args=(0, free_q, full_q, t.actor_model, t.buffers, t.rnn_state_buffers, 3))
    th.start(); th.join(timeout=120)
    assert not th.is_alive()
    assert sorted(full_q.get() for _ in range(3)) == [0, 1, 3]
    for m in (0, 1, 3):
        assert int(t.buffers['obs'][m].sum()) > 0 and torch.isfinite(t.buffers['policy_logits'][m]).all()
        assert [int(v) for v in t.buffers['episode_step'][m][1:]] == [1, 2, 3]
        # the stored action of row t+1 is the agent's action that produced it (key collision kept as the reference behaves)
        assert int(t.buffers['action'][m].max()) < a.num_actions
    assert int(t.buffers['obs'][2].sum()) == 0
    # distinct environments wrote distinct frames
    assert not torch.equal(t.buffers['obs'][0], t.buffers['obs'][1])
