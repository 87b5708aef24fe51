"""GPU parity tests: every kernel of the hot path, through the C ABI, against the CPU oracle on the same
seeded inputs, against the reference-generated golden fixtures, and size-independent properties at
BASELINE.json's full sizes.  Tolerances:
  * V-trace / losses / head gradients / optimizer (fp32 kernels): normalised max error <= 1e-4 (north_star)
    -- measured errors are ~1e-6.
  * encoder (bf16 tensor-core operands, fp32 accumulation) vs the bf16-emulating oracle: rel-L2 <= 5e-3
    (summation order + rare rounding-boundary / ReLU-mask flips); vs the fp32 reference goldens: rel-L2 <= 0.12
    for gradients at the tiny golden batch (mask flips dominate, see tests/test_oracle_golden.py), 2e-2 for logits.
"""
import os

import numpy as np
import pytest
import torch

from oracle import impala_oracle as O
from tests.conftest import GOLDEN
from tests.helpers import assert_close, rel_l2, strided_sample

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops():
    from scalerl_b200 import ops as _ops
    return _ops


def dev(t):
    return t.cuda()


# ------------------------------------------------------------------------------------------------
# tcgen05 mainloop in isolation
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('simt', [True, False])
@pytest.mark.parametrize('M,N,K', [(128, 64, 64), (128, 64, 256), (300, 128, 576), (1000, 192, 3136)])
def test_gemm_kmajor(ops, M, N, K, simt):
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g).bfloat16()
    b = torch.randn(N, K, generator=g).bfloat16()
    ref = a.float() @ b.float().t()
    d = ops.test_gemm(dev(a), dev(b), mn_major=False, simt=simt)
    assert_close(d, ref, 1e-5, f'gemm_k {M}x{N}x{K} simt={simt}')


@pytest.mark.parametrize('simt', [True, False])
@pytest.mark.parametrize('M,N,K', [(128, 64, 64), (128, 64, 100), (256, 128, 1000), (512, 192, 640)])
def test_gemm_mnmajor(ops, M, N, K, simt):
    g = torch.Generator().manual_seed(M + N + K + 1)
    at = torch.randn(K, M, generator=g).bfloat16()
    bt = torch.randn(K, N, generator=g).bfloat16()
    ref = at.float().t() @ bt.float()
    d = ops.test_gemm(dev(at), dev(bt), mn_major=True, simt=simt)
    assert_close(d, ref, 1e-5, f'gemm_mn {M}x{N}x{K} simt={simt}')


# ------------------------------------------------------------------------------------------------
# V-trace
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('variant', [0, 1])
def test_vtrace_goldens(ops, variant):
    z = np.load(os.path.join(GOLDEN, 'vtrace_cases.npz'))
    n = len([k for k in z.files if k.endswith('_meta')])
    for i in range(n):
        T, B, cr, cp, _ = z[f'c{i}_meta']
        cr = None if cr < 0 else float(cr)
        cp = None if cp < 0 else float(cp)
        args = [dev(torch.from_numpy(z[f'c{i}_{k}'])) for k in ('log_rhos', 'discounts', 'rewards', 'values', 'boot')]
        r = ops.from_importance_weights(*args, clip_rho_threshold=cr, clip_pg_rho_threshold=cp, variant=variant)
        assert_close(r.vs, z[f'c{i}_vs'], 1e-4, f'vs c{i} v{variant}')
        assert_close(r.pg_advantages, z[f'c{i}_pg'], 1e-4, f'pg c{i} v{variant}')
        assert torch.allclose(r.vs.cpu(), torch.from_numpy(z[f'c{i}_vs']), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('variant', [0, 1])
@pytest.mark.parametrize('T,B', [(20, 32), (20, 512), (100, 128), (20, 1), (1, 7), (20, 4099), (37, 33)])
def test_vtrace_vs_oracle(ops, T, B, variant):
    rng = np.random.RandomState(T * 1000 + B)
    log_rhos = torch.from_numpy((rng.randn(T, B) * 0.8).astype(np.float32))
    discounts = torch.from_numpy(((rng.rand(T, B) > 0.05) * 0.99).astype(np.float32))
    rewards = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    values = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    boot = torch.from_numpy(rng.randn(B).astype(np.float32))
    vs, pg = O.vtrace_from_importance_weights(log_rhos, discounts, rewards, values, boot)
    r = ops.from_importance_weights(dev(log_rhos), dev(discounts), dev(rewards), dev(values), dev(boot), variant=variant)
    assert_close(r.vs, vs, 1e-4, 'vs')
    assert_close(r.pg_advantages, pg, 1e-4, 'pg')
    assert torch.allclose(r.vs.cpu(), vs, rtol=1e-4, atol=1e-5) and torch.allclose(r.pg_advantages.cpu(), pg, rtol=1e-4, atol=1e-5)


def test_vtrace_edge_cases(ops):
    # empty inputs are a no-op, like the reference's empty loop
    e = torch.empty(0, 5, device='cuda')
    r = ops.from_importance_weights(e, e, e, e, torch.zeros(5, device='cuda'))
    assert r.vs.shape == (0, 5)
    # known answer: all-done, on-policy, r=1, V=0 -> vs = pg = 1
    T, B = 9, 130
    z = torch.zeros(T, B, device='cuda')
    for variant in (0, 1):
        r = ops.from_importance_weights(z, z, torch.ones_like(z), z, torch.zeros(B, device='cuda'), variant=variant)
        assert torch.equal(r.vs, torch.ones_like(z)) and torch.equal(r.pg_advantages, torch.ones_like(z))
    with pytest.raises(ValueError):
        ops.from_importance_weights(z, z[:-1], z, z, torch.zeros(B, device='cuda'))
    with pytest.raises(ValueError):
        ops.from_importance_weights(z.cpu(), z.cpu(), z.cpu(), z.cpu(), torch.zeros(B))


def test_vtrace_full_size_properties(ops):
    """T=20, B=2^20 (the bandwidth-bound size): the two kernels agree; columns are independent (permutation
    equivariance); with discounts == 0 the recursion collapses to the closed form vs = V + min(rho,1)(r - V)."""
    T, B = 20, 1 << 20
    g = torch.Generator(device='cuda').manual_seed(0)
    lr = torch.randn(T, B, device='cuda', generator=g) * 0.5
    disc = (torch.rand(T, B, device='cuda', generator=g) > 0.02).float() * 0.99
    r = torch.randn(T, B, device='cuda', generator=g)
    v = torch.randn(T, B, device='cuda', generator=g)
    boot = torch.randn(B, device='cuda', generator=g)
    a = ops.from_importance_weights(lr, disc, r, v, boot, variant=0)
    b = ops.from_importance_weights(lr, disc, r, v, boot, variant=1)
    assert_close(b.vs, a.vs, 1e-5, 'scan vs seq')
    assert_close(b.pg_advantages, a.pg_advantages, 1e-5, 'scan vs seq pg')
    perm = torch.randperm(B, device='cuda', generator=g)
    c = ops.from_importance_weights(lr[:, perm].contiguous(), disc[:, perm].contiguous(), r[:, perm].contiguous(),
                                    v[:, perm].contiguous(), boot[perm].contiguous(), variant=0)
    assert torch.equal(c.vs, a.vs[:, perm])
    d = ops.from_importance_weights(lr, torch.zeros_like(disc), r, v, boot, variant=0)
    closed = v + torch.clamp(torch.exp(lr), max=1.0) * (r - v)
    assert_close(d.vs, closed, 1e-6, 'closed form')
    # spot-check 64 columns against the oracle
    idx = torch.arange(0, B, B // 64, device='cuda')
    vs, pg = O.vtrace_from_importance_weights(lr[:, idx].cpu(), disc[:, idx].cpu(), r[:, idx].cpu(), v[:, idx].cpu(), boot[idx].cpu())
    assert_close(a.vs[:, idx], vs, 1e-4, 'full-size vs sample')


@pytest.mark.parametrize('T,B,A', [(20, 32, 6), (5, 3, 4), (20, 512, 4), (7, 129, 18)])
def test_from_logits_vs_oracle(ops, T, B, A):
    rng = np.random.RandomState(T + B + A)
    bl = torch.from_numpy(rng.randn(T, B, A).astype(np.float32))
    tl = torch.from_numpy(rng.randn(T, B, A).astype(np.float32))
    actions = torch.from_numpy(rng.randint(0, A, size=(T, B)).astype(np.int64))
    discounts = torch.from_numpy(((rng.rand(T, B) > 0.05) * 0.99).astype(np.float32))
    rewards = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    values = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    boot = torch.from_numpy(rng.randn(B).astype(np.float32))
    ref = O.vtrace_from_logits(bl, tl, actions, discounts, rewards, values, boot)
    r = ops.from_logits(dev(bl), dev(tl), dev(actions), dev(discounts), dev(rewards), dev(values), dev(boot))
    for got, want, name in zip(r, ref, r._fields):
        assert_close(got, want, 1e-4, name)


@pytest.mark.parametrize('T,B,A,clip', [(20, 32, 6, 'abs_one'), (20, 64, 4, 'none'), (3, 200, 18, 'abs_one'), (20, 512, 4, 'abs_one')])
def test_fused_tail_vs_oracle(ops, T, B, A, clip):
    batch = O.synthetic_batch(T, B, A, seed=B, done_p=0.05)
    rng = np.random.RandomState(B)
    tl = torch.from_numpy(rng.randn(T + 1, B, A).astype(np.float32))
    baseline = torch.from_numpy(rng.randn(T + 1, B).astype(np.float32))
    rewards = batch['reward'][1:]
    if clip == 'abs_one':
        rewards = torch.clamp(rewards, -1, 1)
    discounts = (~batch['done'][1:]).float() * 0.99
    vs, pg, *_ = O.vtrace_from_logits(batch['policy_logits'][1:], tl[:-1], batch['action'][1:], discounts, rewards, baseline[:-1], baseline[-1])
    l = O.impala_losses(tl[:-1], batch['action'][1:], baseline[:-1], vs, pg, 0.5, 0.0006)
    dl, dv = O.head_grads(tl[:-1], batch['action'][1:], baseline[:-1], vs, pg, 0.5, 0.0006)
    out = ops.impala_loss_and_head_grads(dev(batch['policy_logits']), dev(tl), dev(baseline), dev(batch['action']), dev(batch['reward']),
                                         dev(batch['done']), reward_clipping=clip)
    assert_close(out['vs'], vs, 1e-4, 'vs')
    assert_close(out['pg_advantages'], pg, 1e-4, 'pg')
    assert_close(out['dlogits'], dl, 1e-4, 'dlogits')
    assert_close(out['dbaseline'], dv, 1e-4, 'dbaseline')
    want = np.array([float(l[0]), float(l[1]), float(l[2]), float(l[0] + l[1] + l[2])])
    got = out['losses'].cpu().numpy()
    assert np.all(np.abs(got - want) <= 1e-4 * np.abs(want).max()), (got, want)
    # the kernel re-arms its reduction ticket: a second call gives identical losses
    out2 = ops.impala_loss_and_head_grads(dev(batch['policy_logits']), dev(tl), dev(baseline), dev(batch['action']), dev(batch['reward']),
                                          dev(batch['done']), reward_clipping=clip)
    assert torch.equal(out2['losses'], out['losses'])


# ------------------------------------------------------------------------------------------------
# learner: forward, full step
# ------------------------------------------------------------------------------------------------
def _learner(T, B, A, seed, **kw):
    from scalerl_b200.learner import B200ImpalaLearner, ImpalaHParams
    hp = ImpalaHParams(rollout_length=T, batch_size=B, num_actions=A, **kw)
    params = O.init_params(A, seed=seed)
    return B200ImpalaLearner(hp, init_state_dict=params, process_group=False), params


def _nhwc_to_nchw(flat, N, H, C):
    return flat.float().view(N, H, H, C).permute(0, 3, 1, 2).contiguous().cpu()


def _a1_planes_to_nchw(flat, N):
    """a1 is stored as two row-parity planes [hp][n][h>>1][w>>1][(w&1)*32 + c] (res_problems.cuh)"""
    t = flat.float().view(2, N, 10, 10, 2, 32)            # hp, n, h2, w2, wp, c
    return t.permute(1, 5, 2, 0, 3, 4).reshape(N, 32, 20, 20).contiguous().cpu()


@pytest.mark.parametrize('T,B', [(4, 5), (2, 1), (6, 23), (1, 1), (3, 50)])
def test_forward_vs_emulating_oracle(T, B):
    A = 6
    L, params = _learner(T, B, A, 2)
    batch = O.synthetic_batch(T, B, A, seed=3)
    out = L.forward({k: dev(v) for k, v in batch.items()})
    lg, bs, saved = O.atari_forward(params, batch['obs'], batch['reward'], batch['action'], emulate_bf16=True, keep=True)
    N = (T + 1) * B
    assert rel_l2(_a1_planes_to_nchw(L.debug_buffer('a1'), N), saved['a1']) < 2e-3
    assert rel_l2(_nhwc_to_nchw(L.debug_buffer('a2'), N, 9, 64), saved['a2']) < 3e-3
    assert rel_l2(_nhwc_to_nchw(L.debug_buffer('a3'), N, 7, 64), saved['a3']) < 4e-3
    assert rel_l2(L.debug_buffer('h').view(N, 512).cpu(), saved['h']) < 5e-3
    assert rel_l2(out['policy_logits'].cpu(), lg) < 5e-3
    assert rel_l2(out['baseline'].cpu(), bs) < 5e-3
    # and within bf16 distance of the fp32 reference arithmetic
    lg32, bs32 = O.atari_forward(params, batch['obs'], batch['reward'], batch['action'])
    assert rel_l2(out['policy_logits'].cpu(), lg32) < 2e-2


@pytest.mark.parametrize('precision', ['bf16', 'fp32_split'])
def test_packed_weight_copies_are_the_documented_permutations(precision):
    """pack_weights_kernel: every bf16 operand copy (kernels.h WPack) is bit-for-bit the bf16 rounding of the fp32 master in the
    documented layout -- and in the fp32-accurate mode the low copy is the rounding of the remainder"""
    A = 6
    L, params = _learner(2, 2, A, 5, precision=precision)
    L.forward({k: dev(v) for k, v in O.synthetic_batch(2, 2, A, seed=1).items()})       # runs the pack
    w1, w2, w3, wf = (params[k].float() for k in ('conv1.weight', 'conv2.weight', 'conv3.weight', 'fc.weight'))
    want = [
        w1.view(32, 4, 2, 4, 2, 4).permute(0, 2, 4, 1, 3, 5).reshape(-1),                # w1k[co][(kh2,kw2)][c,dy,dx]
        w2.permute(0, 2, 3, 1).reshape(-1),                                              # w2k[co][(kh,kw)][c]
        w3.permute(0, 2, 3, 1).reshape(-1),                                              # w3k[co][(kh,kw)][c]
        wf.view(512, 64, 49).permute(0, 2, 1).reshape(-1),                               # wfk[j][hw][c]
        wf.view(512, 64, 49).permute(2, 1, 0).reshape(-1),                               # wfd[hw][c][j]
        w3.permute(1, 2, 3, 0).reshape(-1),                                              # w3d[c][(kh,kw)][co]
        w2.view(64, 32, 2, 2, 2, 2).permute(3, 5, 1, 2, 4, 0).reshape(-1),               # w2d[(ph,pw)][c][(kh',kw')][co], kh = ph + 2 kh'
    ]
    want = torch.cat(want)
    hi = want.to(torch.bfloat16)
    got = L.debug_buffer('wpack').cpu()
    assert got.numel() == want.numel()
    assert torch.equal(got.view(torch.int16), hi.view(torch.int16))
    if precision == 'fp32_split':
        lo = (want - hi.float()).to(torch.bfloat16)
        assert torch.equal(L.debug_buffer('wpack_lo').cpu().view(torch.int16), lo.view(torch.int16))
    L.close()


@pytest.mark.parametrize('rows', [1, 3])
def test_forward_with_fewer_rows_than_the_context_holds(rows):
    """srl_learner_forward(rows < T+1) (the actor-inference use): round 1 strided conv1's output planes by the rows of the CALL
    while conv2's tensor map is built for the context's capacity -- wrong logits whenever rows != T+1"""
    T, B, A = 4, 5, 6
    L, params = _learner(T, B, A, 2)
    batch = O.synthetic_batch(T, B, A, seed=3)
    sub = {k: v[:rows].contiguous() for k, v in batch.items()}
    out = L.forward({k: dev(v) for k, v in sub.items()})
    lg, bs = O.atari_forward(params, sub['obs'], sub['reward'], sub['action'], emulate_bf16=True)
    assert rel_l2(out['policy_logits'].cpu(), lg) < 5e-3 and rel_l2(out['baseline'].cpu(), bs) < 5e-3


@pytest.mark.parametrize('T,B,optimizer', [(5, 6, 'rmsprop'), (5, 6, 'adam'), (3, 1, 'rmsprop'), (7, 19, 'rmsprop')])
def test_learn_step_vs_emulating_oracle(T, B, optimizer):
    """Two consecutive steps.  Gradients are compared with the bf16-emulating oracle; the integrated
    clip + optimizer update is checked by replaying the ORACLE's clip/optimizer on the gradients the GPU
    produced (RMSprop/Adam normalise the step, so comparing post-step weights across slightly different
    gradients would only measure sign flips of near-zero gradients).  After each step the oracle state is
    re-synchronised to the device state so step 2 starts from identical weights."""
    A = 6
    L, params = _learner(T, B, A, 4, optimizer=optimizer)
    opt = O.new_opt_state(params, optimizer)
    hp = dict(optimizer=optimizer)
    for step in range(2):
        batch = O.synthetic_batch(T, B, A, seed=20 + step, done_p=0.1)
        before = {k: v.clone() for k, v in params.items()}
        opt_before = {k: ({n: t.clone() for n, t in v.items()} if isinstance(v, dict) else v) for k, v in opt.items()}
        ref = O.learn_step(params, opt, batch, hp, emulate_bf16=True)
        stats = L.learn({k: dev(v) for k, v in batch.items()})
        assert_close(L._vs, ref['vs'], 2e-2, 'vs')          # inputs differ by bf16-level logits differences
        for k in ('pg_loss', 'baseline_loss', 'entropy_loss', 'total_loss'):
            assert abs(stats[k] - ref[k]) <= 2e-2 * max(1.0, abs(ref[k])), (k, stats[k], ref[k])
        assert np.allclose(stats['episode_returns'], ref['episode_returns'])
        for k in O.PARAM_ORDER:
            e = rel_l2(L.grads[k].cpu(), ref['grads'][k])
            assert e < 2e-2, (step, k, e)
        assert abs(stats['grad_norm'] - ref['grad_norm']) <= 1e-2 * ref['grad_norm']
        # replay clip + optimizer of the oracle on the device gradients
        g_dev = {k: L.grads[k].cpu().clone() for k in O.PARAM_ORDER}
        gn, coef = O.clip_grad_norm(g_dev, 40.0)
        assert abs(gn - stats['grad_norm']) <= 1e-5 * gn
        if optimizer == 'rmsprop':
            O.rmsprop_step(before, g_dev, opt_before['square_avg'], 1e-4, 0.99, 1e-5)
        else:
            O.adam_step(before, g_dev, opt_before['exp_avg'], opt_before['exp_avg_sq'], step + 1, 1e-4)
        for k in O.PARAM_ORDER:
            assert_close(L.params[k], before[k], 2e-6, f'post-step {k}')
        # re-synchronise the oracle to the device state
        for k in O.PARAM_ORDER:
            params[k].copy_(L.params[k].cpu())
        for name, d in L._opt_tensors().items():
            for k in O.PARAM_ORDER:
                opt[name][k].copy_(d[k].cpu())


@pytest.mark.parametrize('T,B', [(5, 4), (3, 7), (1, 1), (7, 19), (12, 24)])
def test_learn_step_ignores_stale_shared_memory(T, B):
    """Ragged frame counts (T*B not a multiple of any tile/slab) after every SM's shared memory was filled with NaN
    patterns: the gradients must be finite and equal those of a run on clean shared memory up to the summation
    order of the atomics (regression: 0 * stale-smem in the head weight-gradient slab)."""
    from scalerl_b200 import _lib
    A = 6
    batch = {k: dev(v) for k, v in O.synthetic_batch(T, B, A, seed=77, done_p=0.2).items()}
    grads = []
    for poison in (False, True):
        L, _ = _learner(T, B, A, 4, learning_rate=0.0)     # lr = 0: the three steps see identical weights
        for _ in range(3):                      # eager, capture, replay
            if poison:
                _lib.check_hook(_lib.hooks().srl_test_poison_smem(None))
                torch.cuda.synchronize()
            L.learn(batch)
        g = L.flat_grads.clone()
        assert bool(torch.isfinite(g).all()) and bool(torch.isfinite(L.flat_params).all())
        grads.append(g)
    assert rel_l2(grads[1].cpu(), grads[0].cpu()) < 1e-5


@pytest.mark.parametrize('T,B', [(7, 19), (12, 24)])
def test_conv_bias_gradients_equal_dy_column_sums_every_run(T, B):
    """conv1/conv2 bias gradients are column sums of dy tiles staged in shared memory, read by the epilogue warps while the
    MMAs run.  Regression for a release hazard (the stage was handed back to the TMA producer while the warp's loads were
    still in flight -> rows of the NEXT chunk were summed, sporadically, only when kernels overlap via programmatic
    dependent launch): 30 back-to-back runs on a non-default stream, each compared with sum(da1) / sum(da2) taken from
    the debug buffers of the same run, and all gradients compared with the first run."""
    A = 4
    L, _ = _learner(T, B, A, 1)
    batch = {k: dev(v) for k, v in O.synthetic_batch(T, B, A, seed=5).items()}
    first = None
    with torch.cuda.stream(torch.cuda.Stream()):
        for it in range(30):
            L.forward_backward(batch)
            torch.cuda.current_stream().synchronize()
            b1 = L.debug_buffer('da1').float().view(-1, 32).sum(0)
            b2 = L.debug_buffer('da2').float().view(-1, 64).sum(0)
            assert rel_l2(L.grads['conv1.bias'].cpu(), b1.cpu()) < 1e-4, it
            assert rel_l2(L.grads['conv2.bias'].cpu(), b2.cpu()) < 1e-4, it
            g = L.flat_grads.clone()
            if first is None:
                first = g
            assert rel_l2(g.cpu(), first.cpu()) < 1e-5, it


@pytest.mark.parametrize('T,B,A', [(5, 6, 6), (7, 19, 6), (33, 3, 6), (6, 5, 18), (4, 3, 1)])
def test_column_kernel_equals_three_kernel_path(T, B, A, monkeypatch):
    """heads + V-trace/losses + dh as ONE column kernel vs the head_fwd / impala_tail / head_bwd_dh kernels it replaces
    (still used when (T+1) * 2 KB of shared memory does not fit): same losses, vs, advantages and gradients.
    A = 18 exercises the 32-action instantiation, T = 33 the two-chunk scan."""
    batch = {k: dev(v) for k, v in O.synthetic_batch(T, B, A, seed=31, done_p=0.15).items()}
    outs = []
    for no_fuse in ('0', '1'):
        monkeypatch.setenv('SRL_NO_COLUMN_FUSION', no_fuse)
        L, _ = _learner(T, B, A, 3, learning_rate=0.0)
        st = L.learn(batch)
        outs.append((st, L._vs.clone(), L._pg_adv.clone(), L.flat_grads.clone(), L.debug_buffer('logits'), L.debug_buffer('dh').float()))
    (s0, vs0, pg0, g0, lg0, dh0), (s1, vs1, pg1, g1, lg1, dh1) = outs
    for k in ('pg_loss', 'baseline_loss', 'entropy_loss', 'total_loss'):
        assert abs(s0[k] - s1[k]) <= 1e-5 * max(1.0, abs(s1[k])), k
    assert rel_l2(lg0.cpu(), lg1.cpu()) < 1e-6 and rel_l2(vs0.cpu(), vs1.cpu()) < 1e-5 and rel_l2(pg0.cpu(), pg1.cpu()) < 1e-4
    assert rel_l2(dh0.cpu(), dh1.cpu()) < 2e-3                # bf16 rounding of values that differ in the last fp32 bits
    assert rel_l2(g0.cpu(), g1.cpu()) < 2e-3


@pytest.mark.parametrize('fusion', ['column_kernel', 'three_kernels'])
@pytest.mark.parametrize('name', ['t5b4a6', 't3b5a4'])
def test_learn_step_vs_reference_goldens(name, fusion, monkeypatch):
    monkeypatch.setenv('SRL_NO_COLUMN_FUSION', '0' if fusion == 'column_kernel' else '1')   # heads+V-trace+dh fused or not
    g = np.load(os.path.join(GOLDEN, f'learn_{name}.npz'))
    T, B, A, seed, steps, clip = [int(v) for v in g['meta']]
    L, params = _learner(T, B, A, seed, reward_clipping='abs_one' if clip else 'none')
    batch = O.synthetic_batch(T, B, A, seed=seed * 10)
    stats = L.learn({k: dev(v) for k, v in batch.items()})
    lg = L.debug_buffer('logits').view(T + 1, B, A).cpu()
    assert rel_l2(lg, g['s0_policy_logits']) < 2e-2
    assert rel_l2(L.debug_buffer('baseline').view(T + 1, B).cpu(), g['s0_baseline']) < 2e-2
    assert rel_l2(L._vs.cpu(), g['s0_vs']) < 3e-2
    assert abs(stats['total_loss'] - g['s0_losses'][3]) <= 3e-2 * max(1.0, abs(g['s0_losses'][3]))
    for k in O.PARAM_ORDER:
        samp = strided_sample(L.grads[k].reshape(-1).cpu())
        assert rel_l2(samp, g['s0_gradsamp_' + k]) < 0.15, k
        gn = float(L.grads[k].double().norm())
        assert abs(gn - g['s0_gradnorm_' + k][0]) <= 0.1 * g['s0_gradnorm_' + k][0] + 1e-6, k


def test_vtrace_given_identical_inputs_matches_1e4():
    """north_star: V-trace returns/advantages within 1e-4 of the reference path on IDENTICAL inputs --
    feed the learner's own logits/baseline to the oracle's V-trace."""
    T, B, A = 20, 32, 6
    L, params = _learner(T, B, A, 0)
    batch = O.synthetic_batch(T, B, A, seed=0)
    L.learn({k: dev(v) for k, v in batch.items()})
    lg = L.debug_buffer('logits').view(T + 1, B, A).cpu()
    bs = L.debug_buffer('baseline').view(T + 1, B).cpu()
    rewards = torch.clamp(batch['reward'][1:], -1, 1)
    discounts = (~batch['done'][1:]).float() * 0.99
    vs, pg, *_ = O.vtrace_from_logits(batch['policy_logits'][1:], lg[:-1], batch['action'][1:], discounts, rewards, bs[:-1], bs[-1])
    assert_close(L._vs, vs, 1e-4, 'vs')
    assert_close(L._pg_adv, pg, 1e-4, 'pg_adv')
    assert torch.allclose(L._vs.cpu(), vs, rtol=1e-4, atol=1e-5)


def test_full_size_properties_cfg3_shard():
    """T=20, B=64 (config 3's per-GPU shard): (i) the step is deterministic up to fp32 atomics,
    (ii) gradients are additive over column shards: grads(B=64) == grads(cols 0..31) + grads(cols 32..63)
    -- the property the NCCL SUM all-reduce relies on (SURVEY.md §8e)."""
    T, A = 20, 4
    full, params = _learner(T, 64, A, 1)
    batch = {k: dev(v) for k, v in O.synthetic_batch(T, 64, A, seed=5).items()}
    full.forward_backward(batch)
    g_full = full.flat_grads.clone()
    half, _ = _learner(T, 32, A, 1)
    acc = torch.zeros_like(g_full)
    for s in (slice(0, 32), slice(32, 64)):
        half.forward_backward({k: v[:, s].contiguous() for k, v in batch.items()})
        acc += half.flat_grads
    assert rel_l2(acc.cpu(), g_full.cpu()) < 1e-4
    full.forward_backward(batch)
    assert rel_l2(full.flat_grads.cpu(), g_full.cpu()) < 1e-5


def test_optimizer_ops_vs_oracle():
    from scalerl_b200 import _lib
    L = _lib.lib()
    n = 1687768 + 3
    g = torch.Generator().manual_seed(0)
    p = torch.randn(n, generator=g)
    gr = torch.randn(n, generator=g) * 0.3
    v = torch.rand(n, generator=g)
    P, G, V = dev(p), dev(gr), dev(v)
    coef = torch.zeros(2, device='cuda')
    scratch = torch.zeros(2048, device='cuda')
    _lib.check(L.srl_grad_norm_clip_coef(G.data_ptr(), n, 40.0, coef.data_ptr(), scratch.data_ptr(), None))
    torch.cuda.synchronize()
    norm = float(gr.double().norm())
    assert abs(coef[0].item() - norm) <= 1e-5 * norm
    assert abs(coef[1].item() - min(1.0, 40.0 / (norm + 1e-6))) <= 1e-6
    _lib.check(L.srl_rmsprop_step(P.data_ptr(), G.data_ptr(), V.data_ptr(), n, coef.data_ptr(), 1e-4, 0.99, 1e-5, None))
    pr, vr, gc = {'x': p.clone()}, {'x': v.clone()}, {'x': gr * coef[1].item()}
    O.rmsprop_step(pr, gc, vr, 1e-4, 0.99, 1e-5)
    assert_close(P, pr['x'], 1e-6, 'rmsprop p')
    assert_close(V, vr['x'], 1e-6, 'rmsprop v')
    m = torch.zeros(n)
    M, V2, P2 = dev(m), dev(v), dev(p)
    pa, ma, va = {'x': p.clone()}, {'x': m.clone()}, {'x': v.clone()}
    for step in (1, 2):
        _lib.check(L.srl_adam_step(P2.data_ptr(), G.data_ptr(), M.data_ptr(), V2.data_ptr(), n, None, 1e-3, 0.9, 0.999, 1e-8, step, None))
        O.adam_step(pa, {'x': gr}, ma, va, step, 1e-3)
    assert_close(P2, pa['x'], 1e-6, 'adam p')


def test_graph_replay_equals_eager():
    """the CUDA-graph path (wgrads on a parallel branch) gives the same update as eager single-stream launches"""
    T, B, A = 5, 6, 6
    La, params = _learner(T, B, A, 7)
    Lb, _ = _learner(T, B, A, 7)
    La.use_graph, Lb.use_graph = True, False
    batch = {k: dev(v) for k, v in O.synthetic_batch(T, B, A, seed=3, done_p=0.1).items()}
    for step in range(4):          # eager warm-up, capture, replay, replay
        sa = La.learn(batch)
        sb = Lb.learn(batch)
        assert abs(sa['total_loss'] - sb['total_loss']) <= 1e-5 * max(1.0, abs(sb['total_loss'])), step
        assert rel_l2(La.flat_grads.cpu(), Lb.flat_grads.cpu()) < 1e-4, step      # fp32 atomics order differs
        assert rel_l2(La.flat_params.cpu(), Lb.flat_params.cpu()) < 1e-4, step    # RMSprop normalises: near-zero grads may flip sign
    assert len(La._graphs) == 1 and len(Lb._graphs) == 0


@pytest.mark.parametrize('mn_major', [0, 1])
def test_shifted_operand_descriptors(mn_major):
    """Hardware property the resident-window kernels rely on: a UMMA operand descriptor may start at ANY 128-byte row
    of a SWIZZLE_128B tile with base_offset = 0 (the swizzle is applied to absolute shared-memory address bits)."""
    from scalerl_b200 import _lib
    Lb = _lib.hooks()
    g = torch.Generator().manual_seed(mn_major)
    if mn_major == 0:
        A = torch.randn(160, 64, generator=g).bfloat16().cuda()
        Bm = torch.randn(64, 64, generator=g).bfloat16().cuda()
    else:
        A = torch.randn(96, 128, generator=g).bfloat16().cuda()
        Bm = torch.randn(96, 64, generator=g).bfloat16().cuda()
    for shift in range(0, 25):
        D = torch.zeros(128, 64, device='cuda')
        _lib.check_hook(Lb.srl_test_shifted_operand(A.data_ptr(), Bm.data_ptr(), D.data_ptr(), shift, mn_major, 0, None))
        torch.cuda.synchronize()
        ref = (A[shift:shift + 128].float() @ Bm.float().t()) if mn_major == 0 else (A[shift:shift + 64].float().t() @ Bm[shift:shift + 64].float())
        assert_close(D, ref, 1e-5, f'shift {shift}')


def test_graft_smoke():
    import __graft_entry__ as ge
    ge.smoke()


def test_full_size_cfg3_sharding_property():
    """BASELINE.json configs[2]: T=20, B=512 sharded 8 x 64 columns.  The full-batch gradient on one GPU equals the SUM of
    the eight shard gradients (what the NCCL SUM all-reduce computes); exercises the B=512 buffers / tensor maps."""
    T, A, B, shards = 20, 4, 512, 8
    full, params = _learner(T, B, A, 2)
    g = torch.Generator(device='cuda').manual_seed(0)
    batch = {
        'obs': torch.randint(0, 256, (T + 1, B, 4, 84, 84), dtype=torch.uint8, device='cuda', generator=g),
        'reward': torch.randn(T + 1, B, device='cuda', generator=g),
        'done': torch.rand(T + 1, B, device='cuda', generator=g) < 0.02,
        'action': torch.randint(0, A, (T + 1, B), device='cuda', generator=g),
        'policy_logits': torch.randn(T + 1, B, A, device='cuda', generator=g),
        'episode_return': torch.randn(T + 1, B, device='cuda', generator=g)}
    full.forward_backward(batch)
    g_full = full.flat_grads.clone()
    loss_full = full._losses.clone()
    part, _ = _learner(T, B // shards, A, 2)
    acc = torch.zeros_like(g_full)
    loss_acc = torch.zeros_like(loss_full)
    for s in range(shards):
        sl = slice(s * 64, (s + 1) * 64)
        part.forward_backward({k: v[:, sl].contiguous() for k, v in batch.items()})
        acc += part.flat_grads
        loss_acc += part._losses
    assert rel_l2(acc.cpu(), g_full.cpu()) < 2e-4
    assert torch.allclose(loss_acc.cpu(), loss_full.cpu(), rtol=1e-4, atol=1e-2)
    assert torch.isfinite(g_full).all()


def test_programmatic_dependent_launch_waits_for_the_primary_grid():
    """The step's kernels are chained with programmatic stream serialization; every kernel relies on
    griddepcontrol.wait returning only after the previous grid completed and flushed.  Self-test: kernel A spins ~20 us
    then sets a flag, kernel B (512 blocks, launched with the attribute) records the flag after its wait -- on the
    legacy default stream and on a created stream."""
    from scalerl_b200 import _lib
    L = _lib.hooks()
    flag = torch.zeros(1, dtype=torch.int32, device='cuda')
    out = torch.zeros(512, dtype=torch.int32, device='cuda')
    for st in (None, torch.cuda.Stream()):
        for _ in range(20):
            out.zero_()
            torch.cuda.synchronize()
            _lib.check_hook(L.srl_test_pdl(flag.data_ptr(), out.data_ptr(), 512, 20000, st.cuda_stream if st else None))
            torch.cuda.synchronize()
            assert int((out != 1).sum()) == 0
