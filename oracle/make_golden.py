"""Generate tests/golden/*.npz by running the REFERENCE's own importable modules.

Run in the build container only (needs /root/reference, which does not exist on the GPU box):

    python oracle/make_golden.py

It imports, by path, the three leaf modules of the reference hot path
  /root/reference/scalerl/algorithms/impala/vtrace.py
  /root/reference/scalerl/algorithms/impala/loss_fn.py
  /root/reference/scalerl/algorithms/utils/atari_model.py
(the trainer module impala_atari.py itself cannot be imported: wrong import roots + gymnasium missing,
SURVEY.md §0) and drives them with the statements of ImpalaTrainer.learn (impala_atari.py:288-346).
Inputs are NOT stored: they are regenerated from seeds by oracle.impala_oracle.{init_params,
synthetic_batch} (numpy RNG), so the fixtures stay a few KB.
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import impala_oracle as O  # noqa: E402

REF = '/root/reference/scalerl/algorithms'


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _samp(flat):
    """the strided sample of tests.helpers.strided_sample"""
    return flat[torch.linspace(0, flat.numel() - 1, steps=min(257, flat.numel())).long()]


# ---------------- seeded inputs of the randomised comparisons (tests/test_oracle_vs_live_reference.py,
# tests/test_host_logic_cpu.py, tests/test_ref_learner_cpu.py): the tests build the same inputs with these functions ----------------
def vtrace_random_inputs(seed):
    """keyword arguments of vtrace.from_logits: random (T, B, A), terminal steps, every clip-threshold combination incl. None"""
    rng = np.random.RandomState(100 + seed)
    T, B, A = int(rng.randint(1, 40)), int(rng.randint(1, 9)), int(rng.randint(1, 19))
    t = lambda *s: torch.from_numpy(rng.randn(*s).astype(np.float32))
    bl, tl = t(T, B, A) * 1.5, t(T, B, A) * 1.5
    actions = torch.from_numpy(rng.randint(0, A, size=(T, B)).astype(np.int64))
    discounts = torch.from_numpy(((rng.rand(T, B) > 0.15) * 0.99).astype(np.float32))
    rewards, values, boot = t(T, B), t(T, B), t(B)
    return dict(behavior_policy_logits=bl, target_policy_logits=tl, actions=actions, discounts=discounts, rewards=rewards,
                values=values, bootstrap_value=boot, clip_rho_threshold=[1.0, None, 2.5, 0.3][seed % 4],
                clip_pg_rho_threshold=[1.0, 0.7, None][seed % 3])


def loss_random_inputs(seed):
    """(logits, values, actions, vs, advantages, baseline_cost, entropy_cost) of the loss functions"""
    rng = np.random.RandomState(200 + seed)
    T, B, A = int(rng.randint(1, 25)), int(rng.randint(1, 7)), int(rng.randint(2, 19))
    logits = torch.from_numpy(rng.randn(T, B, A).astype(np.float32))
    values = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    actions = torch.from_numpy(rng.randint(0, A, size=(T, B)).astype(np.int64))
    vs = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    adv = torch.from_numpy(rng.randn(T, B).astype(np.float32))
    return logits, values, actions, vs, adv, 0.5, 0.0006 * (1 + seed)


def lstm_random_inputs(A, seed):
    """(params, lstm params, batch, initial state) of a T=4, B=3 AtariNet(use_lstm=True) forward"""
    T, B = 4, 3
    batch = O.synthetic_batch(T, B, A, seed=seed + 7, done_p=0.3)
    g = torch.Generator().manual_seed(seed)
    state = (torch.randn(2, B, 513 + A, generator=g) * 0.1, torch.randn(2, B, 513 + A, generator=g) * 0.1)
    return O.init_params(A, seed=seed), O.init_lstm_params(A, seed=seed), batch, state


def per_random_inputs(seed):
    """(memory size, alpha, beta, rounds): per round the number of adds, the update indices (duplicates on purpose: last
    write wins) and priorities, and the uniforms of one stratified sample; capacities include wrap-around of the ring"""
    rng = np.random.RandomState(300 + seed)
    mem = int(rng.choice([7, 64, 100, 333, 1024]))
    alpha, beta = float(rng.choice([0.4, 0.6, 1.0])), float(rng.choice([0.4, 0.7, 1.0]))
    rounds, size = [], 0
    for _ in range(3):
        nadd = int(rng.randint(1, 2 * mem))
        size = min(size + nadd, mem)
        k = int(rng.randint(1, 50))
        idx = rng.randint(0, size, size=k)
        pr = rng.rand(k) * 4 + 1e-3
        u = rng.rand(int(rng.randint(1, 40)))
        rounds.append((nadd, idx, pr, u))
    return mem, alpha, beta, rounds


def actor_weights(A, use_lstm):
    """the state_dict both the reference AtariNet and the actor stand-in hold in the one-step actor comparison"""
    return {**O.init_params(A, seed=0), **(O.init_lstm_params(A, seed=0) if use_lstm else {})}


LEARNER_CASES = [(5, 4, 6, 'abs_one'), (3, 7, 4, 'none')]       # (T, B, A, reward clipping), two steps each


def learner_inputs(T, B, A):
    """(initial params, batch) of the two-step reference-learner comparison"""
    return O.init_params(A, seed=2), O.synthetic_batch(T, B, A, seed=5, done_p=0.2)


def reference_cases(vtrace, loss_fn, atari_model):
    """-> dict of arrays: the reference's outputs on the seeded inputs above (tests/golden/reference_cases.npz)"""
    from scalerl_b200.algorithms.utils.atari_model import SyntheticAtariEnv
    from oracle import make_ref
    from oracle import ref_learner as R
    seg = _load('ref_segment_tree', os.path.join(REF, '..', 'data', 'segment_tree.py'))
    prof = _load('ref_profile', os.path.join(REF, '..', 'utils', 'profile.py'))
    g = {}
    for seed in range(12):
        r = vtrace.from_logits(**vtrace_random_inputs(seed))
        for k, v in dict(vs=r.vs, pg=r.pg_advantages, log_rhos=r.log_rhos, balp=r.behavior_action_log_probs,
                         talp=r.target_action_log_probs).items():
            g[f'vtrace_s{seed}_{k}'] = v.numpy()
    for seed in range(6):
        logits, values, actions, vs, adv, bc, ec = loss_random_inputs(seed)
        logits.requires_grad_(True)
        values.requires_grad_(True)
        pg = loss_fn.compute_policy_gradient_loss(logits, actions, adv)
        bl = bc * loss_fn.compute_baseline_loss(vs - values)
        en = ec * loss_fn.compute_entropy_loss(logits)
        (pg + bl + en).backward()
        g[f'loss_s{seed}_losses'] = np.array([pg.item(), bl.item(), en.item()])
        g[f'loss_s{seed}_dlogits'], g[f'loss_s{seed}_dvalues'] = logits.grad.numpy(), values.grad.numpy()
    for A, seed in [(6, 0), (18, 1), (3, 2)]:
        net = atari_model.AtariNet((4, 84, 84), A, use_lstm=False)
        net.load_state_dict(O.init_params(A, seed=seed))
        with torch.no_grad():
            out, _ = net(O.synthetic_batch(3, 2, A, seed=seed), ())
        g[f'atari_a{A}_s{seed}_logits'], g[f'atari_a{A}_s{seed}_baseline'] = out['policy_logits'].numpy(), out['baseline'].numpy()
    for A, seed in [(6, 0), (3, 1)]:
        params, lp, batch, state = lstm_random_inputs(A, seed)
        net = atari_model.AtariNet((4, 84, 84), A, use_lstm=True)
        net.load_state_dict({**params, **lp})
        with torch.no_grad():
            out, ns = net(batch, state)
        p = f'lstm_a{A}_s{seed}_'
        g[p + 'logits'], g[p + 'baseline'], g[p + 'h'], g[p + 'c'] = out['policy_logits'].numpy(), out['baseline'].numpy(), ns[0].numpy(), ns[1].numpy()
    for seed in range(6):          # segment_tree.py driven by the statements of PrioritizedReplayBuffer (replay_buffer.py:318-381)
        mem, alpha, beta, rounds = per_random_inputs(seed)
        cap = 1
        while cap < mem:
            cap *= 2
        st, mt = seg.SumSegmentTree(cap), seg.MinSegmentTree(cap)
        max_p, ptr, size = 1.0, 0, 0
        for rnd, (nadd, idx, pr, u) in enumerate(rounds):
            for _ in range(nadd):
                st[ptr] = max_p ** alpha
                mt[ptr] = max_p ** alpha
                ptr = (ptr + 1) % mem
                size = min(size + 1, mem)
            for i, p in zip(idx, pr):
                st[int(i)] = float(p) ** alpha
                mt[int(i)] = float(p) ** alpha
                max_p = max(max_p, float(p))
            segment = st.sum(0, size - 1) / len(u)
            want = [st.find_prefixsum_idx(segment * i + (segment * (i + 1) - segment * i) * float(u[i])) for i in range(len(u))]
            max_w = (mt.min() / st.sum() * size) ** (-beta)
            p = f'per_s{seed}_r{rnd}_'
            g[p + 'idx'] = np.array(want, dtype=np.int64)
            g[p + 'w'] = np.array([((st[i] / st.sum()) * size) ** (-beta) / max_w for i in want], dtype=np.float64)
            g[p + 'sum'], g[p + 'min'] = np.array([st.sum()]), np.array([mt.min()])
    for use_lstm in (False, True):
        A, p = 6, f'actor_lstm{int(use_lstm)}_'
        net = atari_model.AtariNet((4, 84, 84), A, use_lstm=use_lstm)
        g[f'param_order_lstm{int(use_lstm)}'] = np.array([n for n, _ in net.named_parameters()])
        sd = net.state_dict()
        g[p + 'keys'] = np.array(list(sd))
        for k, v in sd.items():
            g[p + 'shape_' + k] = np.array(v.shape, dtype=np.int64)
        net.load_state_dict(actor_weights(A, use_lstm))
        net.eval()
        state = net.initial_hidden_state(1)
        g[p + 'state_shapes'] = np.array([s.shape for s in state], dtype=np.int64).reshape(-1, 3)
        torch.manual_seed(0)                       # SyntheticAtariEnv mixes torch.initial_seed() into its seed
        env = SyntheticAtariEnv((4, 84, 84), A, seed=3)
        out = env.reset()
        for t in range(4):
            with torch.no_grad():
                o, state = net(out, state)
            g[f'{p}t{t}_logits'], g[f'{p}t{t}_baseline'], g[f'{p}t{t}_action'] = o['policy_logits'].numpy(), o['baseline'].numpy(), o['action'].numpy()
            for i, s in enumerate(state):
                g[f'{p}t{t}_state{i}'] = s.numpy()
            out = env.step(o['action'])
            if t == 1:
                out['done'] = torch.ones(1, 1, dtype=torch.bool)          # exercises the state reset (atari_model.py:114-116)
    import timeit                                  # Timings fed the samples 0.5, 0.25, 1.0, 0.75 through a stubbed clock
    tm = prof.Timings()
    real = timeit.default_timer
    try:
        for x in (0.5, 0.25, 1.0, 0.75):
            tm.last_time = 0.0
            timeit.default_timer = lambda x=x: x
            tm.time('k')
    finally:
        timeit.default_timer = real
    g['timings_mean_var'] = np.array([tm.means()['k'], tm.vars()['k']])
    assert make_ref.build(verbose=False)           # the reference learner of bench.py's reference arm, two steps
    for T, B, A, clip in LEARNER_CASES:
        params, batch = learner_inputs(T, B, A)
        L = R.ReferenceLearner(A, state_dict=params, reward_clipping=clip)
        for step in range(2):
            st = L.learn(batch)
            p = f'learner_t{T}b{B}a{A}_{clip}_s{step}_'
            g[p + 'stats'] = np.array([st[k] for k in ('pg_loss', 'baseline_loss', 'entropy_loss', 'total_loss', 'grad_norm')])
            for k, v in L.model.state_dict().items():
                g[p + 'param_' + k] = _samp(v.reshape(-1)).numpy().copy()
    return g


def main():
    torch.set_num_threads(8)
    vtrace = _load('ref_vtrace', f'{REF}/impala/vtrace.py')
    loss_fn = _load('ref_loss_fn', f'{REF}/impala/loss_fn.py')
    atari_model = _load('ref_atari_model', f'{REF}/utils/atari_model.py')
    out_dir = os.path.join(ROOT, 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)

    # ---------------- V-trace known-answer vectors (vtrace.py:78-172) ----------------
    vt = {}
    cases = [(5, 3, 1.0, 1.0, 0), (20, 32, 1.0, 1.0, 1), (20, 7, None, None, 2), (33, 5, 2.0, 0.5, 3),
             (100, 4, 1.0, 1.0, 4), (1, 1, 1.0, 1.0, 5), (64, 2, 1.0, None, 6)]
    for i, (T, B, cr, cp, seed) in enumerate(cases):
        rng = np.random.RandomState(seed)
        log_rhos = (rng.randn(T, B) * 0.7).astype(np.float32)
        discounts = ((rng.rand(T, B) > 0.1) * 0.99).astype(np.float32)
        rewards = rng.randn(T, B).astype(np.float32)
        values = rng.randn(T, B).astype(np.float32)
        boot = rng.randn(B).astype(np.float32)
        r = vtrace.from_importance_weights(torch.from_numpy(log_rhos), torch.from_numpy(discounts),
                                           torch.from_numpy(rewards), torch.from_numpy(values),
                                           torch.from_numpy(boot), clip_rho_threshold=cr, clip_pg_rho_threshold=cp)
        vt[f'c{i}_meta'] = np.array([T, B, -1 if cr is None else cr, -1 if cp is None else cp, seed], dtype=np.float64)
        for k, v in dict(log_rhos=log_rhos, discounts=discounts, rewards=rewards, values=values, boot=boot,
                         vs=r.vs.numpy(), pg=r.pg_advantages.numpy()).items():
            vt[f'c{i}_{k}'] = v
    np.savez_compressed(os.path.join(out_dir, 'vtrace_cases.npz'), **vt)

    # ---------------- whole learn() step through the reference modules ----------------
    step_cases = [dict(name='t5b4a6', T=5, B=4, A=6, seed=0, reward_clipping='abs_one', steps=2),
                  dict(name='t3b5a4', T=3, B=5, A=4, seed=1, reward_clipping='none', steps=1)]
    for c in step_cases:
        T, B, A = c['T'], c['B'], c['A']
        hp = dict(O.DEFAULT_HP, reward_clipping=c['reward_clipping'])
        params = O.init_params(A, seed=c['seed'])
        model = atari_model.AtariNet((4, 84, 84), A, use_lstm=False)
        model.load_state_dict(params)
        model.train()
        opt = torch.optim.RMSprop(model.parameters(), lr=hp['learning_rate'], momentum=hp['momentum'],
                                  eps=hp['epsilon'], alpha=hp['alpha'])            # impala_atari.py:99-105
        g = {}
        for step in range(c['steps']):
            batch = O.synthetic_batch(T, B, A, seed=c['seed'] * 10 + step)
            torch.manual_seed(0)
            learner_outputs, _ = model(batch, ())                                  # :289
            bootstrap_value = learner_outputs['baseline'][-1]                      # :293
            b1 = {k: t[1:] for k, t in batch.items()}                              # :296
            lo = {k: t[:-1] for k, t in learner_outputs.items()}                   # :297-300
            rewards = b1['reward']
            clipped = torch.clamp(rewards, -1, 1) if hp['reward_clipping'] == 'abs_one' else rewards
            discounts = (~b1['done']).float() * hp['discounting']                  # :308
            vr = vtrace.from_logits(behavior_policy_logits=b1['policy_logits'],
                                    target_policy_logits=lo['policy_logits'], actions=b1['action'],
                                    discounts=discounts, rewards=clipped, values=lo['baseline'],
                                    bootstrap_value=bootstrap_value)               # :310-318
            pg_loss = loss_fn.compute_policy_gradient_loss(lo['policy_logits'], b1['action'], vr.pg_advantages)
            baseline_loss = hp['baseline_cost'] * loss_fn.compute_baseline_loss(vr.vs - lo['baseline'])
            entropy_loss = hp['entropy_cost'] * loss_fn.compute_entropy_loss(lo['policy_logits'])
            total_loss = pg_loss + baseline_loss + entropy_loss                    # :330
            opt.zero_grad()
            total_loss.backward()                                                  # :343
            grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
            gn = torch.nn.utils.clip_grad_norm_(model.parameters(), hp['max_grad_norm'])  # :344
            opt.step()                                                             # :346
            s = f's{step}_'
            g[s + 'policy_logits'] = learner_outputs['policy_logits'].detach().numpy()
            g[s + 'baseline'] = learner_outputs['baseline'].detach().numpy()
            g[s + 'vs'] = vr.vs.numpy()
            g[s + 'pg_advantages'] = vr.pg_advantages.numpy()
            g[s + 'log_rhos'] = vr.log_rhos.detach().numpy()
            g[s + 'losses'] = np.array([pg_loss.item(), baseline_loss.item(), entropy_loss.item(), total_loss.item()])
            g[s + 'grad_norm'] = np.array([float(gn)])
            for k, v in grads.items():
                flat = v.reshape(-1).double()
                g[s + 'gradnorm_' + k] = np.array([float(flat.norm())])
                g[s + 'gradsum_' + k] = np.array([float(flat.sum())])
                g[s + 'gradhead_' + k] = v.reshape(-1)[:64].numpy().copy()
                # a strided sample across the whole tensor
                idx = torch.linspace(0, flat.numel() - 1, steps=min(257, flat.numel())).long()
                g[s + 'gradsamp_' + k] = v.reshape(-1)[idx].numpy().copy()
            for k, p in model.named_parameters():
                flat = p.detach().reshape(-1)
                idx = torch.linspace(0, flat.numel() - 1, steps=min(257, flat.numel())).long()
                g[s + 'param_' + k] = flat[idx].numpy().copy()
                g[s + 'paramsum_' + k] = np.array([float(flat.double().sum())])
        g['meta'] = np.array([T, B, A, c['seed'], c['steps'], 1 if c['reward_clipping'] == 'abs_one' else 0])
        np.savez_compressed(os.path.join(out_dir, f"learn_{c['name']}.npz"), **g)
        print('wrote', c['name'], 'total_loss', float(total_loss))

    # ---------------- LSTM core through the reference AtariNet(use_lstm=True) (atari_model.py:52-55,109-120) ----------------
    T, B, A = 4, 3, 6
    params = O.init_params(A, seed=2)
    lp = O.init_lstm_params(A, seed=2)
    model = atari_model.AtariNet((4, 84, 84), A, use_lstm=True)
    model.load_state_dict({**params, **lp})
    model.train()
    batch = O.synthetic_batch(T, B, A, seed=42, done_p=0.25)
    rng = np.random.RandomState(5)
    state = (torch.from_numpy(rng.randn(2, B, 513 + A).astype(np.float32) * 0.3), torch.from_numpy(rng.randn(2, B, 513 + A).astype(np.float32) * 0.3))
    torch.manual_seed(0)
    out, new_state = model(batch, state)
    baseline = out['baseline']
    tl, tv = out['policy_logits'][:-1], baseline[:-1]
    b1 = {k: t[1:] for k, t in batch.items()}
    discounts = (~b1['done']).float() * 0.99
    vr = vtrace.from_logits(behavior_policy_logits=b1['policy_logits'], target_policy_logits=tl, actions=b1['action'], discounts=discounts,
                            rewards=torch.clamp(b1['reward'], -1, 1), values=tv, bootstrap_value=baseline[-1])
    total = (loss_fn.compute_policy_gradient_loss(tl, b1['action'], vr.pg_advantages) + 0.5 * loss_fn.compute_baseline_loss(vr.vs - tv) +
             0.0006 * loss_fn.compute_entropy_loss(tl))
    model.zero_grad()
    total.backward()
    g = {'policy_logits': out['policy_logits'].detach().numpy(), 'baseline': baseline.detach().numpy(), 'vs': vr.vs.numpy(),
         'h_out': new_state[0].detach().numpy(), 'c_out': new_state[1].detach().numpy(), 'total_loss': np.array([total.item()]),
         'state_h': state[0].numpy(), 'state_c': state[1].numpy(), 'meta': np.array([T, B, A, 2, 42])}
    for k, p_ in model.named_parameters():
        flat = p_.grad.detach().reshape(-1)
        idx = torch.linspace(0, flat.numel() - 1, steps=min(257, flat.numel())).long()
        g['gradsamp_' + k] = flat[idx].numpy().copy()
        g['gradnorm_' + k] = np.array([float(flat.double().norm())])
    np.savez_compressed(os.path.join(out_dir, 'lstm_t4b3a6.npz'), **g)
    print('wrote lstm_t4b3a6 total_loss', total.item())

    # ---------------- prioritized replay: the reference's own tree classes driven by the statements of
    # PrioritizedReplayBuffer._add / update_priorities / _sample_proprtional / _calculate_weight (replay_buffer.py:318-381);
    # `retrieve` (missing upstream) -> find_prefixsum_idx ----------------
    seg = _load('ref_segment_tree', '/root/reference/scalerl/data/segment_tree.py')
    per = {}
    for ci, (mem, alpha, beta, nadd, batch, seed) in enumerate([(100, 0.6, 0.4, 100, 32, 0), (1000, 0.7, 0.5, 700, 64, 1), (64, 0.6, 1.0, 200, 16, 2)]):
        cap = 1
        while cap < mem:
            cap *= 2
        st, mt = seg.SumSegmentTree(cap), seg.MinSegmentTree(cap)
        rng = np.random.RandomState(seed)
        max_p, ptr, size = 1.0, 0, 0
        for _ in range(nadd):
            st[ptr] = max_p ** alpha
            mt[ptr] = max_p ** alpha
            ptr = (ptr + 1) % mem
            size = min(size + 1, mem)
        upd_idx = rng.randint(0, size, size=3 * batch)
        upd_p = rng.rand(3 * batch) * 5 + 1e-3
        for i, pr in zip(upd_idx, upd_p):
            st[int(i)] = float(pr) ** alpha
            mt[int(i)] = float(pr) ** alpha
            max_p = max(max_p, float(pr))
        for _ in range(5):                                   # adds after updates use the new max priority
            st[ptr] = max_p ** alpha
            mt[ptr] = max_p ** alpha
            ptr = (ptr + 1) % mem
            size = min(size + 1, mem)
        u = rng.rand(batch)
        p_total = st.sum(0, size - 1)
        segment = p_total / batch
        idxs = []
        for i in range(batch):
            a, b = segment * i, segment * (i + 1)
            idxs.append(st.find_prefixsum_idx(a + (b - a) * float(u[i])))
        p_min = mt.min() / st.sum()
        max_w = (p_min * size) ** (-beta)
        w = [((st[i] / st.sum()) * size) ** (-beta) / max_w for i in idxs]
        per[f'c{ci}_meta'] = np.array([mem, alpha, beta, nadd, batch, seed, size, max_p], dtype=np.float64)
        per[f'c{ci}_upd_idx'], per[f'c{ci}_upd_p'], per[f'c{ci}_u'] = upd_idx.astype(np.int64), upd_p, u
        per[f'c{ci}_idxs'], per[f'c{ci}_w'] = np.array(idxs, dtype=np.int64), np.array(w, dtype=np.float64)
        per[f'c{ci}_sum_root'], per[f'c{ci}_min_root'] = np.array([st.sum()]), np.array([mt.min()])
    np.savez_compressed(os.path.join(out_dir, 'per_cases.npz'), **per)
    print('wrote per_cases')

    np.savez_compressed(os.path.join(out_dir, 'reference_cases.npz'), **reference_cases(vtrace, loss_fn, atari_model))
    print('wrote reference_cases')


if __name__ == '__main__':
    main()
