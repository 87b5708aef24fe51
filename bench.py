#!/usr/bin/env python
"""bench.py -- IMPALA learner frames/s on synthetic 84x84x4 uint8 trajectories (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one full learner step (ImpalaTrainer.learn, impala_atari.py:288-346): encoder forward over
(T+1)*B frames, fused V-trace + losses + head gradients, full backward over T*B frames, [NCCL SUM all-reduce],
clip_grad_norm_ + RMSprop, weight re-pack.  The metric counts T*B frames per step (impala_atari.py:391).
Workload: BASELINE.json configs[1] (T=20, B=32 columns per GPU, A=6 Pong) -- weak scaling: every rank keeps 32
columns, global batch = 32*N.

Printed JSON (one line, rank 0):
  value     device-resident whole-job frames/s (inputs already in HBM), CUDA events, max over ranks
  e2e       same metric through the reference-facing API, ImpalaTrainer.get_batch + ImpalaTrainer.learn (impala_atari.py:222-349):
            every step copies its batch from the pinned shared-memory trajectory ring to the device, runs the learner step,
            reads the step's stats back and publishes the new weights (6.75 MB D2H) into the shared actor parameters -- all
            inside the timed region (e2e.feeder_* keeps round 1's HostBatchFeeder loop for comparison)
  roofline  dominant kernel of the step: algorithmic FLOPs per launch / per-launch duration (CUDA events recorded
            around every launch, srl_learner_set_profiling) vs MEASURED_PEAKS.json
  cpu_baseline  the oracle port of the reference learner step timed on this box's host cores (rank 0, N=1)
`--impl reference` times that CPU learner alone: the reference's own AtariNet / vtrace / loss_fn modules (oracle/_ref, built by
oracle/make_ref.py in the build container) under the learn() statements of impala_atari.py:288-346 -- the trainer module
itself cannot be imported (SURVEY.md §0); without oracle/_ref the arm falls back to the oracle port and says so (kind).
`--dump-outputs DIR` writes what the last timed step computed (step_outputs) as DIR/<name>.npy, float32.  That step starts from the
seeded initial weights and a zero optimizer state and reads a seeded batch, so two builds run with the same arguments can be compared
output for output (to the rounding of fp32 atomics).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree, which may be read-only (no __pycache__ either)
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_DEFAULT, B_DEFAULT, A_DEFAULT = 20, 32, 6
POOL = 8   # distinct batches cycled through: 8 x 19.5 MB = 156 MB > 126 MB L2, so a step's inputs are never L2-resident

# algorithmic MACs per frame (SURVEY.md §8a): conv1, conv2, conv3, fc
MACS = {'conv1': 3276800, 'conv2': 2654208, 'conv3': 1806336, 'fc': 1605632, 'conv1+conv2': 3276800 + 2654208}
# Algorithmic HBM bytes per frame of each GEMM kernel: every operand read once and every result written once at the
# storage precision (bf16 activations / gradients; xs = space-to-depth frame 21x21x64, a1 20x20x32, a2 9x9x64,
# a3 7x7x64, h 512).  The dgrads also read the forward activation for the ReLU mask.  (fixed bytes: weights.)
_XS, _A1, _A2, _A3, _H = 28224 * 2, 12800 * 2, 5184 * 2, 3136 * 2, 512 * 2
SLOT_BYTES = {   # slot -> (bytes per frame, fixed bytes per launch)
    'conv1_fwd': (_XS + _A1, 8192 * 2), 'conv2_fwd': (_A1 + _A2, 32768 * 2), 'conv3_fwd': (_A2 + _A3, 36864 * 2),
    'fc_fwd': (_A3 + 512 * 4, 1605632 * 2), 'fc_dgrad': (_H + 2 * _A3, 1605632 * 2), 'fc_wgrad': (_H + _A3, 1605632 * 4),
    'conv3_dgrad': (_A3 + 2 * _A2, 36864 * 2), 'conv3_wgrad': (_A2 + _A3, 36864 * 4),
    'conv2_dgrad': (_A2 + 2 * _A1, 32768 * 2), 'conv2_wgrad': (_A1 + _A2, 32768 * 4), 'conv1_wgrad': (_XS + _A1, 8192 * 4),
    # fused front (u8 frame -> space-to-depth -> conv1 -> conv2): reads the u8 frame once, writes xs / a1 (for the backward) and a2
    'enc_fused_fwd': (28224 + _XS + _A1 + _A2, (8192 + 32768) * 4)}
SLOT_FLOPS = {  # slot -> (MACs per frame, frames = 'fwd' (T+1)*B or 'bwd' T*B)
    'conv1_fwd': ('conv1', 'fwd'), 'conv2_fwd': ('conv2', 'fwd'), 'conv3_fwd': ('conv3', 'fwd'), 'fc_fwd': ('fc', 'fwd'),
    'fc_wgrad': ('fc', 'bwd'), 'fc_dgrad': ('fc', 'bwd'), 'conv3_wgrad': ('conv3', 'bwd'), 'conv3_dgrad': ('conv3', 'bwd'),
    'conv2_wgrad': ('conv2', 'bwd'), 'conv2_dgrad': ('conv2', 'bwd'), 'conv1_wgrad': ('conv1', 'bwd'), 'enc_fused_fwd': ('conv1+conv2', 'fwd')}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_sustained=d.get('bf16_tflops_sustained'), source='measured')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {'sm_mhz': med, 'sm_max_mhz': mx, 'samples': len(sm), 'reasons': sorted(reasons)}


def workload_config(T, B, A, world, use_lstm=False):
    """the workload both arms run -- identical dict in the b200 and the reference line (the driver compares them)"""
    return {'workload': f'IMPALA Pong 84x84x4 uint8, T={T}, B={B}/GPU, A={A}, synthetic trajectories (BASELINE.json configs[1] per GPU)',
            'rollout_length': T, 'columns_per_gpu': B, 'global_batch': B * world, 'num_actions': A, 'optimizer': 'rmsprop',
            'use_lstm': bool(use_lstm), 'reward_clipping': 'abs_one', 'discounting': 0.99, 'baseline_cost': 0.5, 'entropy_cost': 0.0006,
            'max_grad_norm': 40.0, 'learning_rate': 1e-4}


def make_host_pool(T, B, A, n, seed):
    """n distinct synthetic [T+1,B] batches in pinned host memory (distributions of SURVEY.md §8d)."""
    import numpy as np
    import torch
    from scalerl_b200.data.feeder import pinned_batch
    pool = []
    for i in range(n):
        rng = np.random.RandomState(seed * 1000 + i)
        hb = pinned_batch(T, B, A)
        hb['obs'].copy_(torch.from_numpy(rng.randint(0, 256, size=(T + 1, B, 4, 84, 84), dtype=np.uint8)))
        hb['reward'].copy_(torch.from_numpy(rng.randn(T + 1, B).astype(np.float32)))
        hb['done'].copy_(torch.from_numpy(rng.rand(T + 1, B) < 0.02))
        hb['action'].copy_(torch.from_numpy(rng.randint(0, A, size=(T + 1, B)).astype(np.int64)))
        hb['policy_logits'].copy_(torch.from_numpy(rng.randn(T + 1, B, A).astype(np.float32)))
        hb['episode_return'].copy_(torch.from_numpy(rng.randn(T + 1, B).astype(np.float32)))
        pool.append(hb)
    return pool


DUMP_LIMIT = 64 << 20     # bytes written by --dump-outputs at most


def step_outputs(learner):
    """what one learner step hands its caller: the four losses and the gradient norm of the stats dict, the V-trace targets and
    policy-gradient advantages [T, B], the updated parameters and the step's gradients (AtariNet state_dict names)"""
    r = learner._resdev.cpu().numpy()
    out = {'pg_loss': r[0:1], 'baseline_loss': r[1:2], 'entropy_loss': r[2:3], 'total_loss': r[3:4], 'grad_norm': r[4:5],
           'vs': learner._vs.cpu().numpy(), 'pg_advantages': learner._pg_adv.cpu().numpy()}
    out.update({f'param.{n}': v.cpu().numpy() for n, v in learner.params.items()})
    out.update({f'grad.{n}': v.cpu().numpy() for n, v in learner.grads.items()})
    return out


def dump_outputs(d, arrays):
    """DIR/<name>.npy in float32.  Should the arrays exceed DUMP_LIMIT together, each large one is replaced by the same seeded
    sample of its flattened elements (same sizes and indices in every run with the same arguments)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if total > DUMP_LIMIT and a.size > 4096:
            keep = max(4096, a.size * DUMP_LIMIT // (2 * total))
            a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(d, name + '.npy'), a)


def usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class _CpuLearner:
    """the CPU learner step of the reference: its OWN modules from oracle/_ref (kind "reference") when that build output is
    present, else the oracle port (kind "port")"""

    def __init__(self, T, B, A, use_lstm=False):
        from oracle import impala_oracle as O
        from oracle import ref_learner as R
        self.O = O
        self.params = O.init_params(A, seed=0)
        self.batch = O.synthetic_batch(T, B, A, seed=0)
        self.use_lstm = use_lstm
        self.state = ()
        if R.available():
            self.kind = 'reference'
            sd = dict(self.params)
            if use_lstm:
                sd.update(O.init_lstm_params(A, seed=0))
            self.ref = R.ReferenceLearner(A, use_lstm=use_lstm, state_dict=sd)
            if use_lstm:
                import torch
                self.state = tuple(torch.zeros(2, B, 513 + A) for _ in range(2))
        else:
            if use_lstm:
                raise RuntimeError('the LSTM CPU arm needs oracle/_ref (python oracle/make_ref.py)')
            self.kind = 'port'
            self.opt = O.new_opt_state(self.params)

    def step(self):
        if self.kind == 'reference':
            return self.ref.learn(self.batch, self.state)
        return self.O.learn_step(self.params, self.opt, self.batch, use_autograd=True)


def pick_threads(cpu):
    """torch-CPU convs on this small batch do not scale to every core of a 128-core host: try a few intra-op
    thread counts (one step each) and keep the fastest -- the baseline gets its best configuration."""
    import torch
    cores = usable_cores()
    best, best_t = None, None
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(n)
        cpu.step()
        t0 = time.perf_counter()
        cpu.step()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best, cores


def cpu_learner_fps(T, B, A, budget_s, warmup=1, max_steps=50, min_steps=3):
    """the reference's CPU learner step (fp32, autograd, RMSprop) on the host cores"""
    cpu = _CpuLearner(T, B, A)
    cores, avail = pick_threads(cpu)
    for _ in range(warmup):
        cpu.step()
    n, t0 = 0, time.perf_counter()
    while n < max_steps and (n < min_steps or time.perf_counter() - t0 < budget_s):
        cpu.step()
        n += 1
    dt = time.perf_counter() - t0
    return n * T * B / dt, n, dt / n, cores, cpu.kind


def run_reference(args, rank, world, real_stdout):
    if rank != 0:
        return
    T, B, A = args.T, args.B, args.A
    cpu = _CpuLearner(T, B, A, use_lstm=args.use_lstm)
    cores, avail = pick_threads(cpu)
    for _ in range(args.warmup):
        cpu.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu.step()
    dt = time.perf_counter() - t0
    fps = args.steps * T * B / dt
    what = ("the reference's own AtariNet / vtrace / loss_fn modules (oracle/_ref) under the learn() statements of impala_atari.py:288-346"
            if cpu.kind == 'reference' else 'the oracle port of the reference learner step')
    sample = (f'{args.steps} learner steps of T={T}, B={B} columns (one GPU-rank shard of the global batch {B * world}), fp32 torch-CPU, {what}, '
              f'{cores} intra-op threads (fastest of the tried counts; {avail} cores usable)')
    out = {'impl': 'reference', 'metric': 'learner_frames_per_sec', 'value': fps, 'unit': 'frames/s', 'n_gpus': world,
           'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True,
           'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'config': workload_config(T, B, A, world, args.use_lstm),
           'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': cpu.kind, 'sample': sample},
           'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    emit(real_stdout, out)


def main():
    # keep stdout clean for the single JSON line: anything libraries print (NCCL banner, warnings) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main(real_stdout)
    finally:
        os.dup2(real_stdout, 1)


def emit(real_stdout, obj):
    os.write(real_stdout, (json.dumps(obj) + '\n').encode())


def _main(real_stdout):
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--T', type=int, default=T_DEFAULT)
    ap.add_argument('--B', type=int, default=B_DEFAULT, help='columns per GPU')
    ap.add_argument('--A', type=int, default=A_DEFAULT)
    ap.add_argument('--cpu-budget', type=float, default=15.0, help='seconds of CPU-baseline work (rank 0, N=1)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the other_configs / per_sampler measurements')
    ap.add_argument('--publish-every', type=int, default=1, help='weight publish cadence of the end-to-end loop (reference: every step)')
    ap.add_argument('--use-lstm', action='store_true', help='AtariNet(use_lstm=True) learner (BASELINE.json configs[4]: use with --T 100)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed as DIR/<name>.npy (rank 0)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, rank, world, real_stdout)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run --nproc-per-node N for --gpus N > 1')

    import torch
    import torch.distributed as dist
    from scalerl_b200.learner import B200ImpalaLearner, ImpalaHParams
    from scalerl_b200.data.feeder import HostBatchFeeder, H2D_KEYS
    from scalerl_b200 import _lib
    import ctypes as C

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    from scalerl_b200.utils.numa import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local_rank)            # before any pinned allocation: first touch lands on the GPU's node
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    T, B, A, K, W = args.T, args.B, args.A, args.steps, args.warmup
    hp = ImpalaHParams(rollout_length=T, batch_size=B, num_actions=A, use_lstm=args.use_lstm)
    learner = B200ImpalaLearner(hp, device=dev, seed=0)
    init_weights = learner.state_dict() if args.dump_outputs else None       # the seeded initial weights, on the device
    host_pool = make_host_pool(T, B, A, POOL, seed=rank)
    dev_pool = [{k: v.to(dev, non_blocking=True) for k, v in hb.items()} for hb in host_pool]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident throughput ----------------
    for i in range(max(W, 2 * POOL)):          # every pool batch is seen twice: eager warm-up, then graph capture
        learner.learn(dev_pool[i % POOL], sync_stats=False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(K):
        if init_weights is not None and i == K - 1:
            # the dumped step starts from the same state in every run: the gradient kernels sum with fp32 atomics, and over many
            # RMSprop steps their rounding grows into a different trajectory.  The restore is excluded from the timed window.
            r0.record()
            learner.load_state_dict(init_weights)
            learner.opt_state0.zero_()
            r1.record()
        learner.learn(dev_pool[(W + i) % POOL], sync_stats=False)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1) - (r0.elapsed_time(r1) if init_weights is not None else 0.0))
    clocks = sampler.stop() if rank == 0 else None
    frames = K * T * B * world
    value = frames / (ms_total * 1e-3)
    losses_finite = bool(torch.isfinite(learner._losses).all().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_outputs(learner))

    # ---------------- end to end through the host-batch API ----------------
    feeder = HostBatchFeeder(learner, depth=2)
    def e2e_loop(n, off):
        last = None
        feeder.submit(host_pool[off % POOL])
        for i in range(n):
            if i + 1 < n:
                feeder.submit(host_pool[(off + i + 1) % POOL])
            s = feeder.learn()
            if last is not None:
                feeder.result(last)             # D2H read of the previous step's losses (one step behind)
            last = s
        return feeder.result(last)
    e2e_loop(max(W, 6), 0)
    barrier()
    t0 = time.perf_counter()
    stats = e2e_loop(K, W)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        dist.barrier(device_ids=[local_rank])
    e2e_s = max_over_ranks(dt)
    e2e_value = frames / e2e_s
    # diagnostics: the H2D copies alone, and the same loop with eager launches instead of CUDA graphs
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        s_ = feeder.submit(host_pool[i % POOL])
        feeder.ready[s_].synchronize()
        feeder._learned += 1          # slot handed back without a learner step
    h2d_only_ms = (time.perf_counter() - t0) / K * 1e3
    learner.use_graph = False
    e2e_loop(3, 0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_loop(K, W)
    torch.cuda.synchronize()
    e2e_eager_ms = (time.perf_counter() - t0) / K * 1e3
    learner.use_graph = True

    # ---------------- end to end through ImpalaTrainer.get_batch / learn (ring -> device, step, stats, weight publish) ----------------
    import tempfile
    from scalerl_b200.algorithms.impala.impala_atari import ImpalaArguments, ImpalaTrainer
    from scalerl_b200.data.slot_queue import SlotQueue
    targs = ImpalaArguments(num_actors=1, batch_size=B, rollout_length=T, num_buffers=POOL * B, num_actions=A, use_lstm=args.use_lstm,
                            output_dir=tempfile.mkdtemp(prefix='srl_bench_'), disable_checkpoint=True, stats_lag=2, publish_every=args.publish_every)
    trainer = ImpalaTrainer(targs, learner=learner)
    for i, hb in enumerate(host_pool):                      # slot i*B + b = column b of pool batch i (what B actors would have written)
        for b in range(B):
            for k in H2D_KEYS:
                trainer.buffers[k][i * B + b].copy_(hb[k][:, b])
    free_q, full_q = SlotQueue(4 * POOL * B), SlotQueue(4 * POOL * B)

    def trainer_loop(n, off):
        st = None
        for i in range(n):
            base = ((off + i) % POOL) * B
            for b in range(B):
                full_q.put(base + b)
            batch, state = trainer.get_batch(free_q, full_q)
            st = trainer.learn(trainer.actor_model, None, batch, state)
            while not free_q.empty():
                free_q.get_nowait()
        trainer.flush()
        return st
    trainer_loop(max(W, 6), 0)
    barrier()
    trainer.wait_seconds = 0.0
    t0 = time.perf_counter()
    tstats = trainer_loop(K, W)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        dist.barrier(device_ids=[local_rank])
    tr_s = max_over_ranks(dt)
    tr_value = frames / tr_s
    tr_host_ms = (dt - trainer.wait_seconds) / K * 1e3          # host time per step outside the wait for the lagged result
    # diagnostic: the ring -> device DMA alone (one merged copy of B slots from the pinned shared-memory block)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        base = (i % POOL) * B
        trainer._staging[0].view(-1).copy_(trainer.ring.block[base * trainer.ring.slot_bytes:(base + B) * trainer.ring.slot_bytes], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ring_h2d_ms = (time.perf_counter() - t0) / K * 1e3
    tr_h2d = B * trainer.ring.slot_bytes + (trainer._rnn_host[0].numel() * 4 if args.use_lstm else 0)
    tr_d2h = learner.numel * 4 + 8 + (8 * 4 + T * B * 5)       # weight publish + version counter + step result (scalars, episode_return, done)
    published = int(trainer.weights_version[0])

    # ---------------- per-kernel durations (events around every launch) ----------------
    L = _lib.lib()
    _lib.check(L.srl_learner_set_profiling(learner._h, 1))
    nslot = L.srl_profile_slot_count()
    names = [L.srl_profile_slot_name(i).decode() for i in range(nslot)]
    acc = [0.0] * nslot
    buf = (C.c_float * nslot)()
    nprof = min(K, 20)
    if args.use_lstm:
        nprof = 0          # the per-slot event bracketing covers the non-LSTM step only
    for i in range(nprof):
        learner.learn(dev_pool[i % POOL], sync_stats=False, use_graph=False)
        torch.cuda.synchronize()
        _lib.check(L.srl_learner_profile_collect(learner._h, buf))
        for j in range(nslot):
            acc[j] += max(0.0, buf[j])
    nprof = max(nprof, 1)
    _lib.check(L.srl_learner_set_profiling(learner._h, 0))
    per_kernel_ms = {names[j]: acc[j] / nprof for j in range(nslot)}
    pk = peaks()
    NF, NBk = (T + 1) * B, T * B
    gemm = {}
    ridge = pk['bf16_tflops'] * 1e12 / (pk['hbm_gbs'] * 1e9)         # flop/byte above which a kernel can be tensor-bound
    for slot, (layer, which) in SLOT_FLOPS.items():
        nfr = NF if which == 'fwd' else NBk
        fl = 2.0 * MACS[layer] * nfr
        by = SLOT_BYTES[slot][0] * nfr + SLOT_BYTES[slot][1]
        ms = per_kernel_ms.get(slot, 0.0)
        gemm[slot] = {'ms': ms, 'gflop': fl / 1e9, 'tflops': fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0, 'bytes': by,
                      'gbs': by / (ms * 1e-3) / 1e9 if ms > 0 else 0.0, 'intensity': fl / by,
                      'bound': 'tensor' if fl / by >= ridge else 'hbm'}
    # dominant kernel = the longest GEMM on the step's critical chain (fc/conv3/conv2 wgrad run on side branches beside it)
    CHAIN = ('enc_fused_fwd', 'conv1_fwd', 'conv2_fwd', 'conv3_fwd', 'fc_fwd', 'fc_dgrad', 'conv3_dgrad', 'conv2_dgrad', 'conv1_wgrad')
    dom = max(CHAIN, key=lambda s: gemm[s]['ms'])
    traffic, traffic_src, tensor_pct = None, None, None
    tp = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(tp) and (T, B) == (T_DEFAULT, B_DEFAULT):      # the ncu capture was taken at the default workload
        tj = json.load(open(tp))
        if dom in tj['kernels']:
            traffic = tj['kernels'][dom]['dram_bytes_per_launch']
            tensor_pct = tj['kernels'][dom]['tensor_pipe_active_pct']
            traffic_src = tj['source']
    step_flops = NF * 18.693e6 + NBk * 30.833e6
    if args.use_lstm:     # 2 layers x (Wih + Whh) x 4H x H MACs per frame forward; backward = dX/dh + dW (2x)
        Hh = 513 + A
        step_flops += NF * 2 * (2 * 2 * 4 * Hh * Hh) + NBk * 2 * 2 * (2 * 2 * 4 * Hh * Hh)
    sum_kernel_ms = sum(per_kernel_ms.values())
    d = gemm[dom]
    hbm_bound = d['bound'] == 'hbm'
    roofline = {'bound': d['bound'], 'kernel': dom,
                'achieved': d['gbs'] if hbm_bound else d['tflops'], 'peak': pk['hbm_gbs'] if hbm_bound else pk['bf16_tflops'],
                'unit': 'GB/s' if hbm_bound else 'TFLOP/s',
                'frac': d['gbs'] / pk['hbm_gbs'] if hbm_bound else d['tflops'] / pk['bf16_tflops'],
                'traffic': traffic, 'traffic_unit': 'bytes (dram read+write per launch)',
                'traffic_source': traffic_src, 'ncu_tensor_pipe_active_pct': tensor_pct,
                'peak_source': pk['source'] + (' HBM copy bandwidth' if hbm_bound else ' burst bf16') + ' (MEASURED_PEAKS.json)',
                'dominant_rule': 'longest GEMM launch on the critical chain of the step graph (side-branch wgrads overlap it; all kernels in per_gemm)',
                'bound_why': f"arithmetic intensity {d['intensity']:.0f} flop/B (algorithmic) vs ridge {ridge:.0f} flop/B "
                             f"(measured bf16 peak / measured HBM peak)",
                'algorithmic_bytes_per_launch': d['bytes'], 'flops_per_launch': d['gflop'] * 1e9, 'ms_per_launch': d['ms'],
                'tensor_view': {'achieved_tflops': d['tflops'], 'frac_of_bf16_peak': d['tflops'] / pk['bf16_tflops']},
                'how': f'CUDA events around each launch on the launch stream, mean of {nprof} steps after the timed region',
                'step': {'gflop': step_flops / 1e9, 'tflops_device_resident': step_flops / (ms_total / K * 1e-3) / 1e12,
                         'frac_of_peak': step_flops / (ms_total / K * 1e-3) / 1e12 / pk['bf16_tflops'], 'sum_kernel_ms': sum_kernel_ms},
                'per_kernel_ms': {k: round(v, 5) for k, v in per_kernel_ms.items()},
                'per_gemm': {k: {'tflops': round(v['tflops'], 1), 'gbs': round(v['gbs'], 0), 'flop_per_byte': round(v['intensity'], 0),
                                 'bound': v['bound']} for k, v in gemm.items()}}

    # ---------------- stand-alone V-trace kernel: GB/s vs measured HBM peak (BASELINE.json metric, second half) ----------------
    # Kernel-only: a CUDA graph of 100 C-ABI launches on preallocated buffers, CUDA events around the replay -> time per launch
    # INCLUDING the ~1-2 us between dependent graph nodes (a lone launch cannot be timed finer with events).  At the spec size
    # (T=20,B=512: 248 KB) the inputs are L2-resident and the kernel is latency-bound; the bandwidth-regime rows rotate inputs > L2.
    vtrace = None
    if rank == 0:
        Lc = _lib.lib()
        vtrace = {}
        for (vt, vb, variant) in ((20, 512, 1), (20, 512, 0), (100, 128, 1), (100, 128, 0), (20, 1 << 20, 0), (20, 1 << 22, 0)):
            g = torch.Generator(device=dev).manual_seed(1)
            big = vb >= (1 << 18)
            nrot = max(2, int(200e6 // (24 * vt * vb)) + 1) if big else 1          # rotate > L2 worth of inputs at the large sizes
            sets = [[torch.randn(vt, vb, device=dev, generator=g) * 0.5, (torch.rand(vt, vb, device=dev, generator=g) > 0.02).float() * 0.99,
                     torch.randn(vt, vb, device=dev, generator=g), torch.randn(vt, vb, device=dev, generator=g),
                     torch.randn(vb, device=dev, generator=g)] for _ in range(nrot)]
            o_vs, o_pg = torch.empty(vt, vb, device=dev), torch.empty(vt, vb, device=dev)

            def launch(i):
                a = sets[i % nrot]
                _lib.check(Lc.srl_vtrace_from_importance_weights(a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), a[3].data_ptr(), a[4].data_ptr(),
                                                                 vt, vb, 1.0, 1.0, o_vs.data_ptr(), o_pg.data_ptr(), variant,
                                                                 torch.cuda.current_stream().cuda_stream), 'vtrace')
            nl = 20 if big else 100
            for i in range(3):
                launch(i)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for i in range(nl):
                    launch(i)
            gr.replay()
            torch.cuda.synchronize()
            a_ev, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            a_ev.record()
            for _ in range(reps):
                gr.replay()
            b_ev.record()
            torch.cuda.synchronize()
            ms = a_ev.elapsed_time(b_ev) / (reps * nl)
            nbytes = 24 * vt * vb + 4 * vb
            vtrace[f'T{vt}_B{vb}_{"scan" if variant else "seq"}'] = {
                'us': ms * 1e3, 'algorithmic_bytes': nbytes, 'GBps': nbytes / (ms * 1e-3) / 1e9,
                'frac_of_hbm_peak': nbytes / (ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                'how': f'CUDA graph of {nl} srl_vtrace_from_importance_weights launches, events around {reps} replays; '
                       + ('inputs rotate through > L2 worth of buffers' if big else 'inputs L2-resident (spec size)')}
            del gr

    # ---------------- CPU baseline (rank 0, N=1) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps, n, s_per, cores, kind = cpu_learner_fps(T, B, A, args.cpu_budget)
        cpu = {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
               'sample': f'{n} full learner steps of the same workload (T={T}, B={B}, fp32 torch-CPU autograd + RMSprop; '
                         + ("the reference's own modules from oracle/_ref" if kind == 'reference' else 'oracle port') + f'), {s_per * 1e3:.1f} ms/step'}

    # ---------------- further BASELINE.json configurations, measured in the same run (short, device-resident) ----------------
    def short_run(hp2, steps=10, warm=6, pool=3):
        """ms/step of a second learner configuration (weak-scaling shard of this rank), device-resident, max over ranks"""
        L2 = B200ImpalaLearner(hp2, device=dev, seed=0)
        hp_ = make_host_pool(hp2.rollout_length, hp2.batch_size, hp2.num_actions, pool, seed=100 + rank)
        dp_ = [{k: v.to(dev, non_blocking=True) for k, v in hb.items()} for hb in hp_]
        st_ = ()
        if hp2.use_lstm:
            st_ = tuple(torch.zeros(2, hp2.batch_size, 513 + hp2.num_actions, device=dev) for _ in range(2))
        for i in range(max(warm, 2 * pool)):
            L2.learn(dp_[i % pool], st_, sync_stats=False)
        barrier()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record()
        for i in range(steps):
            L2.learn(dp_[i % pool], st_, sync_stats=False)
        b_.record()
        barrier()
        ms_ = max_over_ranks(a_.elapsed_time(b_)) / steps
        fin = bool(torch.isfinite(L2._losses).all().item())
        L2.release_graphs()
        L2.close()
        fr = hp2.rollout_length * hp2.batch_size * world
        return {'ms_per_step': ms_, 'frames_per_sec': fr / (ms_ * 1e-3), 'global_batch': hp2.batch_size * world, 'columns_per_gpu': hp2.batch_size,
                'rollout_length': hp2.rollout_length, 'num_actions': hp2.num_actions, 'use_lstm': hp2.use_lstm, 'losses_finite': fin}

    extra_cfg = {}
    if not args.use_lstm and (T, B, A) == (T_DEFAULT, B_DEFAULT, A_DEFAULT) and not args.no_extras:
        try:      # configs[2]: IMPALA Breakout T=20, B=512 over 8 GPUs = 64 columns per GPU, A=4 (global B = 64 N here)
            extra_cfg['config3_breakout_64col'] = short_run(ImpalaHParams(rollout_length=20, batch_size=64, num_actions=4))
        except Exception as e:      # noqa: BLE001
            extra_cfg['config3_breakout_64col'] = {'error': repr(e)}
        if world in (1, 2, 4, 8):
            try:  # configs[4]: IMPALA + LSTM, T=100, global B=128 split over the ranks
                extra_cfg['config5_lstm_T100_B128'] = short_run(ImpalaHParams(rollout_length=100, batch_size=128 // world, num_actions=6, use_lstm=True),
                                                                steps=5, warm=4, pool=2)
            except Exception as e:  # noqa: BLE001
                extra_cfg['config5_lstm_T100_B128'] = {'error': repr(e)}

    # ---------------- configs[3]: GPU prioritized-replay sampler vs the reference's CPU segment trees (rank 0, N=1) ----------------
    per = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            from scalerl_b200.data.per_sampler import GpuPrioritizedSampler
            from oracle import per_oracle as PO
            cap, bsz = 1 << 20, 512
            smp = GpuPrioritizedSampler(cap, alpha=0.6)
            smp.add(cap)
            gidx = torch.randint(0, cap, (bsz,), device=dev)
            gpr = torch.rand(bsz, device=dev, dtype=torch.float64) + 0.01
            for _ in range(3):
                smp.sample(bsz, 0.4); smp.update_priorities(gidx, gpr, validate=False)
            torch.cuda.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nit = 200
            a_.record()
            for _ in range(nit):
                smp.sample(bsz, 0.4); smp.update_priorities(gidx, gpr, validate=False)
            b_.record()
            torch.cuda.synchronize()
            gpu_us = a_.elapsed_time(b_) / nit * 1e3
            cpu_cap = 1 << 16           # the pure-Python trees of the reference are slow: smaller buffer, bounded time
            import numpy as np
            ref_t = PO.PerOracle(cpu_cap, 0.6)      # the reference's tree arithmetic (segment_tree.py / replay_buffer.py) restated on the CPU
            ref_t.add(cpu_cap)
            rng = np.random.RandomState(0)
            t0 = time.perf_counter(); n = 0
            while n < 3 or time.perf_counter() - t0 < 3.0:
                ref_t.sample(rng.rand(bsz), 0.4); ref_t.update_priorities(rng.randint(0, cpu_cap, bsz), rng.rand(bsz) + 0.01); n += 1
            cpu_us = (time.perf_counter() - t0) / n * 1e6
            per = {'batch': bsz, 'gpu_capacity': cap, 'gpu_us_per_sample_plus_update': gpu_us, 'gpu_transitions_per_sec': bsz / (gpu_us * 1e-6),
                   'cpu_capacity': cpu_cap, 'cpu_us_per_sample_plus_update': cpu_us,
                   'cpu_transitions_per_sec': (bsz / (cpu_us * 1e-6)) if cpu_us else None,
                   'what': 'stratified proportional sample of 512 + priority update of 512 (float64 sum/min trees; replay_buffer.py:346-381)'}
            smp.close()
        except Exception as e:      # noqa: BLE001
            per = {'error': repr(e)}

    if rank == 0:
        peer = getattr(learner, '_peers', None) is not None
        cfg = workload_config(T, B, A, world, args.use_lstm)
        impl = {'parallelism': f'dp{world}' if world > 1 else 'single',
                'grad_allreduce': 'none' if world == 1 else ((('NVLS multimem.ld_reduce (in-switch sum)' if getattr(learner, 'dp_path', '') == 'nvls multimem'
                                                                else 'peer memory (NVLink loads)') + ' fused into the clip+optimizer kernel') if peer else 'nccl sum'),
                'l2': f'inputs cycle through {POOL} distinct batches ({POOL * feeder.h2d_bytes / 1e6:.0f} MB > 126 MB L2)',
                'operands': 'bf16 tensor-core operands, fp32 accumulate, fp32 master weights / V-trace / optimizer',
                'launch': 'one CUDA graph per step (wgrad GEMMs on parallel branches, programmatic dependent launch)'
                          if (world == 1 or peer) else 'CUDA graphs begin|finish|apply; NCCL all-reduce of fc.weight overlaps the conv backward',
                'numa': numa}
        # gpu_launches: 18 kernels of this library per step (tests/diag/diag_timeline.py lists them; + 1 memset)
        out = {'metric': 'learner_frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': W,
               'ms_per_step': ms_total / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
               'data': 'synthetic', 'config': cfg, 'impl_details': impl,
               'e2e': {'value': tr_value, 'unit': 'frames/s', 'h2d_bytes_per_step': tr_h2d, 'd2h_bytes_per_step': tr_d2h,
                       'ms_per_step': tr_s / K * 1e3,
                       'api': 'ImpalaTrainer.get_batch + ImpalaTrainer.learn (pinned shared-memory trajectory ring -> device, step, lagged stats, '
                              'asynchronous versioned weight publish into the shared actor parameters)',
                       'weights_published': published, 'last_total_loss': tstats['total_loss'], 'host_ms_per_step': tr_host_ms, 'ring_h2d_only_ms_per_step': ring_h2d_ms,
                       'stats_lag_steps': targs.stats_lag, 'publish_every': targs.publish_every,
                       'feeder_value': e2e_value, 'feeder_ms_per_step': e2e_s / K * 1e3, 'feeder_h2d_bytes_per_step': feeder.h2d_bytes,
                       'feeder_api': 'HostBatchFeeder.submit/learn/result (time-major pinned batches, no ring, no weight publish: round-1 e2e)',
                       'h2d_only_ms_per_step': h2d_only_ms, 'eager_launch_ms_per_step': e2e_eager_ms},
               'gpu_launches': 18 * K, 'clocks': clocks, 'roofline': roofline, 'cpu_baseline': cpu, 'losses_finite': losses_finite,
               'vtrace_standalone': vtrace, 'other_configs': extra_cfg, 'per_sampler': per}
        emit(real_stdout, out)
    trainer.close() if False else None
    learner.release_graphs()
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(device_ids=[local_rank])
        # no destroy_process_group(): tearing NCCL down at interpreter exit has been seen to hang; the JSON line is out,
        # so leave immediately (os._exit skips atexit handlers of the NCCL watchdog)
        os.dup2(real_stdout, 1)
        os._exit(0)


if __name__ == '__main__':
    main()
