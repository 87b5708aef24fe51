"""In-graph timeline of one learner step (which kernel started when, when its predecessor had completed).  Needs a diagnostics build:
    SRL_DEFINES=SRL_KSTAMP python -m scalerl_b200.build --force && python tests/diag/diag_timeline.py 20 32 ; python -m scalerl_b200.build --force
Every kernel's thread (0,0) appends {id, t_entry, t_after_griddepcontrol.wait}; with the step replayed as ONE CUDA graph (the measured
configuration) `t_after_wait` of kernel k+1 on the main chain is the moment kernel k was complete."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch                                    # noqa: E402
from oracle import impala_oracle as O           # noqa: E402
from scalerl_b200 import _lib                   # noqa: E402
from scalerl_b200.learner import B200ImpalaLearner, ImpalaHParams   # noqa: E402

NAMES = {1: 'obs_s2d', 2: 'pack_weights', 11: 'conv1_fwd', 12: 'conv2_fwd', 13: 'conv3_fwd', 14: 'conv3_dgrad', 15: 'conv2_dgrad',
         21: 'conv3_wgrad', 22: 'conv2_wgrad', 23: 'conv1_wgrad', 31: 'fc_fwd', 32: 'fc_dgrad', 33: 'fc_wgrad', 34: 'lstm_gemm_k', 35: 'lstm_gemm_mn', 36: 'fc_wgrad',
         41: 'column_step', 44: 'impala_tail', 45: 'impala_tail_warp', 46: 'head_fwd', 47: 'head_bwd_dh', 48: 'head_wgrad', 51: 'conv_wgrad_finalize',
         52: 'clip_optim', 53: 'a3_transpose'}
T, B = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (20, 32)
A = 6
L = B200ImpalaLearner(ImpalaHParams(rollout_length=T, batch_size=B, num_actions=A), init_state_dict=O.init_params(A, seed=1), process_group=False)
batch = {k: v.cuda() for k, v in O.synthetic_batch(T, B, A, seed=2).items()}
for _ in range(5):
    L.learn(batch)                               # warm-up: the graph is captured and replayed
torch.cuda.synchronize()
buf = torch.zeros(1 + 3 * 2000, dtype=torch.int64, device='cuda')
_lib.check(L._L.srl_debug_kernel_timeline(buf.data_ptr()), 'timeline')
STEPS = 4
for _ in range(STEPS):
    L.learn(batch)
torch.cuda.synchronize()
_lib.check(L._L.srl_debug_kernel_timeline(None), 'timeline off')
h = buf.cpu().tolist()
n = min(h[0], 2000)
ev = sorted(((h[2 + 3 * i], h[3 + 3 * i], h[1 + 3 * i]) for i in range(n)), key=lambda e: e[1])
per = n // STEPS
last = ev[-per:]                                 # the last replay
t0 = min(e[0] for e in last)
print(f'{n} kernel starts over {STEPS} replays ({per} per step); last step, us relative to its first kernel entry:')
print(f'{"kernel":22s} {"entry":>8s} {"pred. done":>10s}   (kernel k+1 of the main chain "pred. done" = kernel k complete)')
for a, b, kid in sorted(last, key=lambda e: e[1]):
    print(f'{NAMES.get(kid, kid):22s} {(a - t0) / 1e3:8.2f} {(b - t0) / 1e3:10.2f}')
first_prev = min(e[0] for e in ev[-2 * per:-per]) if n >= 2 * per else None
if first_prev is not None:
    print(f'step period (first entry to first entry): {(t0 - first_prev) / 1e3:.2f} us')
