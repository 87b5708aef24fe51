"""diagnostic: is forward_backward repeatable (per tensor) with / without shared-memory poisoning; conv1.bias vs sum(da1)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from oracle import impala_oracle as O
from scalerl_b200 import _lib
from scalerl_b200.learner import B200ImpalaLearner, ImpalaHParams

T, B, A = int(sys.argv[1]), int(sys.argv[2]), 4
N = int(sys.argv[3]) if len(sys.argv) > 3 else 6
params = O.init_params(A, seed=1)
L = B200ImpalaLearner(ImpalaHParams(rollout_length=T, batch_size=B, num_actions=A), init_state_dict=params, process_group=False)
batch = {k: v.cuda() for k, v in O.synthetic_batch(T, B, A, seed=5).items()}
gs, d1 = [], []
ctx = torch.cuda.stream(torch.cuda.Stream()) if os.environ.get('DIAG_STREAM') else torch.cuda.stream(torch.cuda.current_stream())
with ctx:
    for it in range(N):
        if it in (1, 3):
            _lib.check(_lib.lib().srl_test_poison_smem(None)); torch.cuda.synchronize()
        L.forward_backward(batch); torch.cuda.synchronize()
        gs.append({k: v.clone() for k, v in L.grads.items()})
        da1 = L.debug_buffer('da1').float().view(-1, 32)
        d1.append(da1.sum(0).clone())
        torch.cuda.synchronize()
tag = 'PDL=%s MASK=%s STREAM=%s' % tuple(os.environ.get(k, '-') for k in ('SRL_PDL', 'SRL_PDL_MASK', 'DIAG_STREAM'))
nbad = 0
for it in range(N):
    bad = {k: float((gs[it][k] - gs[0][k]).norm() / gs[0][k].norm()) for k in gs[0]}
    b = gs[it]['conv1.bias']
    e = float((b - d1[it]).norm() / d1[it].norm())
    nbad += int(e > 1e-4 or any(v > 1e-5 for v in bad.values()))
    if N > 8 and e < 1e-4:
        continue
    print(tag, 'run', it, {k: '%.1e' % v for k, v in bad.items() if v > 1e-6}, 'b1 vs sum(da1) %.1e' % e,
          'da1 stable %.1e' % float((d1[it] - d1[0]).norm() / d1[0].norm()),
          'ratio', [round(float(x), 3) for x in (b / d1[it])[:8]] if e > 1e-3 else '')
print(tag, T, B, 'bad runs', nbad, 'of', N)
