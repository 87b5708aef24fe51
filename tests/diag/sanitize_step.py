"""One small learner step of every kernel family, eager launches -- the workload for compute-sanitizer (tools/sanitize.sh):
    compute-sanitizer --tool memcheck|racecheck|synccheck|initcheck python tests/diag/sanitize_step.py [mode ...]
modes: bf16 (default step), split (fp32-accurate operands), three (no column fusion), lstm, ops"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch                                    # noqa: E402
from oracle import impala_oracle as O           # noqa: E402  (input generator only)
from scalerl_b200 import ops                    # noqa: E402
from scalerl_b200.learner import B200ImpalaLearner, ImpalaHParams   # noqa: E402


def step(tag, T=3, B=5, A=6, state=False, **kw):
    opts = kw.pop('opts', {})
    L = B200ImpalaLearner(ImpalaHParams(rollout_length=T, batch_size=B, num_actions=A, **kw), process_group=False, use_graph=False, seed=1)
    for k, v in opts.items():
        L.set_option(k, v)
    batch = {k: v.cuda() for k, v in O.synthetic_batch(T, B, A, seed=3, done_p=0.2).items()}
    st = tuple(torch.zeros(2, B, 513 + A, device='cuda') for _ in range(2)) if state else ()
    for _ in range(2):
        s = L.learn(batch, st)
    torch.cuda.synchronize()
    print(f'{tag}: total_loss {s["total_loss"]:.5f} grad_norm {s["grad_norm"]:.4f}', flush=True)
    L.close()


def main():
    modes = sys.argv[1:] or ['bf16', 'split', 'three', 'lstm', 'ops']
    if 'bf16' in modes:
        step('bf16')
        step('bf16 adam', optimizer='adam')
    if 'split' in modes:
        step('fp32_split', precision='fp32_split')
    if 'three' in modes:
        step('three-kernel tail', opts={'column_fusion': 0})
    if 'lstm' in modes:
        step('lstm', use_lstm=True, state=True)
    if 'ops' in modes:
        g = torch.Generator(device='cuda').manual_seed(0)
        T, B, A = 7, 33, 6
        r = lambda *s: torch.randn(*s, device='cuda', generator=g)
        for variant in (0, 1):
            ops.from_importance_weights(r(T, B) * .3, torch.full((T, B), 0.99, device='cuda'), r(T, B), r(T, B), r(B), variant=variant)
        lg = r(T, B, A).requires_grad_(True)
        act = torch.randint(0, A, (T, B), device='cuda', generator=g)
        out = ops.from_logits(r(T, B, A), lg, act, torch.full((T, B), 0.99, device='cuda'), r(T, B), r(T, B), r(B))
        loss = ops.compute_policy_gradient_loss(lg, act, out.pg_advantages) + 0.01 * ops.compute_entropy_loss(lg) + ops.compute_baseline_loss(out.vs)
        loss.backward()
        torch.cuda.synchronize()
        print('ops: ok', float(loss), flush=True)


if __name__ == '__main__':
    main()
