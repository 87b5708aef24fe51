"""LSTM core alone (srl_lstm_forward / srl_lstm_backward, one launch pair per step), each replayed as a CUDA graph.
    python tests/diag/diag_lstm_time.py [T1 B A]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch                                    # noqa: E402
from scalerl_b200.lstm import B200LstmCore      # noqa: E402


def main():
    T1, B, A = [int(x) for x in sys.argv[1:4]] if len(sys.argv) >= 4 else (101, 128, 6)
    H = 513 + A
    core = B200LstmCore(T1, B, H, seed=0)
    g = torch.Generator(device='cuda').manual_seed(0)
    x = torch.randn(T1, B, H, device='cuda', generator=g) * 0.5
    done = torch.rand(T1, B, device='cuda', generator=g) < 0.02
    st = (torch.zeros(2, B, H, device='cuda'), torch.zeros(2, B, H, device='cuda'))
    dout = torch.randn(T1 - 1, B, H, device='cuda', generator=g) * 0.1
    gr = torch.cuda.CUDAGraph()
    for _ in range(2):
        out, _ = core.forward(x, done, st)
        core.backward(dout)
    torch.cuda.synchronize()
    res = {}
    for name, fn in (('forward', lambda: core.forward(x, done, st)), ('backward', lambda: core.backward(dout))):
        g1 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g1):
            fn()
        g1.replay(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            g1.replay()
        b.record(); torch.cuda.synchronize()
        res[name] = a.elapsed_time(b) / 5
    print(f'T1={T1} B={B} H={H}: forward {res["forward"]:.3f} ms  backward {res["backward"]:.3f} ms'
          f'  checksum {float(out.double().sum()):.6f} {float(core.grads["rnn_layer.weight_hh_l0"].double().sum()):.6f}')


if __name__ == '__main__':
    main()
