"""linear_tf32 / wgrad_tf32 timing at the encoder's layer shape: python profiles/exp_gemm.py [rows]"""
import importlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
rows = int(sys.argv[1]) if len(sys.argv) > 1 else 65536 * 36
x = torch.randn(rows, 128, device="cuda")
W = torch.randn(128, 128, device="cuda") / 11.3
b = torch.randn(128, device="cuda")
sc, sh = torch.rand(128, device="cuda") + 0.5, torch.randn(128, device="cuda")
gz = torch.randn(rows, 128, device="cuda")


def timeit(fn, n=10):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


z = enc.linear_tf32(x, W, b)
ref = x.double() @ W.double().T + b.double()
err = float((z.double() - ref).abs().max())
gb = rows * 128 * 4 * 2 / 1e9
t_plain = timeit(lambda: enc.linear_tf32(x, W, b))
stats = torch.zeros(256, dtype=torch.float64, device="cuda")
t_aff = timeit(lambda: enc.linear_tf32(x, W, b, sc, sh, relu=True, stats=stats))
t_wg = timeit(lambda: enc.wgrad_tf32(gz, x))
print("rows %d: plain %.1f us (%.2f TB/s, max err %.2e)  affine+stats %.1f us (%.2f TB/s)  wgrad %.1f us (%.2f TB/s)"
      % (rows, t_plain, gb / t_plain * 1e3, err, t_aff, gb / t_aff * 1e3, t_wg, gb / t_wg * 1e3))
