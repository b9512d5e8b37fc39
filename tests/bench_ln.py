"""Not a pytest file: device-timed LayerNorm forward / backward at the encoder's shapes.
    python tests/bench_ln.py [batch]
"""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vitk  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
M, D = B * 197, 768
x = torch.randn(M, D, device="cuda")
g = torch.randn(D, device="cuda")
bta = torch.randn(D, device="cuda")
dy = torch.randn(M, D, device="cuda").bfloat16()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    e = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for e0, e1 in e:
        flush.zero_()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in e)
    return t[len(t) // 2]


y, mean, rstd = vitk.ops.layernorm(x, g, bta, return_stats=True)
ms = timeit(lambda: vitk.ops.layernorm(x, g, bta))
print(f"layernorm fwd  rows={M}: {ms*1e3:7.1f} us  {M*D*6/ms/1e6:7.0f} GB/s")
dx = torch.randn(M, D, device="cuda")
dgam, dbet = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
dxb = torch.empty(M, D, device="cuda", dtype=torch.bfloat16)
st = torch.cuda.current_stream().cuda_stream
ms = timeit(lambda: vitk._lib.check(vitk._lib.lib().vitk_layernorm_bwd(
    dy.data_ptr(), 0, x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), g.data_ptr(), dx.data_ptr(), 1,
    dxb.data_ptr(), dgam.data_ptr(), dbet.data_ptr(), M, D, None, 0.0, 0, 0, 0, st)))
print(f"layernorm bwd rows={M}: {ms*1e3:7.1f} us  {M*D*16/ms/1e6:7.0f} GB/s (algorithmic 16 B/elem)")
