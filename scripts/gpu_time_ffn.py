"""Time the fused FFN kernel vs FF (chunks) to separate fixed overhead from per-chunk cost; check vs torch."""
import sys, torch
import torch.nn.functional as F
sys.path.insert(0, '.')
from ppasr_b200 import _lib as L
lib = L.load(); dev = torch.device('cuda:0'); torch.manual_seed(0)
M = 7936
for FF in (512, 1024, 2048, 4096):
    y = torch.randn(M, 256, device=dev).to(torch.bfloat16)
    w1 = (torch.randn(FF, 256, device=dev) / 16).to(torch.bfloat16)
    w2 = (torch.randn(256, FF, device=dev) / FF ** 0.5 * 0.5).to(torch.bfloat16)
    b1 = torch.randn(FF, device=dev) * 0.1; b2 = torch.randn(256, device=dev) * 0.1
    g1 = torch.rand(256, device=dev) + 0.5; bn1 = torch.randn(256, device=dev) * 0.1
    g2 = torch.rand(256, device=dev) + 0.5; bn2 = torch.randn(256, device=dev) * 0.1
    x0 = torch.randn(M, 256, device=dev)
    for dbl, split in ((0, 1), (0, 2), (1, 1), (1, 2)):
        L.check(lib.ppasr_b200_set_ffn_split(split))
        x = x0.clone(); yo = torch.zeros(M, 256, device=dev, dtype=torch.bfloat16)
        args = lambda: lib.ppasr_b200_op_fused_ffn(L.ptr(y), L.ptr(w1), L.ptr(w2), L.ptr(x), L.ptr(yo), L.ptr(b1), L.ptr(b2), L.ptr(g1), L.ptr(bn1),
                                                   L.ptr(g2) if dbl else None, L.ptr(bn2) if dbl else None, M, FF, 1e-5, L.stream_ptr())
        L.check(args()); torch.cuda.synchronize()
        h = y.float() @ w1.float().t() + b1; h = (h * torch.sigmoid(h)).to(torch.bfloat16).float()
        xr = x0 + h @ w2.float().t() + b2
        if dbl:
            xr = F.layer_norm(xr, (256,), g1, bn1, 1e-5); yr = F.layer_norm(xr, (256,), g2, bn2, 1e-5)
        else:
            yr = F.layer_norm(xr, (256,), g1, bn1, 1e-5)
        ex = (x - xr).abs().max().item() / xr.abs().max().item(); ey = (yo.float() - yr).abs().max().item() / yr.abs().max().item()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        for _ in range(3): args()
        e0.record()
        for _ in range(20): args()
        e1.record(); torch.cuda.synchronize()
        print(f"FF={FF:5d} double={dbl} split={split}: {e0.elapsed_time(e1)/20*1e3:7.1f} us  x rel err {ex:.2e}  y rel err {ey:.2e}", flush=True)
