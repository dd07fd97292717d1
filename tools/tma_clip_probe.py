import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from liteasr_b200 import ops
for cdt in (torch.bfloat16, torch.float32):
    for n in (299, 297, 290):
        m, k = 256, 64
        g = torch.Generator(device="cuda").manual_seed(1)
        a = (torch.randn(m, k, generator=g, device="cuda")).bfloat16()
        b = (torch.randn(n, k, generator=g, device="cuda")).bfloat16()
        ld = 320
        buf = torch.full((m, ld), 7.0, device="cuda", dtype=cdt)
        ops.gemm(a, b, buf[:, :n], m, n, k, lda=k, ldb=k, ldc=ld)
        torch.cuda.synchronize()
        changed = (buf[:, n:] != 7.0).any(0).nonzero().flatten().tolist()
        print(cdt, n, "padding columns changed:", [n + c for c in changed], "values", buf[0, n:n+8].tolist())
