"""Selective-scan backward at the north-star shape with and without the dB/dC reduction (VMB_BWD_NORED=1 skips the smem read-back +
red.global of the group reduction): what that stage costs."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from vmambair_b200 import ops
from tools.scan_bench import bench
dev="cuda"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for B in (1, 4, 8, 32):
    D,K,N,L=384,4,16,4096
    torch.manual_seed(0)
    dt=torch.bfloat16
    u = torch.randn(B, D, L, device=dev).to(dt); delta = (0.5 * torch.rand(B, D, L, device=dev)).to(dt)
    A = -0.5 * torch.rand(D, N, device=dev); Bm = torch.randn(B, K, N, L, device=dev).to(dt); Cm = torch.randn(B, K, N, L, device=dev).to(dt)
    Dv = torch.randn(D, device=dev); bias = 0.5 * torch.rand(D, device=dev); dout = torch.randn_like(u)
    out, ck = ops.selective_scan_fwd(u, delta, A, Bm, Cm, Dv, bias, True, True)
    rec=dict(B=B)
    for nored in (0, 1):
        os.environ["VMB_BWD_NORED"] = str(nored)
        ms = bench(lambda: ops.selective_scan_bwd(u, delta, A, Bm, Cm, Dv, bias, dout, ck, True), flush=flush)
        rec[f"nored{nored}"] = round(ms * 1e3 / B, 1)
    os.environ["VMB_BWD_NORED"] = "0"
    print(json.dumps(rec), flush=True)
