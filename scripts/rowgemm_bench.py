"""Times rowgemm_kernel alone (lab entry point) on a training-sized layer, for each of its epilogue cases."""
import os, sys, json
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pixel_nerf_yolo_b200 import _lib
lib = _lib.load()
M, N, K = 147456, 512, int(os.environ.get("KK", "512"))
dev = torch.device("cuda", 0)
st = _lib.stream_ptr(dev)
A = torch.randn(M, K, device=dev); W = torch.randn(N, K, device=dev) / K ** 0.5
bias = torch.randn(N, device=dev); res = torch.randn(M, N, device=dev); mask = torch.randn(M, N, device=dev)
o32 = torch.empty(M, N, device=dev); o16 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
ws = torch.empty(lib.pnr_lab_gemm_workspace_bytes(M, N, K) + 1024, dtype=torch.uint8, device=dev)
cases = {"h-layer (bias, bf16 relu out)": (bias, None, None, None, o16, 1),
         "x-layer (bias, res in place, f32 + bf16 out)": (bias, None, res, res, o16, 1),
         "dx-layer (mask, res in place, f32 + bf16 out)": (None, mask, res, res, o16, 0),
         "plain f32 out": (None, None, None, o32, None, 0),
         "f32 out + bias": (bias, None, None, o32, None, 0),
         "bf16 out, no bias": (None, None, None, None, o16, 0),
         "bf16 relu out, no bias": (None, None, None, None, o16, 1),
         "f32 + bf16 out": (None, None, None, o32, o16, 0)}
out = {}
for name, (b, m, r, f, h, relu) in cases.items():
    def go():
        rc = lib.pnr_lab_rowgemm(A.data_ptr(), W.data_ptr(), _lib.ptr(b), _lib.ptr(m), _lib.ptr(r), _lib.ptr(f), _lib.ptr(h), M, N, K, relu,
                                 ws.data_ptr(), ws.numel(), st)
        _lib.check(rc, "rowgemm")
    go(); torch.cuda.synchronize()
    # the lab entry converts / packs first: time the whole call minus a run with M tiny? simpler: events around 3 calls, min
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); go(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    out[name] = round(best * 1e3)
print(json.dumps({"K": K, "us (incl. fp32->bf16 conversion of A ~ 150 us)": out}))
