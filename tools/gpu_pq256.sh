#!/bin/bash
# wide-codebook PQ encode (pq_tensor.cuh, 24 x 256 at d = 768): parity against the fp32 sub-vector kernel, then timing
timeout 400 python - <<'PY'
import os, sys, torch
sys.path.insert(0, os.getcwd())
import mevi_b200
ctx = mevi_b200.get_context(0)
torch.manual_seed(3)
def both(X, cb):
    os.environ["MEVI_PQ_TENSOR"] = "1"; a = ctx.pq_encode(X, cb); ctx.check()
    os.environ["MEVI_PQ_TENSOR"] = "0"; e = ctx.pq_encode(X, cb); ctx.check()
    os.environ["MEVI_PQ_TENSOR"] = "1"
    return a, e
for (n, M, metric_scale, shift) in ((200003, 24, 1.0, 0.0), (65536, 24, 1e-3, 0.0), (50001, 24, 40.0, 0.7), (4097, 32, 1.0, 0.0), (300000, 24, 1.0, 0.0)):
    d = 32 * M
    X = (torch.randn((n, d), device="cuda") * metric_scale + shift).contiguous()
    # centroids = data rows (k-means-like codebook: scores near zero distance exist) for the last case, random otherwise
    if n == 300000:
        cb = torch.stack([X[torch.randint(0, n, (256,), device="cuda"), 32 * j:32 * j + 32] for j in range(M)]).contiguous()
    else:
        cb = (torch.randn((M, 256, 32), device="cuda") * metric_scale + shift).contiguous()
    a, e = both(X, cb)
    print(f"n {n} M {M} scale {metric_scale} shift {shift}: mismatching codes {int((a != e).sum())} of {a.numel()}", flush=True)
for (n, M) in ((100003, 32), (4100, 8)):
    X = torch.randn((n, 24 * M), device="cuda"); cb = torch.randn((M, 256, 24), device="cuda")
    a, e = both(X, cb)
    print(f"width 24: n {n} M {M}: mismatching codes {int((a != e).sum())} of {a.numel()}", flush=True)
n = 8841823
X = torch.randn((n, 768), device="cuda")
cb = torch.randn((24, 256, 32), device="cuda")
def run(tag, reps=5):
    for _ in range(2): ctx.pq_encode(X, cb)
    torch.cuda.synchronize()
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps): ctx.pq_encode(X, cb)
    t.record(); torch.cuda.synchronize(); ms = s.elapsed_time(t) / reps
    print(f"{tag:40s} {ms:8.3f} ms  {n*3072/ms/1e6:7.0f} GB/s  frac {n*3072/ms/1e6/6541.8:.3f}", flush=True)
run("pq 24x256 tensor")
cb24 = torch.randn((32, 256, 24), device="cuda"); cb32 = cb; cb = cb24; run("pq 32x256 (width 24) tensor"); cb = cb32
a = ctx.pq_encode(X[:200000], cb); os.environ["MEVI_PQ_TENSOR"] = "0"; e = ctx.pq_encode(X[:200000], cb)
print("mismatch on 200k of the timed matrix:", int((a != e).sum()))
ctx.check()
PY
echo "rc=$?"
