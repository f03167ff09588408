"""BASELINE.json configs[4]: synthetic sweep N = 10k-1M, d = 64-512, k_max = 8-64 for the all-pairs score GEMM +
streaming top-k, and the CSR SpMM, one JSON line per point (CUDA events, warm, inputs resident).

    python scripts/sweep.py > profiles/rNN_sweep.jsonl

Score GEMM + top-k: Gpairs/s and the TF32 tensor throughput it implies (3 x 2 N^2 d flop for 3xTF32) against the
1.1 PFLOP/s dense TF32 peak of B200_PROFILING.md.  SpMM: algorithmic bytes (SURVEY 8d) / time against the measured
HBM peak in MEASURED_PEAKS.json (hits in the 126 MB L2 can push the ratio above 1)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dgg_b200 import CSRGraph, functional as K

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
HBM = json.load(open(pk))["hbm_gbs"] if os.path.isfile(pk) else 6650.0
TF32_PEAK = 1100.0   # TFLOP/s dense, B200_PROFILING.md
dev = "cuda"


def timed(fn, it):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(it): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / it * 1e-3


def allpairs(n, d, kc, noise=True):
    z = torch.softmax(torch.randn(n, d, device=dev), -1)
    t = torch.tensor([4.0], device=dev)
    kw = dict(noise=None, kc=kc, precision=3)
    if noise: kw.update(seed=1, noise_scale=1.0)
    try:
        with torch.no_grad():
            s = timed(lambda: K.allpairs_topk(z, t, **kw), 1 if n >= 400000 else 3)
    except Exception as e:   # an unsupported shape (kc > 64): say so
        print(json.dumps(dict(op="allpairs_topk_fwd", n=n, d=d, kc=kc, error=str(e)[:120])), flush=True)
        return
    flops = 3 * 2.0 * n * n * d
    print(json.dumps(dict(op="allpairs_topk_fwd", n=n, d=d, kc=kc, noise="philox" if noise else "none", ms=s * 1e3,
                          gpairs_s=n * n / s / 1e9, tf32_tflops=flops / s / 1e12, tensor_frac=flops / s / 1e12 / TF32_PEAK)),
          flush=True)


def spmm(n, deg, f):
    g = torch.Generator().manual_seed(n + deg)
    m = n * deg
    a = torch.sparse_coo_tensor(torch.stack([torch.randint(0, n, (m,), generator=g), torch.randint(0, n, (m,), generator=g)]),
                                torch.ones(m), (n, n)).coalesce()
    G = CSRGraph.from_indices(a.indices().to(dev), n); nnz = G.nnz
    vals = torch.rand(nnz, device=dev); x = torch.randn(n, f, device=dev); dy = torch.randn(n, f, device=dev)
    with torch.no_grad():
        tf = timed(lambda: K.spmm(vals, x, G), 10)
    vg, xg = vals.clone().requires_grad_(True), x.clone().requires_grad_(True)
    y = K.spmm(vg, xg, G)
    def bwd():
        vg.grad = None; xg.grad = None
        y.backward(dy, retain_graph=True)
    tb = timed(bwd, 10)
    bf = nnz * (8 + f * 4) + 4 * (n + 1) + n * f * 4
    bb = bf + nnz * (f * 4 + 4) + nnz * f * 4
    print(json.dumps(dict(op="spmm_csr", n=n, nnz=nnz, f=f, fwd_us=tf * 1e6, fwd_gbs=bf / tf / 1e9, fwd_frac=bf / tf / 1e9 / HBM,
                          bwd_us=tb * 1e6, bwd_gbs=bb / tb / 1e9, bwd_frac=bb / tb / 1e9 / HBM)), flush=True)


if __name__ == "__main__":
    for n in (10000, 37888, 100000, 232965, 1000000):
        allpairs(n, 64, 32)
    for d in (32, 128, 256, 512):
        allpairs(37888, d, 32)
    for kc in (8, 16, 64):
        allpairs(37888, 64, kc)
    allpairs(37888, 64, 32, noise=False)
    for (n, deg, f) in [(10000, 8, 64), (100000, 16, 64), (232965, 50, 64), (232965, 50, 128), (232965, 16, 512),
                        (1000000, 16, 64), (1000000, 8, 256)]:
        spmm(n, deg, f)
