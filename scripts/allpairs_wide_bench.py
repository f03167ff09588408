"""All-pairs score + top-K forward at embedding widths around and above 128, against the chunked fp32 torch route.

    python scripts/allpairs_wide_bench.py [--n 37888 100000 232965] [--d 128 192 256 384 512] [--kc 32]

One JSON line per point (CUDA events, after a warm-up call, inputs resident on the device):
  * kernel: ``functional.allpairs_topk`` at 3xTF32 with no noise and with in-kernel Philox Gumbel noise; Gpairs/s
    (N^2 / t) and the TF32 rate that implies (3 x 2 N^2 d flop: hi*hi, hi*lo and lo*hi passes);
  * torch: what a user has without the kernel at these widths -- TF32 disabled, ``torch.cdist`` over row chunks, then
    ``topk(kc)`` of -t D per chunk (no noise), timed in the same process.
d = 128 is the resident-tile kernel (v2), for context; d > 128 is the k-block-streamed instantiation.  The first line
records the GPU name and its power limit, which every number here depends on."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from dgg_b200 import functional as K  # noqa: E402


def timed(fn, min_s=0.3, max_it=50):
    """Mean seconds per call: one warm-up call, then enough calls for about min_s seconds of work."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    once = e0.elapsed_time(e1) * 1e-3
    it = max(1, min(max_it, int(min_s / max(once, 1e-6))))
    e0.record()
    for _ in range(it):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / it


def torch_route(z, t, kc, chunk_bytes=4 << 30):
    n = z.shape[0]
    rows = max(1, chunk_bytes // (4 * n))
    out_i, out_v = [], []
    for r0 in range(0, n, rows):
        y = torch.cdist(z[r0:r0 + rows], z).mul_(-t)
        v, i = y.topk(kc, dim=-1)
        out_i.append(i)
        out_v.append(v)
    return torch.cat(out_i), torch.cat(out_v)


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: " + str(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[37888, 100000, 232965])
    ap.add_argument("--d", type=int, nargs="+", default=[128, 192, 256, 384, 512])
    ap.add_argument("--kc", type=int, default=32)
    ap.add_argument("--no-torch", action="store_true", help="skip the chunked fp32 torch route")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("allpairs_wide_bench.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    print(json.dumps(gpu_info()), flush=True)
    t = torch.tensor([1.0], device="cuda")
    for n in a.n:
        for d in a.d:
            gen = torch.Generator(device="cuda").manual_seed(n + d)
            z = torch.softmax(torch.randn(n, d, device="cuda", generator=gen) * 2.0, -1)
            rec = dict(n=n, d=d, kc=a.kc)
            for name, kw in (("none", {}), ("philox", dict(seed=1234, noise_scale=1.0))):
                s = timed(lambda: K.allpairs_topk(z, t, kc=a.kc, precision=3, **kw))
                rec[f"kernel_{name}_ms"] = round(s * 1e3, 3)
                rec[f"kernel_{name}_gpairs_s"] = round(n * n / s * 1e-9, 2)
                rec[f"kernel_{name}_tf32_tflops"] = round(3 * 2 * n * n * d / s * 1e-12, 1)
            if not a.no_torch:
                s = timed(lambda: torch_route(z, 1.0, a.kc), min_s=0.5, max_it=5)
                rec["torch_fp32_ms"] = round(s * 1e3, 3)
                rec["torch_fp32_gpairs_s"] = round(n * n / s * 1e-9, 2)
                rec["kernel_speedup_vs_torch_none"] = round(rec["torch_fp32_ms"] / rec["kernel_none_ms"], 2)
            print(json.dumps(rec), flush=True)
            del z
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
