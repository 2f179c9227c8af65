"""b200_fm_channels_exec throughput at R = 10 (the reference's default down factor, cbb_main.c:80).

256 streams x 2^23 - 8 samples (the largest multiple of 4R below 2^23; 4.3 GB of IQ, far past the 126 MB L2), channel counts C = 1, 2, 4, 10, 16, 32.  Every
number is CUDA events around >= 1 s of back-to-back launches after a warm-up.  Algorithmic bytes per input sample:
2 (IQ) + C * 4 / (4R) (f32 audio).  Also times b200_fm_exec on the same ring, one C = 10 launch against ten C = 1
launches.  Prints one JSON line; with --out it is also written to that file.

    python tools/gpu/fm_channels_bench.py [--streams 256] [--samples 8388600] [--out FILE]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

HBM_GBS = 6543.0          # the project's measured HBM copy bandwidth on B200 (DESIGN.md section 6)
R = 10
CHANNELS = (1, 2, 4, 10, 16, 32)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    first = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    return dict(zip(q.split(","), [v.strip() for v in first.split(",")])) if first else {"error": out.stderr.strip()}


def timed(torch, fn, min_seconds=1.0):
    """ms per call over >= min_seconds of back-to-back calls, after two warm-up calls."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    est = max(e0.elapsed_time(e1), 1e-3)
    n = max(3, math.ceil(min_seconds * 1e3 / est))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=256)
    ap.add_argument("--samples", type=int, default=(1 << 23) // (4 * R) * (4 * R))
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    import __graft_entry__ as graft
    pkg = graft.load_package()
    pkg.init(0)
    S, L = args.streams, args.samples
    info = gpu_info()
    ring = pkg.StreamRing(S, L, R=R)
    g = torch.Generator(device="cuda").manual_seed(0)
    for s0 in range(0, S, 32):        # seeded bytes, in slices to keep the temporary small
        ring.batch[s0:s0 + 32].copy_(torch.randint(0, 256, (min(32, S - s0), L, 2), dtype=torch.uint8, device="cuda",
                                                   generator=g))
    n_audio = L // (4 * R)
    rng = np.random.default_rng(1)
    incs_all = rng.integers(-2**31, 2**31, size=(S, max(CHANNELS)), dtype=np.int64).astype(np.int32)

    def record(ms, C, calls):
        gsps = S * L / ms / 1e6
        bps = 2.0 + C * 4.0 / (4 * R)
        return {"C": C, "ms": round(ms, 4), "launches_timed": calls, "gsamples_per_s": round(gsps, 1),
                "channel_gsamples_per_s": round(gsps * C, 1), "algorithmic_bytes_per_sample": round(bps, 3),
                "algorithmic_gbs": round(gsps * bps, 1), "hbm_fraction": round(gsps * bps / HBM_GBS, 4)}

    res = {"what": "b200_fm_channels_exec, R = 10", "streams": S, "samples_per_stream": L,
           "iq_bytes": 2 * S * L, "hbm_gbs_measured_peak": HBM_GBS, "gpu": info, "channels": []}

    fm_audio = torch.empty((S, n_audio), dtype=torch.float32, device="cuda")
    ms, calls = timed(torch, lambda: pkg.fm_exec(ring, audio=fm_audio), args.seconds)
    r = record(ms, 1, calls)
    res["fm_exec"] = r

    for C in CHANNELS:
        inc = torch.as_tensor(incs_all[:, :C].copy()).cuda()
        out = torch.empty((S, C, n_audio), dtype=torch.float32, device="cuda")
        ms, calls = timed(torch, lambda: pkg.fm_channels_exec(ring, inc, 0, audio=out), args.seconds)
        res["channels"].append(record(ms, C, calls))
        del out

    # one C = 10 launch against ten C = 1 launches of the same channels
    inc10 = torch.as_tensor(incs_all[:, :10].copy()).cuda()
    singles = [torch.as_tensor(incs_all[:, c:c + 1].copy()).cuda() for c in range(10)]
    out10 = torch.empty((S, 10, n_audio), dtype=torch.float32, device="cuda")
    outs1 = [torch.empty((S, 1, n_audio), dtype=torch.float32, device="cuda") for _ in range(10)]
    ms10, _ = timed(torch, lambda: pkg.fm_channels_exec(ring, inc10, 0, audio=out10), args.seconds)

    def ten():
        for c in range(10):
            pkg.fm_channels_exec(ring, singles[c], 0, audio=outs1[c])
    ms1x10, _ = timed(torch, ten, args.seconds)
    res["one_c10_vs_ten_c1"] = {"one_launch_c10_ms": round(ms10, 4), "ten_launches_c1_ms": round(ms1x10, 4),
                                "speedup": round(ms1x10 / ms10, 3)}
    del outs1
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
