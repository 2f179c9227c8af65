"""b200_fm_channels_exec_fir throughput at R = 10 against the boxcar kernel (b200_fm_channels_exec) on the same ring.

256 streams x 2^23 - 8 samples (4.3 GB of IQ, far past the 126 MB L2), C in {1, 10, 32} channels, T in {10 (all-one
taps: the boxcar through the FIR kernel), 80, 160, 200} taps (Kaiser designs, 80 kHz cutoff, 60 dB).  Every number is
CUDA events around >= 1 s of back-to-back launches after a warm-up; the boxcar and the FIR kernels are timed in
alternation, twice each.  Channel Gsamples/s = input samples per second times C.  Reports whether 256 dongles x 10
channels run in real time at 2.048 MS/s (5.24 G channel-samples/s) with T = 200.  Prints one JSON line; with --out it
is also written to that file.

    python tools/gpu/fm_channels_fir_bench.py [--streams 256] [--samples 8388600] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from fm_channels_bench import gpu_info, timed  # noqa: E402

R = 10
FS = 2_048_000.0
CHANNELS = (1, 10, 32)
TAPS = (10, 80, 160, 200)
ROUNDS = 2


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
    hist = max(pkg.fm_channels_fir_history_samples(R, T) for T in TAPS)      # one ring serves every kernel
    ring = pkg.StreamRing(S, L, R=R, history=hist)
    g = torch.Generator(device="cuda").manual_seed(0)
    for s0 in range(0, S, 32):        # seeded bytes, in slices to keep the temporary small
        ring.batch[s0:s0 + 32].copy_(torch.randint(0, 256, (min(32, S - s0), L, 2), dtype=torch.uint8, device="cuda",
                                                   generator=g))
    n_audio = L // (4 * R)
    rng = np.random.default_rng(1)
    incs_all = rng.integers(-2**31, 2**31, size=(S, max(CHANNELS)), dtype=np.int64).astype(np.int32)
    taps = {T: torch.as_tensor(np.ones(T, np.float32) if T == R else pkg.fm_channel_filter(R, T, 80e3, 60.0)).cuda()
            for T in TAPS}

    res = {"what": "b200_fm_channels_exec_fir against b200_fm_channels_exec, R = 10", "streams": S,
           "samples_per_stream": L, "iq_bytes": 2 * S * L, "history_samples": hist, "rounds": ROUNDS, "gpu": info,
           "results": []}
    for C in CHANNELS:
        inc = torch.as_tensor(incs_all[:, :C].copy()).cuda()
        out = torch.empty((S, C, n_audio), dtype=torch.float32, device="cuda")
        runs = {"boxcar": []}
        runs.update({T: [] for T in TAPS})
        for _ in range(ROUNDS):
            ms, _ = timed(torch, lambda: pkg.fm_channels_exec(ring, inc, 0, audio=out), args.seconds)
            runs["boxcar"].append(ms)
            for T in TAPS:
                ms, _ = timed(torch, lambda: pkg.fm_channels_exec(ring, inc, 0, audio=out, taps=taps[T]), args.seconds)
                runs[T].append(ms)
        for key, ms_list in runs.items():
            ms = min(ms_list)
            gsps = S * L / ms / 1e6
            res["results"].append({"C": C, "kernel": "boxcar" if key == "boxcar" else "fir", "T": R if key == "boxcar" else key,
                                   "ms": [round(x, 4) for x in ms_list], "gsamples_per_s": round(gsps, 2),
                                   "channel_gsamples_per_s": round(gsps * C, 1)})
        del out
    need = 256 * 10 * FS / 1e9
    at200 = next(r for r in res["results"] if r["C"] == 10 and r["kernel"] == "fir" and r["T"] == 200)
    res["realtime_256x10_at_T200"] = {"needed_channel_gsamples_per_s": round(need, 3),
                                      "measured_channel_gsamples_per_s": at200["channel_gsamples_per_s"],
                                      "holds": at200["channel_gsamples_per_s"] >= need,
                                      "headroom": round(at200["channel_gsamples_per_s"] / need, 1)}
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
