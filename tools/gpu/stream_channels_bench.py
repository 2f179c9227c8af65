"""FM channels on the push stream: the runs-table kernels against the uniform ones, and the push path with listeners.

(a) b200_fm_channels_exec_runs against b200_fm_channels_exec / _exec_fir at uniform channel counts C in {1, 10, 32},
    R = 10, 256 streams x 8388600 samples (4.3 GB of IQ, far past the 126 MB L2), boxcar and T = 200 (Kaiser, 80 kHz,
    60 dB).  A table holds at most 64 runs, so the runs form covers the 256 rows in 4 launches of 64 runs (tables built
    before timing); the uniform form is one launch, and is also timed as 4 launches over the same 64-row slices, which
    separates the cost of the split from that of the runs kernel.  CUDA events around >= 1 s of back-to-back calls after
    a warm-up, the three forms alternated, two rounds each; the best round counts.
(b) b200_stream_* with 256 dongles, batch 204800, pushes of 131072 samples (one librtlsdr buffer) round robin, centre
    audio and payload sinks on, per-frame dB rows off.  Listener mixes: none, 10 channels per dongle, and a ragged mix
    of 0 to 32 per dongle (seeded).  Samples per second of push plus flush (host clock), mixes alternated, two rounds.
    The sinks only count; each channel call is a Python callback, whose cost is included.

Reads the card's name and power limit before and after.  Prints one JSON line; with --out it is also written there.

    python tools/gpu/stream_channels_bench.py [--out profiles/r05_stream_channels.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from fm_channels_bench import gpu_info, timed  # noqa: E402

R = 10
FS = 2_048_000.0
CHANNELS = (1, 10, 32)
TAPS = (0, 200)
ROUNDS = 2


def kernels(pkg, torch, np, args, res):
    S, L = args.streams, args.samples
    hist = pkg.fm_channels_fir_history_samples(R, max(TAPS))
    ring = pkg.StreamRing(S, L, R=R, history=hist)
    g = torch.Generator(device="cuda").manual_seed(0)
    for s0 in range(0, S, 32):
        ring.batch[s0:s0 + 32].copy_(torch.randint(0, 256, (min(32, S - s0), L, 2), dtype=torch.uint8, device="cuda",
                                                   generator=g))
    n_audio = L // (4 * R)
    rng = np.random.default_rng(1)
    incs_all = rng.integers(0, 2**32, size=(S, max(CHANNELS)), dtype=np.int64)
    taps = {T: torch.as_tensor(pkg.fm_channel_filter(R, T, 80e3, 60.0)).cuda() for T in TAPS if T}
    L_ = pkg.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    for Ch in CHANNELS:
        inc = torch.as_tensor((incs_all[:, :Ch] & 0xFFFFFFFF).astype(np.uint32).view(np.int32)).cuda()
        audio = torch.empty((S, Ch, n_audio), dtype=torch.float32, device="cuda")
        tables = []
        for r0 in range(0, S, pkg.FM_MAX_RUNS):
            n = min(pkg.FM_MAX_RUNS, S - r0)
            t = (pkg.FmChannelRun * n)()
            for k in range(n):
                t[k].stream, t[k].n_channels, t[k].first_sample, t[k].audio_row = r0 + k, Ch, 0, (r0 + k) * Ch
                for c in range(Ch):
                    t[k].phase_inc[c] = int(incs_all[r0 + k, c]) & 0xFFFFFFFF
            tables.append((t, n))
        for T in TAPS:
            tp = taps.get(T)

            def runs_form():
                for t, n in tables:
                    rc = L_.b200_fm_channels_exec_runs(C.c_void_p(ring.batch.data_ptr()), ring.stride_bytes, S, L, R, t,
                                                       n, C.c_void_p(audio.data_ptr()), n_audio, S * Ch,
                                                       C.c_void_p(tp.data_ptr()) if tp is not None else None,
                                                       T, stream)
                    assert rc == 0, pkg.binding.last_error()

            def uniform_form():
                pkg.fm_channels_exec(ring, inc, 0, audio=audio, taps=tp)

            def uniform_split():
                # the uniform kernel over the runs form's 64-row slices: what splitting into 4 launches costs alone
                for r0 in range(0, S, pkg.FM_MAX_RUNS):
                    n = min(pkg.FM_MAX_RUNS, S - r0)
                    a = (C.c_void_p(ring.batch[r0].data_ptr()), ring.stride_bytes, n, L, R, 0,
                         C.c_void_p(inc[r0].data_ptr()), Ch, C.c_void_p(audio[r0].data_ptr()), n_audio, None, 0)
                    rc = (L_.b200_fm_channels_exec_fir(*a, C.c_void_p(tp.data_ptr()), T, stream) if tp is not None
                          else L_.b200_fm_channels_exec(*a, stream))
                    assert rc == 0, pkg.binding.last_error()

            ms = {"uniform": [], "runs": [], "uniform_4x64": []}
            for _ in range(ROUNDS):
                ms["uniform"].append(timed(torch, uniform_form, args.seconds)[0])
                ms["runs"].append(timed(torch, runs_form, args.seconds)[0])
                ms["uniform_4x64"].append(timed(torch, uniform_split, args.seconds)[0])
            best = {k: min(v) for k, v in ms.items()}
            res["kernels"].append({"C": Ch, "filter": "boxcar" if T == 0 else f"fir T={T}",
                                   "uniform_ms": [round(x, 4) for x in ms["uniform"]],
                                   "runs_ms": [round(x, 4) for x in ms["runs"]],
                                   "uniform_4x64_ms": [round(x, 4) for x in ms["uniform_4x64"]],
                                   "uniform_channel_gsamples_per_s": round(S * L * Ch / best["uniform"] / 1e6, 1),
                                   "runs_channel_gsamples_per_s": round(S * L * Ch / best["runs"] / 1e6, 1),
                                   "runs_over_uniform_time": round(best["runs"] / best["uniform"], 4),
                                   "runs_over_uniform_4x64_time": round(best["runs"] / best["uniform_4x64"], 4)})
            out[(Ch, T)] = best
        del audio
    del ring
    torch.cuda.empty_cache()


def push(pkg, np, args, res):
    S, batch, chunk, n_push = 256, 204800, 131072, args.pushes
    L_ = pkg.lib()
    rng = np.random.default_rng(2)
    bufs = [rng.integers(0, 256, size=2 * chunk, dtype=np.uint8) for _ in range(4)]
    counts = {"audio": 0, "channel": 0, "payload": 0}

    def on_audio(u, s, first, n, p):
        counts["audio"] += n

    def on_channel(u, s, cid, first, n, p):
        counts["channel"] += n

    def on_payload(u, s, first, k, p):
        counts["payload"] += 1

    cbs = (pkg.binding.AUDIO_SINK(on_audio), pkg.binding.CHANNEL_SINK(on_channel), pkg.binding.PAYLOAD_SINK(on_payload))
    mixes = {"none": [0] * S, "10_per_dongle": [10] * S,
             "ragged_0_32": [int(x) for x in rng.integers(0, 33, size=S)]}

    def run(per_dongle):
        h = L_.b200_stream_create(S, batch, 0)
        assert h, pkg.binding.last_error()
        L_.b200_stream_set_sinks(h, pkg.binding.SPECTRUM_SINK(), cbs[0], None)
        assert L_.b200_stream_set_payload_sink(h, 6, cbs[2]) == 0
        if any(per_dongle):
            assert L_.b200_stream_set_channel_sink(h, 32, cbs[1]) == 0
            for s, n in enumerate(per_dongle):
                incs = (C.c_uint32 * 32)(*[(0x9E3779B9 * (s * 32 + c + 1)) & 0xFFFFFFFF for c in range(32)])
                ids = (C.c_int32 * 32)(*range(32))
                assert L_.b200_stream_set_channels(h, s, n, incs, ids) == 0
        for k in counts:
            counts[k] = 0
        t0 = time.perf_counter()
        for i in range(n_push):
            p = bufs[i % len(bufs)].ctypes.data
            for s in range(S):
                assert L_.b200_stream_push(h, s, p, chunk) == 0
        assert L_.b200_stream_flush(h) == 0
        dt = time.perf_counter() - t0
        L_.b200_stream_destroy(h)
        return dt, dict(counts)

    run([10] * S)            # warm-up: module loads, attributes, pinned allocations
    times = {k: [] for k in mixes}
    delivered = {}
    for _ in range(ROUNDS):
        for k, v in mixes.items():
            dt, c = run(v)
            times[k].append(dt)
            delivered[k] = c
    total = S * n_push * chunk
    for k, v in mixes.items():
        res["push"].append({"mix": k, "channels_total": sum(v), "seconds": [round(x, 3) for x in times[k]],
                            "msamples_per_s": round(total / min(times[k]) / 1e6, 1),
                            "realtime_dongles_at_2048k": round(total / min(times[k]) / FS, 1),
                            "delivered": delivered[k]})
    res["push_setup"] = {"dongles": S, "batch": batch, "push_samples": chunk, "pushes_per_dongle": n_push,
                         "samples_pushed": total}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=256)
    ap.add_argument("--samples", type=int, default=(1 << 23) // (4 * R) * (4 * R))
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--pushes", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    import __graft_entry__ as graft
    pkg = graft.load_package()
    pkg.init(0)
    res = {"what": "FM channels: runs-table kernels against the uniform ones (R = 10), and the push stream with "
                   "listeners", "streams": args.streams, "samples_per_stream": args.samples, "rounds": ROUNDS,
           "gpu": gpu_info(), "kernels": [], "push": []}
    kernels(pkg, torch, np, args, res)
    push(pkg, np, args, res)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
