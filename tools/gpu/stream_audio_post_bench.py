"""Audio post-processing (de-emphasis, 15/16 resampler): the row-table kernel against the uniform one, and the push
stream with listeners with post-processing off and on.

(a) b200_audio_post_rows against b200_audio_post on the same 512 rows x 5120 samples, flags AUDIO_DEEMPH_75US |
    AUDIO_RESAMPLE_48K at 51.2 kHz.  The table names the rows in order with carried state (no row fresh), so both forms
    do the same work.  Each call is two launches.  CUDA events around >= 1 s of back-to-back calls after a warm-up, the
    two forms alternated, two rounds each; the best round counts.
(b) b200_stream_* with 256 dongles, batch 204800, 10 listeners per dongle, pushes of 131072 samples (one librtlsdr
    buffer) round robin, centre audio, channel and payload sinks on, per-frame dB rows off; post-processing off against
    AUDIO_DEEMPH_75US | AUDIO_RESAMPLE_48K.  Samples per second of push plus flush (host clock), the two settings
    alternated, two rounds.  The sinks only count; each channel call is a Python callback, whose cost is included.

Reads the card's name, power limit and SM clock before and after.  Prints one JSON line; with --out it is also written
there.

    python tools/gpu/stream_audio_post_bench.py [--out profiles/r06_stream_audio_post.json]
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

FS = 2_048_000.0
RATE = 51200.0
ROUNDS = 2


def kernels(pkg, torch, args, res):
    S, n = args.rows, args.samples
    flags = pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K
    n_out = int(pkg.lib().b200_audio_post_out_samples(n, flags))
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand((S, n), dtype=torch.float32, device="cuda", generator=g) * 2 - 1
    out = torch.empty((S, n_out), dtype=torch.float32, device="cuda")
    st_u = torch.zeros((S, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    st_r = torch.zeros_like(st_u)
    table = (pkg.AudioPostRow * S)()
    for k in range(S):
        table[k].audio_row, table[k].out_row, table[k].state_row, table[k].fresh = k, k, k, 0
    L_ = pkg.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    px, po, pu, pr = (C.c_void_p(t.data_ptr()) for t in (x, out, st_u, st_r))

    # both forms are called through ctypes with their arguments built beforehand (the table too), so that the host
    # side of a call is the library's own
    def uniform():
        assert L_.b200_audio_post(px, n, S, n, RATE, flags, pu, po, n_out, stream) == 0

    def rows():
        assert L_.b200_audio_post_rows(px, n, S, n, RATE, flags, table, S, pr, S, po, n_out, S, stream) == 0

    ms = {"uniform": [], "rows": []}
    for _ in range(ROUNDS):
        ms["uniform"].append(timed(torch, uniform, args.seconds)[0])
        ms["rows"].append(timed(torch, rows, args.seconds)[0])
    best = {k: min(v) for k, v in ms.items()}
    res["kernels"] = {"rows": S, "samples_per_row": n, "flags": "75US|RESAMPLE_48K",
                      "uniform_ms": [round(v, 5) for v in ms["uniform"]], "rows_ms": [round(v, 5) for v in ms["rows"]],
                      "uniform_msamples_per_s": round(S * n / best["uniform"] / 1e3, 1),
                      "rows_msamples_per_s": round(S * n / best["rows"] / 1e3, 1),
                      "rows_over_uniform_time": round(best["rows"] / best["uniform"], 4)}


def push(pkg, np, args, res):
    S, batch, chunk, n_push, per_dongle = 256, 204800, 131072, args.pushes, 10
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
    settings = {"post_off": 0, "post_75us_48k": pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K}

    def run(flags):
        h = L_.b200_stream_create(S, batch, 0)
        assert h, pkg.binding.last_error()
        L_.b200_stream_set_sinks(h, pkg.binding.SPECTRUM_SINK(), cbs[0], None)
        assert L_.b200_stream_set_payload_sink(h, 6, cbs[2]) == 0
        assert L_.b200_stream_set_channel_sink(h, 32, cbs[1]) == 0
        assert L_.b200_stream_set_audio_post(h, flags, RATE) == 0, pkg.binding.last_error()
        for s in range(S):
            incs = (C.c_uint32 * 32)(*[(0x9E3779B9 * (s * 32 + c + 1)) & 0xFFFFFFFF for c in range(32)])
            ids = (C.c_int32 * 32)(*range(32))
            assert L_.b200_stream_set_channels(h, s, per_dongle, incs, ids) == 0
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

    run(settings["post_75us_48k"])           # warm-up: module loads, taps upload, pinned allocations
    times = {k: [] for k in settings}
    delivered = {}
    for _ in range(ROUNDS):
        for k, v in settings.items():
            dt, c = run(v)
            times[k].append(dt)
            delivered[k] = c
    total = S * n_push * chunk
    for k in settings:
        res["push"].append({"setting": k, "seconds": [round(x, 3) for x in times[k]],
                            "msamples_per_s": round(total / min(times[k]) / 1e6, 1),
                            "realtime_dongles_at_2048k": round(total / min(times[k]) / FS, 1),
                            "delivered": delivered[k]})
    res["push_setup"] = {"dongles": S, "listeners_per_dongle": per_dongle, "batch": batch, "push_samples": chunk,
                         "pushes_per_dongle": n_push, "samples_pushed": total}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=512)
    ap.add_argument("--samples", type=int, default=5120)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--pushes", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    import __graft_entry__ as graft
    pkg = graft.load_package()
    pkg.init(0)
    res = {"what": "audio post-processing: row-table kernel against the uniform one, and the push stream with 10 "
                   "listeners per dongle, post off against 75US|RESAMPLE_48K", "rounds": ROUNDS,
           "gpu": gpu_info(), "kernels": {}, "push": []}
    kernels(pkg, torch, args, res)
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
