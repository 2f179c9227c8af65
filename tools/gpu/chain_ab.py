"""chain_exec (chain_jobs_kernel) timed on bench.py's ring for one or more builds of libb200sdr.so, alternated.

Each build runs in a fresh process per round, in the order given, so with two builds the rounds go A B A B ...  A
process fills the ring as bench.py does (256 streams x 8 192 000 samples of its synthetic FM, 4.2 GB) and times:
  - burst: 10 back-to-back launches after 3 warm-up launches (CUDA events);
  - sustained: back-to-back launches for >= --seconds and >= 300 launches, power cap included (CUDA events).
The card's name, power limit and SM clock are read before and after each process.  Prints one JSON line; with --out
it is also written there.

    python tools/gpu/chain_ab.py --lib parent=/path/libb200sdr.so --lib new=rtl-ws_b200/libb200sdr.so [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

BURST = 10
MIN_SUSTAINED = 300


def one(lib_path, seconds):
    """Time one build in this process; returns the result as a dict."""
    import torch

    import bench
    import __graft_entry__ as graft
    from fm_channels_bench import gpu_info

    pkg = graft.load_package()
    pkg.binding.LIB_PATH = os.path.abspath(lib_path)     # before the first load: this process runs that build
    pkg.init(0)
    device = torch.device("cuda", 0)
    S, L = bench.N_STREAMS, bench.LAUNCH_SAMPLES_PER_STREAM
    info = gpu_info()
    ring = pkg.StreamRing(S, L)
    for i in range(0, S, 4):
        ring.batch[i:i + 4].copy_(bench.synth_fm_device(torch, list(range(i, min(i + 4, S))), L, device))
    db = torch.empty((S, L // 1024, 1024), dtype=torch.float32, device=device)
    audio = torch.empty((S, L // 40), dtype=torch.float32, device=device)

    def launch():
        pkg.chain_exec(ring, db=db, audio=audio)

    for _ in range(3):
        launch()
    burst_ms = bench.timed_launches(torch, launch, BURST)
    n = max(MIN_SUSTAINED, int(seconds * 1e3 / burst_ms) + 1)
    sustained_ms = bench.timed_launches(torch, launch, n)
    samples = S * L
    return {"lib": lib_path, "gpu": info, "gpu_after": gpu_info(),
            "burst": {"launches": BURST, "ms": round(burst_ms, 4), "gsamples_per_s": round(samples / burst_ms / 1e6, 1)},
            "sustained": {"launches": n, "seconds": round(n * sustained_ms / 1e3, 2), "ms": round(sustained_ms, 4),
                          "gsamples_per_s": round(samples / sustained_ms / 1e6, 1)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH",
                    help="a build to time (repeat; default: the tree's own as 'tree')")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--seconds", type=float, default=1.0, help="minimum length of the sustained window")
    ap.add_argument("--cool", type=float, default=5.0, help="idle seconds before each process")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one(args.one, args.seconds)))
        return
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", os.path.join(ROOT, "rtl-ws_b200", "libb200sdr.so"))]
    runs = {name: [] for name, _ in libs}
    for _ in range(args.rounds):
        for name, path in libs:
            time.sleep(args.cool)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", path, "--seconds", str(args.seconds)],
                                 capture_output=True, text=True, check=True)
            runs[name].append(json.loads(out.stdout.strip().splitlines()[-1]))
    res = {"what": "chain_exec on bench.py's ring (256 streams x 8192000 samples), builds alternated per round",
           "rounds": args.rounds, "order": [name for name, _ in libs], "runs": runs, "summary": {}}
    for name, rs in runs.items():
        b = [r["burst"]["gsamples_per_s"] for r in rs]
        s = [r["sustained"]["gsamples_per_s"] for r in rs]
        res["summary"][name] = {"burst_gsamples_per_s": b, "sustained_gsamples_per_s": s,
                                "burst_spread": round(max(b) - min(b), 1), "sustained_spread": round(max(s) - min(s), 1)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
