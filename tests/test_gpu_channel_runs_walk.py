"""FM channels over a runs table (b200_fm_channels_exec_runs) and on the push stream when every CTA walks many tiles.

The runs kernels (fm_channels_runs_kernel<10, 8> and <0, 4>, fm_channels_fir_runs_kernel) are persistent: a launch
has min(SM count x CTAs per SM, tiles) CTAs and CTA b walks tiles b, b + grid, b + 2 grid, ... through a TMA ring of
one or two stages.  Only past its first tile does a CTA refill a stage (with the tile n_stages steps ahead, whose run
the refill looks up), wait on the flipped mbarrier parity and take a second tile's IQ row, channel count, increments,
first decimated sample and audio rows from that tile's own run.  So every case sizes its table from b200_sm_count()
and an UPPER bound on resident CTAs, as test_gpu_fm_rates.py does, and asserts that the tiles cover every worker at
least WALK times, with an odd prime number of tiles per run (CTAs cross run boundaries mid-walk) and a short last
tile.

References: the uniform calls (b200_fm_channels_exec / _exec_fir) on each run's row, position and increments, bit for
bit; for three runs per table the float64 oracle (mix_boxcar / mix_fir, demodulate) on the uniform call's baseband;
on the push stream, exec_runs over the whole capture and a stream without a channel sink.
"""
import functools
from importlib import import_module

import numpy as np
import pytest

from test_gpu_fm_channels import demodulate, mix_boxcar
from test_gpu_fm_channels_fir import design, dev, fir_ctas_per_sm, mix_fir
from test_gpu_fm_rates import FC_T, WALK, fc_ctas_per_sm, fm_segment, is_prime, short_tile, sm_count, tiles_per_stream
from test_gpu_stream_channels import (COUNTS, CYCLE, joined, listeners, long_runs, random_incs, raw_runs_call,
                                      ring_for, uniform)

pytestmark = pytest.mark.gpu

N_RUNS = 64                     # B200_FM_MAX_RUNS: the whole __grid_constant__ table
ORACLE_RUNS = (0, 29, 63)       # the first run, one of 32 channels in the middle, the 64th
SEG = 299_993                   # samples per generated segment (not a multiple of any tile)


# ---- sizing --------------------------------------------------------------------------------------------------------

def workers(pkg, R, T):
    """Upper bound on the CTAs a runs launch keeps resident: the SM count times the CTAs per SM that threads and
    shared memory allow (fc_ctas_per_sm applies to the runs launcher unchanged: it uses the uniform formula)."""
    return sm_count(pkg) * (fir_ctas_per_sm(R, T) if T else fc_ctas_per_sm(R))


def walk_checks(n, R, n_runs, n_workers):
    """What a launch of n_runs runs of n samples needs to walk: n a multiple of 4R and of 8, an odd prime number of
    tiles per run, a short and even last tile, and at least WALK tiles for every worker.  -> (tiles per run, checks)."""
    n_audio = n // (4 * R)
    tpr = -(-n_audio // FC_T)
    return tpr, dict(aligned=n % (4 * R) == 0 and n % 8 == 0, odd_prime=tpr % 2 == 1 and is_prime(tpr),
                     short_last=n_audio % FC_T != 0 and n_audio % 2 == 0, walks=n_runs * tpr >= WALK * n_workers)


def check_walk(n, R, n_runs, n_workers):
    """Assert every walk check.  -> tiles per run."""
    tpr, checks = walk_checks(n, R, n_runs, n_workers)
    assert all(checks.values()), (n, R, n_runs, n_workers, tpr, checks)
    return tpr


def walk_samples(pkg, R, T, n_runs):
    """n_samples of a runs launch of n_runs runs whose every resident CTA walks at least WALK tiles."""
    w = workers(pkg, R, T)
    tpr = tiles_per_stream(w, n_runs)
    n = 4 * R * ((tpr - 1) * FC_T + short_tile(FC_T))
    assert check_walk(n, R, n_runs, w) == tpr
    return n


# ---- signals and tables --------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def station(carrier):
    synth = import_module("rtl_ws_b200.synth")
    return synth.s3_fm(SEG, seed=int(carrier) % 1000 + 7, deviation=75e3, carrier=carrier)


@functools.lru_cache(maxsize=None)
def noise():
    return np.random.default_rng(17).integers(0, 256, size=(SEG, 2), dtype=np.uint8)


def segments():
    """FM stations at -300, +150 and +600 kHz, white bytes and a full-scale station."""
    return [station(-300e3), noise(), station(150e3), fm_segment("loud", 999_983, 2), station(600e3)]


def table_iq(n):
    """[5, n, 2]: the segments, each repeated to n samples."""
    return np.stack([np.resize(seg, (n, 2)) for seg in segments()])


def run_incs(rng, k, C):
    """random_incs for C channels with its fixed offsets (0, +-fs/2, 200 kHz) rotated by k, so that the runs of one
    channel are not all at offset 0."""
    incs = random_incs(rng, C + 4)
    r = k % (C + 4)
    return (incs[r:] + incs[:r])[:C]


def walk_runs(R, n, n_rows, seed):
    """N_RUNS runs over n_rows rows: run k reads row k % n_rows with COUNTS[k % 6] channels, so neighbouring runs differ
    in row and count.  Distinct positions: near 2^33 (run 0), one whose first decimated sample first_sample / R wraps
    past 2^32 in the middle of the batch (the middle run), near 2^62 (the last), 0 (run 1), scattered multiples of 4R
    for the rest.  -> [(row, first_sample, increments)]."""
    rng = np.random.default_rng(seed)
    q = 4 * R
    firsts = [q * int(v) for v in rng.integers(1, 2**40, size=N_RUNS)]
    firsts[0] = q * (2**33 // q + 1234)
    firsts[1] = 0
    firsts[ORACLE_RUNS[1]] = R * (2**32 - 4 * (n // (8 * R)))
    firsts[-1] = q * (2**62 // q - 777)
    assert len(set(firsts)) == N_RUNS
    wrap = firsts[ORACLE_RUNS[1]] // R
    assert wrap % 4 == 0 and wrap < 2**32 < wrap + n // R
    runs = [(k % n_rows, firsts[k], run_incs(rng, k, COUNTS[k % len(COUNTS)])) for k in range(N_RUNS)]
    assert max(len(incs) for _, _, incs in runs) == 32
    return runs


def check_oracle(bb, got, iq, R, h, first, incs, channels, what):
    """The uniform call's baseband bb [C, n/R, 2] against the float64 oracle; the runs audio got [C, n/(4R)] against
    the oracle's demodulator on that baseband."""
    hs = np.ones(R) if h is None else h
    tol_bb = 4e-6 * 128 * float(np.abs(np.asarray(hs, np.float64)).sum())
    for c in channels:
        ref = mix_boxcar(iq, R, incs[c], first) if h is None else mix_fir(iq, R, incs[c], h, first)
        err = max(np.abs(bb[c][:, 0] - ref.real).max(), np.abs(bb[c][:, 1] - ref.imag).max())
        assert err <= tol_bb, (what, c, err, tol_bb)
        assert np.abs(got[c] - demodulate(bb[c])).max() <= 1e-4, (what, c)


# ---- the runs call -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("R,T", [(10, 0), (7, 0), (109, 0), (110, 0), (256, 0), (10, 200), (7, 300), (256, 1024)])
def test_runs_walk_equal_uniform_and_oracle(pkg, cuda, R, T):
    """Boxcar at R = 10 (the G = 8 kernel), 7 and 109 (the generic kernel, two stages), 110 and 256 (one stage); FIR at
    (10, 200) (production), (7, 300) (two stages, odd R) and (256, 1024) (one stage, one CTA per SM).  A 64-run table
    over 5 rows: every run equals the uniform call on its row, position and increments, bit for bit."""
    torch = cuda
    n = walk_samples(pkg, R, T, N_RUNS)
    iq = table_iq(n)
    ring = ring_for(pkg, iq, R, T)                 # history all 128: mixes to zero at any position
    h = design(pkg, R, T) if T else None
    taps = dev(torch, h) if T else None
    runs = walk_runs(R, n, len(iq), seed=R * 1000 + T)
    before = pkg.launch_count()
    audio = pkg.fm_channels_exec_runs(ring, runs, taps=taps)
    assert pkg.launch_count() == before + 1
    row = 0
    for k, (s, first, incs) in enumerate(runs):
        C = len(incs)
        want, bb = uniform(pkg, torch, ring, s, first, incs, taps)
        assert torch.equal(audio[row:row + C], want), (k, s, C, first)
        if k in ORACLE_RUNS:
            # a 1024-tap float64 FIR per channel: a few channels suffice there
            channels = range(C) if T < 1024 else sorted({0, C // 2, C - 1})
            check_oracle(bb.cpu().numpy(), audio[row:row + C].cpu().numpy(), iq[s], R, h, first, incs, channels,
                         (k, s, first))
        row += C


def test_one_run_of_32_channels_walks(pkg, cuda):
    """One run of 32 channels at R = 10 (boxcar, G = 8): every tile has four channel groups.  Its first decimated sample
    wraps past 2^32 inside the batch."""
    torch = cuda
    R = 10
    n = walk_samples(pkg, R, 0, 1)
    iq = np.resize(station(150e3), (n, 2))[None]
    ring = ring_for(pkg, iq, R, 0)
    incs = run_incs(np.random.default_rng(32), 3, 32)
    first = R * (2**32 - 4 * (n // (16 * R)))
    audio = pkg.fm_channels_exec_runs(ring, [(0, first, incs)])
    want, bb = uniform(pkg, torch, ring, 0, first, incs, None)
    assert torch.equal(audio, want)
    channels = (0, 2, 31)
    check_oracle({c: bb[c].cpu().numpy() for c in channels}, {c: audio[c].cpu().numpy() for c in channels}, iq[0], R,
                 None, first, incs, channels, first)


@pytest.mark.parametrize("T", [0, 200])
def test_runs_walk_layout(pkg, cuda, T):
    """Through the C ABI at R = 10: a 64-run table whose audio rows are not in table order, with unused rows between
    runs, inside NaN rows wider than n_audio and with more rows than the runs use.  Every unused row and padding value
    stays NaN; every run's rows equal those of the same table with packed rows, bit for bit."""
    torch = cuda
    R = 10
    n = walk_samples(pkg, R, T, N_RUNS)
    n_audio = n // (4 * R)
    iq = table_iq(n)
    ring = ring_for(pkg, iq, R, T)
    taps = dev(torch, design(pkg, R, T)) if T else None
    runs = walk_runs(R, n, len(iq), seed=7000 + T)
    packed = pkg.fm_channels_exec_runs(ring, runs, taps=taps)

    rng = np.random.default_rng(T)
    base, row = {}, 3
    for k in rng.permutation(N_RUNS):
        base[int(k)] = row
        row += len(runs[k][2]) + int(k) % 3         # 0, 1 or 2 unused rows after each run's block
    n_rows = row + 5
    assert sorted(base) == list(range(N_RUNS)) and [base[k] for k in range(N_RUNS)] != sorted(base.values())
    table = (pkg.FmChannelRun * N_RUNS)()
    for k, (s, first, incs) in enumerate(runs):
        t = table[k]
        t.stream, t.n_channels, t.first_sample, t.audio_row = s, len(incs), first, base[k]
        for c, v in enumerate(incs):
            t.phase_inc[c] = v
    full = torch.full((n_rows, n_audio + 37), float("nan"), dtype=torch.float32, device="cuda")
    before = pkg.launch_count()
    rc = raw_runs_call(pkg, ring, table, N_RUNS, full, n_rows, taps=taps.data_ptr() if T else None, T=T)
    torch.cuda.synchronize()
    assert rc == 0, pkg.last_error()
    assert pkg.launch_count() == before + 1
    used = torch.zeros(n_rows, dtype=torch.bool, device="cuda")
    off = 0
    for k, (_, _, incs) in enumerate(runs):
        C = len(incs)
        assert torch.equal(full[base[k]:base[k] + C, :n_audio], packed[off:off + C]), (k, base[k], C)
        used[base[k]:base[k] + C] = True
        off += C
    assert torch.isnan(full[:, n_audio:]).all()
    assert torch.isnan(full[~used]).all()


# ---- the push stream -----------------------------------------------------------------------------------------------

N_DONGLES, GROUP, N_BATCHES, STREAM_T = 32, 16, 3, 200


def stream_batch(pkg):
    """The smallest multiple of the chain tile at which each group's runs launch (only dongles with listeners make
    runs) walks WALK tiles per worker with an odd prime number of tiles per run and a short last tile."""
    tile = int(pkg.lib().b200_chain_tile_samples(10))
    n_runs = min(sum(CYCLE[s % len(CYCLE)] > 0 for s in range(g, g + GROUP)) for g in range(0, N_DONGLES, GROUP))
    w = max(workers(pkg, 10, 0), workers(pkg, 10, STREAM_T))
    batch = tile
    while not all(walk_checks(batch, 10, n_runs, w)[1].values()):
        batch += tile
    check_walk(batch, 10, n_runs, w)
    return batch


@pytest.fixture(scope="module")
def walk_stream(pkg, cuda):
    """(IQ [N_DONGLES, N_BATCHES * batch, 2], batch, centre audio of a stream without a channel sink, its launches).
    Dongle s repeats one of the segments from its own start."""
    batch = stream_batch(pkg)
    n = N_BATCHES * batch
    segs = segments()
    iq = np.stack([np.resize(np.roll(segs[s % len(segs)], -7919 * s, axis=0), (n, 2)) for s in range(N_DONGLES)])
    plain = pkg.PushStream(N_DONGLES, batch, frames=False)
    launches = push_batches(pkg, cuda, plain, iq, batch)
    audio = [joined(plain.audio[s]) for s in range(N_DONGLES)]
    plain.close()
    return iq, batch, audio, launches


def push_batches(pkg, torch, ps, iq, batch):
    """Every dongle pushes its batches in step, so both groups go out whole, each on its own lane.  -> launches."""
    torch.cuda.synchronize()
    before = pkg.launch_count()
    for b in range(N_BATCHES):
        for s in range(N_DONGLES):
            ps.push(s, iq[s, b * batch:(b + 1) * batch])
        ps.poll()
    ps.flush()
    return pkg.launch_count() - before


@pytest.mark.parametrize("T", [0, STREAM_T])
def test_push_stream_channels_walk(pkg, cuda, walk_stream, T):
    """32 dongles in two groups of 16, listener counts cycling through 0, 1, 3, 8, 9, 17 and 32, three batches sized
    so that each group's runs launch walks: every (dongle, id) gets exec_runs over the whole capture, bit for bit, with
    the boxcar and with a 200-tap filter; the centre audio is that of a stream without a channel sink."""
    torch = cuda
    iq, batch, plain_audio, plain_launches = walk_stream
    h = design(pkg, 10, T) if T else None
    ps = pkg.PushStream(N_DONGLES, batch, frames=False, channel_capacity=32)
    if T:
        ps.set_channel_filter(h)
    for s in range(N_DONGLES):
        ps.set_channels(s, *listeners(s))
    # one runs launch per group and batch: no group was split into smaller launches
    assert push_batches(pkg, torch, ps, iq, batch) == plain_launches + 2 * N_BATCHES
    runs = [(s, 0, listeners(s)[0]) for s in range(N_DONGLES) if listeners(s)[1]]
    want = long_runs(pkg, iq, runs, taps=dev(torch, h) if T else None, T=T)
    row = 0
    for s in range(N_DONGLES):
        incs, ids = listeners(s)
        assert sorted(ps.channel_audio[s]) == sorted(ids), s
        for c, cid in enumerate(ids):
            got = joined(ps.channel_audio[s][cid])
            assert got.shape == (N_BATCHES * batch // 40,) and np.array_equal(got, want[row + c]), (s, cid)
        row += len(ids)
        assert np.array_equal(joined(ps.audio[s]), plain_audio[s]), s
    ps.close()
