"""FM channels over a runs table (b200_fm_channels_exec_runs) and on the push stream (b200_stream_set_channel_sink,
_set_channels, _set_channel_filter).

The device-form references are the uniform calls b200_fm_channels_exec / _exec_fir: every run of a table, and every
channel a push stream delivers, must equal what they give on the same row, position and increments, bit for bit.
One test ties the chain to the float64 oracle (mix_boxcar / mix_fir) as the uniform calls' own tests do.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_fm_channels import FS, batch_len, demodulate, incs_tensor, mix_boxcar
from test_gpu_fm_channels_fir import design, dev, mix_fir

COUNTS = (1, 3, 8, 9, 17, 32)


def tune(f):
    return round(f / FS * 2**32) & 0xFFFFFFFF


def random_incs(rng, n):
    """Offsets anywhere in +-fs/2, with 0 and the band edges among them."""
    fixed = [0, tune(FS / 2), tune(-FS / 2), tune(200e3)]
    return [fixed[k] if k < len(fixed) else int(rng.integers(0, 2**32)) for k in range(n)]


def ring_for(pkg, iq, R, T):
    hist = pkg.fm_channels_fir_history_samples(R, T) if T else None
    ring = pkg.StreamRing(iq.shape[0], iq.shape[1], R=R, history=hist)
    ring.load(iq)
    return ring


def uniform(pkg, torch, ring, row, first, incs, taps):
    """The uniform call's audio of `row` at `first` with `incs` (every row gets the same increments)."""
    t = incs_tensor(torch, np.tile(np.asarray(incs, np.int64), (ring.n_streams, 1)))
    audio, bb = pkg.fm_channels_exec(ring, t, first, baseband=True, taps=taps)
    return audio[row], bb[row]


# ------------------------------------------------------------------------------------------------------------------
# the runs call
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("R,T", [(10, 0), (10, 10), (10, 200), (10, 83), (7, 0), (7, 7), (7, 200), (7, 59),
                                 (256, 0), (256, 256), (256, 200)])
def test_runs_equal_uniform_calls(pkg, synth, cuda, R, T):
    """A ragged table -- counts 1, 3, 8, 9, 17 and 32 in one launch, each run at its own position, two pairs of runs
    naming the same row -- gives every run the uniform call's audio on that row, bit for bit.  T = 0 is the boxcar."""
    torch = cuda
    rng = np.random.default_rng(R * 1000 + T)
    S = 4
    n = batch_len(R, 62 * 3 + 10)
    iq = np.stack([synth.s3_fm(n, seed=300 + s, carrier=100e3 * (s - 2)) if s != 2 else synth.s1_noise(n, seed=302)
                   for s in range(S)])
    ring = ring_for(pkg, iq, R, T)
    taps = dev(torch, design(pkg, R, T)) if T else None
    rows = (0, 1, 2, 3, 1, 0)
    runs = [(rows[k], 4 * R * (13 * k + 5 * (k % 2)), random_incs(rng, C)) for k, C in enumerate(COUNTS)]
    before = pkg.launch_count()
    audio = pkg.fm_channels_exec_runs(ring, runs, taps=taps)
    assert pkg.launch_count() == before + 1
    audio = audio.cpu()
    row = 0
    for s, first, incs in runs:
        want, _ = uniform(pkg, torch, ring, s, first, incs, taps)
        assert torch.equal(audio[row:row + len(incs)], want.cpu()), (s, first, len(incs))
        row += len(incs)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [0, 200])
def test_runs_far_positions_and_oracle(pkg, synth, cuda, T):
    """Runs at positions near 2^33 and 2^62 (mixed in one table with one at 0) equal the uniform call there, whose
    baseband is within the float64 oracle's tolerance and whose demodulated baseband is this audio within 1e-4."""
    torch = cuda
    R, n = 10, batch_len(10, 62 * 3)
    iq = synth.s3_fm(n, seed=44, carrier=300e3)[None]
    ring = ring_for(pkg, iq, R, T)                 # history all 128: mixes to zero at any position
    h = design(pkg, R, T) if T else None
    taps = dev(torch, h) if T else None
    incs = [tune(300e3), tune(-777_777.0), 2**31 - 1]
    firsts = (2**33 + 4 * R * 3, 0, 2**62 - 4 * R * 7, 2**62 + 4 * R * 1001)
    firsts = tuple(f - f % (4 * R) for f in firsts)
    audio = pkg.fm_channels_exec_runs(ring, [(0, f, incs) for f in firsts], taps=taps).cpu()
    for k, first in enumerate(firsts):
        want, bb = uniform(pkg, torch, ring, 0, first, incs, taps)
        got = audio[3 * k:3 * k + 3]
        assert torch.equal(got, want.cpu()), first
        bb = bb.cpu().numpy()
        hs = np.ones(R) if h is None else h
        tol_bb = 4e-6 * 128 * float(np.abs(np.asarray(hs, np.float64)).sum())
        for c, inc in enumerate(incs):
            ref = mix_boxcar(iq[0], R, inc, first) if h is None else mix_fir(iq[0], R, inc, h, first)
            err = max(np.abs(bb[c, :, 0] - ref.real).max(), np.abs(bb[c, :, 1] - ref.imag).max())
            assert err <= tol_bb, (first, c, err)
            assert np.abs(got[c].numpy() - demodulate(bb[c])).max() <= 1e-4, (first, c)
    # the position matters: the same samples at 0 mix with other phases
    assert not torch.equal(audio[0:3], audio[3:6])


def raw_runs_call(pkg, ring, table, n_runs, audio, n_rows, taps=None, T=0, **over):
    a = dict(iq=ring.batch.data_ptr(), stride=ring.stride_bytes, S=ring.n_streams, n=ring.n_samples, R=ring.R,
             audio_ptr=audio.data_ptr(), audio_stride=audio.stride(0), rows=n_rows)
    a.update(over)
    return pkg.lib().b200_fm_channels_exec_runs(C.c_void_p(a["iq"]), a["stride"], a["S"], a["n"], a["R"], table,
                                                n_runs, C.c_void_p(a["audio_ptr"]), a["audio_stride"], a["rows"],
                                                C.c_void_p(taps) if taps else None, T, None)


@pytest.mark.gpu
def test_runs_arguments_refused_before_launch(pkg, synth, cuda):
    torch = cuda
    R, n = 10, batch_len(10, 62 * 2)
    ring = ring_for(pkg, np.stack([synth.s3_fm(n, seed=s) for s in range(2)]), R, 0)
    audio = torch.zeros((64, n // (4 * R) + 4), dtype=torch.float32, device="cuda")
    taps = dev(torch, design(pkg, R, 200))

    def table(*runs):
        t = (pkg.FmChannelRun * 65)()
        for k, (s, nc, first, row) in enumerate(runs):
            t[k].stream, t[k].n_channels, t[k].first_sample, t[k].audio_row = s, nc, first, row
        return t

    good = table((0, 2, 0, 0), (1, 3, 40, 2))
    before = pkg.launch_count()
    ERR_ARG, ERR_ALIGN = -1, -4
    assert raw_runs_call(pkg, ring, good, 0, audio, 64) == ERR_ARG                     # no runs
    assert raw_runs_call(pkg, ring, table(*[(0, 1, 0, k) for k in range(65)]), 65, audio, 65) == ERR_ARG
    assert raw_runs_call(pkg, ring, table((2, 1, 0, 0)), 1, audio, 64) == ERR_ARG       # stream out of range
    assert raw_runs_call(pkg, ring, table((-1, 1, 0, 0)), 1, audio, 64) == ERR_ARG
    assert raw_runs_call(pkg, ring, table((0, 0, 0, 0)), 1, audio, 64) == ERR_ARG       # no channels
    assert raw_runs_call(pkg, ring, table((0, 33, 0, 0)), 1, audio, 64) == ERR_ARG
    assert raw_runs_call(pkg, ring, table((0, 1, 20, 0)), 1, audio, 64) == ERR_ARG      # not a multiple of 4R
    assert raw_runs_call(pkg, ring, table((0, 1, -40, 0)), 1, audio, 64) == ERR_ARG
    assert raw_runs_call(pkg, ring, table((0, 2, 0, 63)), 1, audio, 64) == ERR_ARG      # rows past n_audio_rows
    assert raw_runs_call(pkg, ring, table((0, 2, 0, -1)), 1, audio, 64) == ERR_ARG
    assert raw_runs_call(pkg, ring, table((0, 3, 0, 0), (1, 2, 0, 2)), 2, audio, 64) == ERR_ARG   # rows overlap
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, R=0) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, n=n + 4) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, audio_stride=n // (4 * R) - 1) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, iq=0) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, iq=ring.batch.data_ptr() + 8) == ERR_ALIGN
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, stride=ring.stride_bytes + 8) == ERR_ALIGN
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, audio_ptr=audio.data_ptr() + 2) == ERR_ALIGN
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, taps=taps.data_ptr(), T=0) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, taps=None, T=200) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, taps=taps.data_ptr(), T=1025) == ERR_ARG
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, taps=taps.data_ptr() + 2, T=200) == ERR_ALIGN
    # R out of range with taps (no (R, T) pair in range fails the shared-memory budget: R = 256, T = 1024 fits)
    assert raw_runs_call(pkg, ring, good, 2, audio, 64, R=257, n=8 * 257, taps=taps.data_ptr(), T=1024) == ERR_ARG
    # n_runs x tiles at 2^31 is refused before anything is touched (the IQ pointer is never read)
    huge = 4 * R * 62 * (2**31 // 64 + 1)
    assert raw_runs_call(pkg, ring, table(*[(0, 1, 0, k) for k in range(64)]), 64, audio, 64, n=huge,
                         audio_stride=huge // (4 * R)) == ERR_ARG
    assert pkg.launch_count() == before
    # the binding: a ring whose history is too short for the taps
    with pytest.raises(pkg.B200Error):
        pkg.fm_channels_exec_runs(ring, [(0, 0, [1])], taps=taps)
    assert pkg.launch_count() == before
    assert raw_runs_call(pkg, ring, good, 2, audio, 64) == 0
    assert pkg.launch_count() == before + 1


# ------------------------------------------------------------------------------------------------------------------
# the push stream
# ------------------------------------------------------------------------------------------------------------------

N_STREAMS, BATCH, N_BATCHES = 20, 5120 * 4, 3
CYCLE = (0, 1, 3, 8, 9, 17, 32)


def listeners(s):
    """Dongle s's channels: a count cycling through 0, 1, 3, 8, 9, 17, 32; increments and ids from s."""
    rng = np.random.default_rng(500 + s)
    n = CYCLE[s % len(CYCLE)]
    return random_incs(rng, n), [1000 * s + 7 * c + 3 for c in range(n)]


def stream_iq(synth, n=N_BATCHES * BATCH, n_streams=N_STREAMS):
    return np.stack([synth.s3_fm(n, seed=160 + s, carrier=50e3 * (s % 5 - 2)) for s in range(n_streams)])


def push_stragglers(ps, iq):
    """test_push_stream_groups_and_stragglers' pattern: stream 5 pushes its three batches first, stream 18 never
    finishes its last one."""
    ps.push(5, iq[5])
    for b in range(N_BATCHES):
        for s in range(N_STREAMS):
            if s == 5:
                continue
            hi = (b + 1) * BATCH if not (s == 18 and b == 2) else (b + 1) * BATCH - 1000
            ps.push(s, iq[s, b * BATCH:hi])
        ps.poll()
    ps.flush()


def joined(chunks):
    chunks = sorted(chunks, key=lambda t: t[0])
    n = len(chunks[0][1])
    assert [f for f, _ in chunks] == [k * n for k in range(len(chunks))]      # in order, once each, from 0
    return np.concatenate([a for _, a in chunks])


def long_runs(pkg, iq, runs, R=10, taps=None, T=0):
    """exec_runs over the whole capture as one batch (three carried batches give the same bits as one long one)."""
    ring = ring_for(pkg, iq, R, T)
    return pkg.fm_channels_exec_runs(ring, runs, taps=taps).cpu().numpy()


@pytest.mark.gpu
def test_push_stream_channels_equal_exec_runs(pkg, synth, cuda):
    """20 dongles (two groups) with 0 to 32 channels each and the straggler pattern: every (dongle, id) gets the audio
    of exec_runs over the same samples, bit for bit; dongles without channels get no channel calls.  Spectra, payloads
    and centre audio are those of a stream without a channel sink, bit for bit."""
    iq = stream_iq(synth)
    ps = pkg.PushStream(N_STREAMS, BATCH, payload_K=6, channel_capacity=32)
    plain = pkg.PushStream(N_STREAMS, BATCH, payload_K=6)
    for s in range(N_STREAMS):
        ps.set_channels(s, *listeners(s))
    push_stragglers(ps, iq)
    push_stragglers(plain, iq)
    runs = [(s, 0, listeners(s)[0]) for s in range(N_STREAMS) if listeners(s)[1]]
    want = long_runs(pkg, iq, runs)
    row = 0
    for s in range(N_STREAMS):
        incs, ids = listeners(s)
        assert sorted(ps.channel_audio[s]) == sorted(ids)
        n_done = (2 if s == 18 else 3) * BATCH // 40
        for c, cid in enumerate(ids):
            got = joined(ps.channel_audio[s][cid])
            assert got.shape == (n_done,) and np.array_equal(got, want[row + c, :n_done]), (s, cid)
        row += len(ids)
        assert np.array_equal(joined(ps.audio[s]), joined(plain.audio[s]))
        assert np.array_equal(joined(ps.spectra[s]), joined(plain.spectra[s]))
        assert [f for f, _, _ in ps.payloads[s]] == [f for f, _, _ in plain.payloads[s]]
        assert all(np.array_equal(a, b) for (_, _, a), (_, _, b) in zip(ps.payloads[s], plain.payloads[s]))
    ps.close()
    plain.close()


@pytest.mark.gpu
def test_push_stream_channel_launches(pkg, synth, cuda):
    """Dongles that push in step go out as one run per group; channels add one launch per run that has any (here
    both groups, then only the first) and nothing for a run without."""
    iq = stream_iq(synth)

    def launches(sets):
        ps = pkg.PushStream(N_STREAMS, BATCH, channel_capacity=32)
        for s, (incs, ids) in sets.items():
            ps.set_channels(s, incs, ids)
        before = pkg.launch_count()
        for b in range(N_BATCHES):
            for s in range(N_STREAMS):
                ps.push(s, iq[s, b * BATCH:(b + 1) * BATCH])
            ps.poll()
        ps.flush()
        n = pkg.launch_count() - before
        ps.close()
        return n

    base = launches({})
    assert launches({s: listeners(s) for s in range(N_STREAMS)}) == base + 2 * N_BATCHES
    assert launches({3: listeners(3)}) == base + N_BATCHES


@pytest.mark.gpu
def test_push_stream_retune_join_leave(pkg, synth, cuda):
    """Changes between pushes: a channel retuned, joined or left at batch b gives exactly the slice of an always-present
    channel from batch b on.  A batch takes the set current at its last sample: a change made while it is partly
    filled applies to it, and a change made while a full batch waits for the rest of its group does not."""
    n_streams = 2
    iq = stream_iq(synth, n_streams=n_streams)
    A, B, J = tune(-300e3), tune(400e3), tune(123_456.0)
    ref = long_runs(pkg, iq, [(0, 0, [A, B]), (1, 0, [J])])
    na = BATCH // 40
    ps = pkg.PushStream(n_streams, BATCH, channel_capacity=4)
    ps.set_channels(0, [A], [7])
    # batch 0: dongle 0 fills first and waits for dongle 1; retuning it now must not touch that batch
    ps.push(0, iq[0, :BATCH])
    ps.set_channels(0, [B], [7])
    ps.push(1, iq[1, :BATCH])
    # batch 1: dongle 1 joins half-way through its batch, which already counts for it
    ps.push(0, iq[0, BATCH:2 * BATCH])
    ps.push(1, iq[1, BATCH:BATCH + 777])
    assert ps.pending(1) == 777
    ps.set_channels(1, [J], [9])
    ps.push(1, iq[1, BATCH + 777:2 * BATCH])
    # batch 2: dongle 0's listener leaves
    ps.set_channels(0, [], [])
    ps.push(0, iq[0, 2 * BATCH:])
    ps.push(1, iq[1, 2 * BATCH:])
    ps.flush()
    got0 = sorted(ps.channel_audio[0][7], key=lambda t: t[0])
    assert [f for f, _ in got0] == [0, na]
    assert np.array_equal(got0[0][1], ref[0, :na])             # A, set before the batch filled
    assert np.array_equal(got0[1][1], ref[1, na:2 * na])       # B from batch 1 on
    got1 = sorted(ps.channel_audio[1][9], key=lambda t: t[0])
    assert [f for f, _ in got1] == [na, 2 * na]
    assert np.array_equal(np.concatenate([a for _, a in got1]), ref[2, na:])
    ps.close()


@pytest.mark.gpu
def test_push_stream_chunking_does_not_matter(pkg, synth, cuda):
    """Pushes of 7777 samples give the channel audio of pushes of 131072, bit for bit."""
    n_streams = 3
    iq = stream_iq(synth, n=7 * BATCH, n_streams=n_streams)
    out = []
    for chunk in (7777, 131072):
        ps = pkg.PushStream(n_streams, BATCH, channel_capacity=32)
        for s in range(n_streams):
            ps.set_channels(s, *listeners(s + 3))
        for pos in range(0, iq.shape[1], chunk):
            for s in range(n_streams):
                ps.push(s, iq[s, pos:pos + chunk])
        ps.flush()
        out.append({(s, cid): joined(v) for s in range(n_streams) for cid, v in ps.channel_audio[s].items()})
        ps.close()
    assert out[0].keys() == out[1].keys() and len(out[0]) == sum(len(listeners(s + 3)[1]) for s in range(n_streams))
    assert all(np.array_equal(out[0][k], out[1][k]) and len(out[0][k]) == 7 * BATCH // 40 for k in out[0])


@pytest.mark.gpu
def test_push_stream_channel_filter(pkg, synth, cuda):
    """With a 200-tap filter the rows carry H(10, 200) samples of history: three carried batches equal exec_runs with
    those taps over the whole capture, and the centre outputs stay those of a stream without channels."""
    torch = cuda
    n_streams, T = 3, 200
    iq = stream_iq(synth, n_streams=n_streams)
    h = design(pkg, 10, T)
    ps = pkg.PushStream(n_streams, BATCH, payload_K=6, channel_capacity=8)
    ps.set_channel_filter(h)
    plain = pkg.PushStream(n_streams, BATCH, payload_K=6)
    sets = {s: listeners(s + 1) for s in range(n_streams)}
    for s, (incs, ids) in sets.items():
        ps.set_channels(s, incs, ids)
    for p in (ps, plain):
        for pos in range(0, iq.shape[1], 131072):
            for s in range(n_streams):
                p.push(s, iq[s, pos:pos + 131072])
        p.flush()
    with pytest.raises(pkg.B200Error):
        ps.set_channel_filter(h)                   # after a push
    want = long_runs(pkg, iq, [(s, 0, sets[s][0]) for s in range(n_streams)], taps=dev(torch, h), T=T)
    row = 0
    for s in range(n_streams):
        for c, cid in enumerate(sets[s][1]):
            assert np.array_equal(joined(ps.channel_audio[s][cid]), want[row + c]), (s, cid)
        row += len(sets[s][1])
        assert np.array_equal(joined(ps.audio[s]), joined(plain.audio[s]))
        assert np.array_equal(joined(ps.spectra[s]), joined(plain.spectra[s]))
        assert all(np.array_equal(a, b) for (_, _, a), (_, _, b) in zip(ps.payloads[s], plain.payloads[s]))
    ps.close()
    plain.close()
    # a history longer than the batch: R = 256 batches of 8192 samples, 1024 taps need 8960
    big = pkg.PushStream(1, 8192, R=256, channel_capacity=1)
    with pytest.raises(pkg.B200Error):
        big.set_channel_filter(np.ones(1024, np.float32))
    big.set_channel_filter(np.ones(256, np.float32))          # 8192: fits exactly
    big.close()


@pytest.mark.gpu
def test_push_stream_channel_arguments(pkg, cuda):
    ps = pkg.PushStream(2, BATCH)
    with pytest.raises(pkg.B200Error):
        ps.set_channels(0, [1], [1])                # no channel sink yet
    L = pkg.lib()
    assert L.b200_stream_set_channel_sink(ps.h, 0, ps._on_channel) == -1
    assert L.b200_stream_set_channel_sink(ps.h, 33, ps._on_channel) == -1
    assert L.b200_stream_set_channel_sink(ps.h, 4, ps._on_channel) == 0
    assert L.b200_stream_set_channel_sink(ps.h, 5, ps._on_channel) == -1     # the capacity stays
    for args in ((2, [1], [1]), (-1, [1], [1]), (0, [1] * 5, list(range(5))), (0, [1, 2], [3, 3])):
        with pytest.raises(pkg.B200Error):
            ps.set_channels(*args)
    ps.set_channels(0, [1, 2, 3, 4], [1, 2, 3, 4])
    ps.set_channels(0, [], [])
    ps.close()
