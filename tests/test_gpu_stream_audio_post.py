"""Audio post-processing over a row table (b200_audio_post_rows) and on the push stream (b200_stream_set_audio_post).

The references are the uniform call b200_audio_post: every row of a table, and every centre and channel batch a push
stream delivers, must equal what it gives on the same row with the same state, bit for bit.  On the stream that state
is the dongle's (centre) or the listener id's (channels), carried from batch to batch or restarted from zero where
the listener rules of include/b200sdr.h say so.  One test ties a listener's whole output to the oracle's sequential
definitions (po.deemphasis, po.resample_15_16).
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_stream_channels import BATCH, N_BATCHES, N_STREAMS, joined, listeners, push_stragglers, stream_iq, tune

BOTH = 2 | 4                 # AUDIO_DEEMPH_75US | AUDIO_RESAMPLE_48K
FLAG_CASES = [pytest.param(f, r, id=f"{f}-{r:.0f}") for r in (51200.0, 512000.0)
              for f in ("AUDIO_DEEMPH_50US", "AUDIO_DEEMPH_75US", "AUDIO_RESAMPLE_48K", "both")]


def flags_of(pkg, name):
    return pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K if name == "both" else getattr(pkg, name)


def zeros(torch, *shape):
    return torch.zeros(shape, dtype=torch.float32, device="cuda")


# ------------------------------------------------------------------------------------------------------------------
# the rows call
# ------------------------------------------------------------------------------------------------------------------

def random_table(rng, n_rows, n_audio_rows, n_out_rows, n_state_rows):
    """Scattered, permuted rows: input rows may repeat, output and state rows may not; about half of them fresh."""
    audio = rng.integers(0, n_audio_rows, n_rows)
    out = rng.permutation(n_out_rows)[:n_rows]
    state = rng.permutation(n_state_rows)[:n_rows]
    fresh = rng.integers(0, 2, n_rows)
    return [(int(a), int(o), int(s), int(f)) for a, o, s, f in zip(audio, out, state, fresh)]


def uniform_reference(pkg, torch, x, state, table, flags, rate):
    """The uniform call on each table row with that row's state (zero if fresh): one call over the gathered rows, whose
    rows are independent.  -> (outputs in table order, next states in table order)."""
    a = torch.tensor([r[0] for r in table], device="cuda")
    s = torch.tensor([r[2] for r in table], device="cuda")
    fresh = torch.tensor([bool(r[3]) for r in table], device="cuda")
    st = state[s].clone()
    st[fresh] = 0.0
    out = pkg.audio_post(x[a].contiguous(), st, flags, rate)
    return out, st


@pytest.mark.gpu
@pytest.mark.parametrize("flags_name,rate", FLAG_CASES)
def test_rows_equal_uniform_call(pkg, cuda, flags_name, rate):
    """Tables of 1024, 37 and 1 rows over 3 chunks and a short one: each row's output and next state are the uniform
    call's on that row with that state (zeroed if fresh), bit for bit; rows and states outside the table are untouched."""
    torch = cuda
    flags = flags_of(pkg, flags_name)
    rng = np.random.default_rng(int(rate) + flags)
    n = 3 * 1024 + 16 * 7
    n_out = int(pkg.lib().b200_audio_post_out_samples(n, flags))
    x = torch.as_tensor(rng.uniform(-1, 1, size=(300, n)).astype(np.float32)).cuda()
    for n_rows in (pkg.AUDIO_POST_MAX_ROWS, 37, 1):
        n_out_rows, n_state_rows = n_rows + 60, n_rows + 40
        state = torch.as_tensor(rng.uniform(-1, 1, size=(n_state_rows, pkg.AUDIO_POST_STATE_FLOATS))
                                .astype(np.float32)).cuda()
        before_state = state.clone()
        out = torch.full((n_out_rows, n_out), float("nan"), dtype=torch.float32, device="cuda")
        table = random_table(rng, n_rows, x.shape[0], n_out_rows, n_state_rows)
        launches = pkg.launch_count()
        pkg.audio_post_rows(x, table, state, flags, rate, out=out)
        assert pkg.launch_count() == launches + 2
        want, want_state = uniform_reference(pkg, torch, x, before_state, table, flags, rate)
        o = torch.tensor([r[1] for r in table], device="cuda")
        s = torch.tensor([r[2] for r in table], device="cuda")
        assert torch.equal(out[o], want)
        assert torch.equal(state[s][:, :16], want_state[:, :16])
        others = torch.ones(n_out_rows, dtype=torch.bool, device="cuda")
        others[o] = False
        assert torch.isnan(out[others]).all()
        others = torch.ones(n_state_rows, dtype=torch.bool, device="cuda")
        others[s] = False
        assert torch.equal(state[others], before_state[others])


@pytest.mark.gpu
@pytest.mark.parametrize("flags_name,rate", FLAG_CASES)
def test_rows_and_uniform_calls_interchange(pkg, cuda, flags_name, rate):
    """The uniform call on batch 0, then the rows call (permuted rows, carried state) on batch 1, equals the uniform
    call twice: both advance the same state layout."""
    torch = cuda
    flags = flags_of(pkg, flags_name)
    rng = np.random.default_rng(7)
    S, n = 6, 2048 + 16 * 3
    x = [torch.as_tensor(rng.uniform(-1, 1, size=(S, n)).astype(np.float32)).cuda() for _ in range(2)]
    st_a, st_b = zeros(torch, S, pkg.AUDIO_POST_STATE_FLOATS), zeros(torch, S, pkg.AUDIO_POST_STATE_FLOATS)
    pkg.audio_post(x[0], st_a, flags, rate)
    want = pkg.audio_post(x[1], st_a, flags, rate)
    pkg.audio_post(x[0], st_b, flags, rate)
    perm = rng.permutation(S)
    # row k reads input perm[k] with its state perm[k] and writes output row (perm[k] + 2) % S
    got = pkg.audio_post_rows(x[1], [(int(p), (int(p) + 2) % S, int(p), 0) for p in perm], st_b, flags, rate)
    assert torch.equal(got[[(s + 2) % S for s in range(S)]], want)
    assert torch.equal(st_b[:, :16], st_a[:, :16])


def raw_rows_call(pkg, x, table, n_rows, st, y, **over):
    """b200_audio_post_rows on input x, state st and output y, any argument replaced by a keyword of `over`."""
    a = dict(audio=x.data_ptr(), audio_stride=x.stride(0), audio_rows=x.shape[0], n=x.shape[1], rate=51200.0,
             flags=BOTH, state=st.data_ptr(), state_rows=st.shape[0], out=y.data_ptr(), out_stride=y.stride(0),
             out_rows=y.shape[0], table=table)
    a.update(over)
    ptr = lambda k: C.c_void_p(a[k]) if a[k] else None
    return pkg.lib().b200_audio_post_rows(ptr("audio"), a["audio_stride"], a["audio_rows"], a["n"], a["rate"],
                                          a["flags"], a["table"], n_rows, ptr("state"), a["state_rows"], ptr("out"),
                                          a["out_stride"], a["out_rows"], None)


@pytest.mark.gpu
def test_rows_arguments_refused_before_launch(pkg, cuda):
    torch = cuda
    n = 1024 + 32
    audio = zeros(torch, 8, n)
    state = zeros(torch, 8, pkg.AUDIO_POST_STATE_FLOATS)
    out = zeros(torch, 8, n)                       # wide enough without the resampler too

    def table(*rows):
        t = (pkg.AudioPostRow * (pkg.AUDIO_POST_MAX_ROWS + 1))()
        for k, r in enumerate(rows):
            t[k].audio_row, t[k].out_row, t[k].state_row, t[k].fresh = r
        return t

    good = table((0, 1, 2, 0), (0, 2, 3, 1))
    ERR_ARG, ERR_ALIGN = -1, -4
    before = pkg.launch_count()
    assert raw_rows_call(pkg, audio, good, 0, state, out) == ERR_ARG                     # no rows
    assert raw_rows_call(pkg, audio, table(*[(0, 0, 0, 0)] * 1025), 1025, state, out) == ERR_ARG
    assert raw_rows_call(pkg, audio, None, 2, state, out) == ERR_ARG                     # no table
    for bad in ((-1, 0, 0, 0), (8, 0, 0, 0), (0, -1, 0, 0), (0, 8, 0, 0), (0, 0, -1, 0), (0, 0, 8, 0)):
        assert raw_rows_call(pkg, audio, table(bad), 1, state, out) == ERR_ARG, bad     # row index outside its count
    assert raw_rows_call(pkg, audio, table((0, 1, 2, 0), (1, 1, 3, 0)), 2, state, out) == ERR_ARG   # shared out_row
    assert raw_rows_call(pkg, audio, table((0, 1, 2, 0), (1, 3, 2, 1)), 2, state, out) == ERR_ARG   # shared state_row
    assert raw_rows_call(pkg, audio, good, 2, state, out, audio_stride=n - 1) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, out_stride=n // 16 * 15 - 1) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, flags=0, out_stride=n - 1) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, audio=0) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, state=0) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, out=0) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, audio=audio.data_ptr() + 2) == ERR_ALIGN
    assert raw_rows_call(pkg, audio, good, 2, state, out, state=state.data_ptr() + 2) == ERR_ALIGN
    assert raw_rows_call(pkg, audio, good, 2, state, out, out=out.data_ptr() + 2) == ERR_ALIGN
    # the output inside the input block (its last row), or the very same block
    assert raw_rows_call(pkg, audio, good, 2, state, out, out=audio[5].data_ptr(), out_rows=3,
                         out_stride=n) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, out=audio.data_ptr(), out_stride=n) == ERR_ARG
    # what b200_audio_post refuses: both time constants, unknown bits, no rate, a run-in past 1024, a resampler
    # length that is not a multiple of 16, a negative length
    assert raw_rows_call(pkg, audio, good, 2, state, out, flags=3) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, flags=8) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, rate=0.0) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, rate=2e6) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, n=n - 8) == ERR_ARG
    assert raw_rows_call(pkg, audio, good, 2, state, out, n=-16) == ERR_ARG
    assert pkg.launch_count() == before
    assert raw_rows_call(pkg, audio, good, 2, state, out) == 0
    assert pkg.launch_count() == before + 2


# ------------------------------------------------------------------------------------------------------------------
# the push stream
# ------------------------------------------------------------------------------------------------------------------

def batches(chunks):
    """A sink's (first_sample, audio) calls -> the list of batches in order (checked to be contiguous from 0)."""
    chunks = sorted(chunks, key=lambda t: t[0])
    joined(chunks)
    return [a for _, a in chunks]


def post_reference(pkg, torch, rows, flags, rate=51200.0):
    """rows: per output row, its raw batches in order.  -> per row, audio_post batch by batch with the row's state
    carried from zero."""
    state = zeros(torch, len(rows), pkg.AUDIO_POST_STATE_FLOATS)
    out = [[] for _ in rows]
    for b in range(max(len(r) for r in rows)):
        idx = [k for k, r in enumerate(rows) if len(r) > b]
        sel = torch.tensor(idx, device="cuda")
        st = state[sel]
        y = pkg.audio_post(torch.as_tensor(np.stack([rows[k][b] for k in idx])).cuda(), st, flags, rate).cpu().numpy()
        state[sel] = st
        for j, k in enumerate(idx):
            out[k].append(y[j])
    return out


def stream_pair(pkg, flags, iq, push, n_streams=N_STREAMS, sets=None, capacity=32):
    """A stream with post-processing and one without, same listeners, pushed the same way."""
    ps = pkg.PushStream(n_streams, BATCH, payload_K=6, channel_capacity=capacity)
    ps.set_audio_post(flags)
    plain = pkg.PushStream(n_streams, BATCH, payload_K=6, channel_capacity=capacity)
    for s in range(n_streams):
        incs, ids = sets[s] if sets else listeners(s)
        ps.set_channels(s, incs, ids)
        plain.set_channels(s, incs, ids)
    push(ps, iq)
    push(plain, iq)
    return ps, plain


@pytest.mark.gpu
@pytest.mark.parametrize("flags_name", ["both", "AUDIO_DEEMPH_50US"])
def test_push_stream_audio_post_equals_reference(pkg, synth, cuda, po, flags_name):
    """20 dongles in two groups, stragglers, 0 to 32 listeners each: centre and channel audio are audio_post over the
    post-off stream's rows, batch by batch with carried state, bit for bit, at the output rate.  Spectra and payloads
    are the post-off stream's.  One dongle's and one listener's whole output match the sequential definitions."""
    torch = cuda
    flags = flags_of(pkg, flags_name)
    n_out = int(pkg.lib().b200_audio_post_out_samples(BATCH // 40, flags))
    iq = stream_iq(synth)
    ps, plain = stream_pair(pkg, flags, iq, push_stragglers)
    keys = [(s, None) for s in range(N_STREAMS)] + [(s, cid) for s in range(N_STREAMS) for cid in listeners(s)[1]]
    raw = [batches(plain.audio[s] if cid is None else plain.channel_audio[s][cid]) for s, cid in keys]
    want = post_reference(pkg, torch, raw, flags)
    for (s, cid), w, r in zip(keys, want, raw):
        got = ps.audio[s] if cid is None else ps.channel_audio[s][cid]
        assert [f for f, _ in sorted(got, key=lambda t: t[0])] == [b * n_out for b in range(len(r))], (s, cid)
        assert all(len(a) == n_out for _, a in got)
        assert np.array_equal(joined(got), np.concatenate(w)), (s, cid)
    assert sorted(len(ps.channel_audio[s]) for s in range(N_STREAMS)) == sorted(len(listeners(s)[1])
                                                                                for s in range(N_STREAMS))
    for s in range(N_STREAMS):
        assert np.array_equal(joined(ps.spectra[s]), joined(plain.spectra[s]))
        assert [f for f, _, _ in ps.payloads[s]] == [f for f, _, _ in plain.payloads[s]]
        assert all(np.array_equal(a, b) for (_, _, a), (_, _, b) in zip(ps.payloads[s], plain.payloads[s]))
    # the sequential definitions over a whole output: dongle 6's centre audio and its listener with the most channels
    tau = 50e-6 if flags & pkg.AUDIO_DEEMPH_50US else 75e-6
    for got, x in ((joined(ps.audio[6]), joined(plain.audio[6])),
                   (joined(ps.channel_audio[6][listeners(6)[1][5]]), joined(plain.channel_audio[6][listeners(6)[1][5]]))):
        y, _ = po.deemphasis(x, 51200.0, tau)
        if flags & pkg.AUDIO_RESAMPLE_48K:
            y, _ = po.resample_15_16(y)
        assert np.abs(got - y).max() <= 2e-6
    ps.close()
    plain.close()


def push_batch(ps, iq, b, streams):
    for s in streams:
        ps.push(s, iq[s, b * BATCH:(b + 1) * BATCH])


@pytest.mark.gpu
def test_push_stream_listener_state_rules(pkg, synth, cuda):
    """One scripted sequence on dongle 0 (dongle 1 keeps one listener throughout): a retune and a reorder keep state;
    a listener that joins as another leaves takes the freed slot from zero; an id gone for a batch comes back from
    zero; every listener starts from zero after a batch submitted without a channel sink.  Each delivered batch equals
    audio_post of the post-off stream's batch with the state the rule gives: carried, or zero where it says fresh."""
    torch = cuda
    A, B, Cc, E = 11, 22, 33, 44
    f = {A: tune(-300e3), B: tune(250e3), Cc: tune(123_456.0), E: tune(-50e3)}
    A2 = tune(410e3)
    script = [                             # dongle 0's set per batch (id, increment); fresh ids of that batch
        ([(A, f[A]), (B, f[B])], {A, B}),
        ([(A, A2), (B, f[B])], set()),     # A retuned
        ([(B, f[B]), (A, A2)], set()),     # reordered
        ([(A, A2), (Cc, f[Cc])], {Cc}),    # B leaves, C joins into B's slot
        ([(Cc, f[Cc])], set()),            # A leaves
        ([(Cc, f[Cc]), (A, A2)], {A}),     # A back two batches after its last
        ([(Cc, f[Cc]), (A, A2)], None),    # submitted without a channel sink
        ([(Cc, f[Cc]), (A, A2)], {Cc, A}),
    ]
    n_b = len(script)
    iq = stream_iq(synth, n=n_b * BATCH, n_streams=2)
    ps = pkg.PushStream(2, BATCH, channel_capacity=4)
    ps.set_audio_post(BOTH)
    plain = pkg.PushStream(2, BATCH, channel_capacity=4)
    ps.set_channels(1, [f[E]], [E])
    plain.set_channels(1, [f[E]], [E])
    L = pkg.lib()
    for b, (chans, _) in enumerate(script):
        for p in (ps, plain):
            p.set_channels(0, [i for _, i in chans], [c for c, _ in chans])
        if script[b][1] is None:
            assert L.b200_stream_set_channel_sink(ps.h, 4, pkg.binding.CHANNEL_SINK()) == 0
        push_batch(ps, iq, b, (0, 1))
        push_batch(plain, iq, b, (0, 1))
        ps.flush()
        if script[b][1] is None:
            assert L.b200_stream_set_channel_sink(ps.h, 4, ps._on_channel) == 0
    plain.flush()
    n_out = BATCH // 40 // 16 * 15
    raw = {(s, cid): dict(v) for s in range(2) for cid, v in plain.channel_audio[s].items()}
    got = {(s, cid): dict(v) for s in range(2) for cid, v in ps.channel_audio[s].items()}
    state = {}
    for b, (chans, fresh) in enumerate(script):
        ids = [(0, c) for c, _ in chans] + [(1, E)]
        if fresh is None:
            assert all(b * n_out not in got[k] for k in ids)
            continue
        for k in ids:
            if k[1] in fresh or (k == (1, E) and (b == 0 or script[b - 1][1] is None)):
                state[k] = zeros(torch, 1, pkg.AUDIO_POST_STATE_FLOATS)
            x = torch.as_tensor(raw[k][b * (BATCH // 40)][None]).cuda()
            want = pkg.audio_post(x, state[k], BOTH).cpu().numpy()[0]
            assert np.array_equal(got[k][b * n_out], want), (b, k)
    # every delivered batch was checked: nothing for ids outside their batches' sets
    assert sum(len(v) for v in got.values()) == sum(len(c) + 1 for c, fr in script if fr is not None)
    # the centre audio carries one state per dongle through all of it
    want = post_reference(pkg, torch, [batches(plain.audio[s]) for s in range(2)], BOTH)
    for s in range(2):
        assert np.array_equal(joined(ps.audio[s]), np.concatenate(want[s]))
    ps.close()
    plain.close()


def push_in_step(ps, iq, chunk=131072):
    for pos in range(0, iq.shape[1], chunk):
        for s in range(iq.shape[0]):
            ps.push(s, iq[s, pos:pos + chunk])
        ps.poll()
    ps.flush()


def outputs(ps):
    return ({s: joined(v) for s, v in enumerate(ps.audio)},
            {(s, cid): joined(v) for s in range(ps.n_streams) for cid, v in ps.channel_audio[s].items()})


@pytest.mark.gpu
def test_push_stream_audio_post_setter(pkg, synth, cuda):
    """Refused after a push and for the resampler on 8 audio samples a batch; setter and channel sink in either order
    give the same audio, and the reference's; flags 0 gives the raw stream bit for bit; pushes of 7777 samples give the
    audio of pushes of 131072."""
    torch = cuda
    n_streams = 3
    sets = {s: listeners(s + 3) for s in range(n_streams)}
    iq = stream_iq(synth, n=5 * BATCH, n_streams=n_streams)

    ps = pkg.PushStream(1, BATCH)
    ps.push(0, iq[0, :100])
    with pytest.raises(pkg.B200Error):
        ps.set_audio_post(BOTH)
    ps.close()
    # R = 256: a batch of 8192 has 8 audio samples, 16384 has 16
    for batch, ok in ((8192, False), (16384, True)):
        ps = pkg.PushStream(1, batch, R=256)
        ps.set_audio_post(pkg.AUDIO_DEEMPH_75US, 2000.0)
        if ok:
            ps.set_audio_post(BOTH, 2000.0)
        else:
            with pytest.raises(pkg.B200Error):
                ps.set_audio_post(BOTH, 2000.0)
        ps.close()
    ps = pkg.PushStream(1, BATCH)
    for flags, rate in ((3, 51200.0), (8, 51200.0), (BOTH, 0.0), (BOTH, 2e6)):
        with pytest.raises(pkg.B200Error):
            ps.set_audio_post(flags, rate)
    ps.close()

    def run(order, flags, chunk=131072):
        ps = pkg.PushStream(n_streams, BATCH)
        if order == "setter first":
            ps.set_audio_post(flags)
        assert pkg.lib().b200_stream_set_channel_sink(ps.h, 32, ps._on_channel) == 0
        if order == "sink first":
            ps.set_audio_post(flags)
        for s in range(n_streams):
            ps.set_channels(s, *sets[s])
        push_in_step(ps, iq, chunk)
        out = outputs(ps)
        ps.close()
        return out

    setter_first = run("setter first", BOTH)
    sink_first = run("sink first", BOTH)
    small_pushes = run("setter first", BOTH, 7777)
    raw = run(None, 0)
    off = run("setter first", 0)
    assert len(setter_first[1]) == sum(len(sets[s][1]) for s in range(n_streams))
    for got in (sink_first, small_pushes):
        for a, b in zip(setter_first, got):
            assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    for a, b in zip(raw, off):
        assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    keys = list(raw[1])
    n_audio = BATCH // 40
    split = lambda x: [x[i:i + n_audio] for i in range(0, len(x), n_audio)]
    want = post_reference(pkg, torch, [split(raw[0][s]) for s in range(n_streams)] + [split(raw[1][k]) for k in keys],
                          BOTH)
    for s in range(n_streams):
        assert np.array_equal(setter_first[0][s], np.concatenate(want[s]))
    for k, w in zip(keys, want[n_streams:]):
        assert np.array_equal(setter_first[1][k], np.concatenate(w)), k


@pytest.mark.gpu
def test_push_stream_audio_post_launches(pkg, synth, cuda):
    """Dongles pushing in step go out as one run per group and batch.  Post-processing adds two launches per run for
    the centre audio and two more per run with listeners (here both groups, then only the first, then neither)."""
    iq = stream_iq(synth)

    def launches(flags, sets):
        ps = pkg.PushStream(N_STREAMS, BATCH, channel_capacity=32)
        ps.set_audio_post(flags)
        for s, (incs, ids) in sets.items():
            ps.set_channels(s, incs, ids)
        before = pkg.launch_count()
        for b in range(N_BATCHES):
            push_batch(ps, iq, b, range(N_STREAMS))
            ps.poll()
        ps.flush()
        n = pkg.launch_count() - before
        ps.close()
        return n

    runs = 2 * N_BATCHES
    for sets, with_listeners in (({s: listeners(s) for s in range(N_STREAMS)}, runs), ({3: listeners(3)}, N_BATCHES),
                                 ({}, 0)):
        assert launches(BOTH, sets) == launches(0, sets) + 2 * runs + 2 * with_listeners
