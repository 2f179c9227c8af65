"""GPU parity: the demodulator behind the reference's own callback signature (b200_fm_exec_cs32,
b200_fm_demod_block, libb200audio.so = audio_main.h) and the opt-in audio extensions (de-emphasis,
15/16 resampler), all through the C ABI against the CPU oracle / the unmodified reference."""
import os

import numpy as np
import pytest

from oracle import pyoracle as _po

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _decimated(po, synth, n_iq, seed, R=10):
    iq = synth.s3_fm(n_iq, seed=seed)
    _, dec, _ = po.cic_decimate(R, iq)
    return dec


# ---- atan2_approx on the device, all three forms, against the reference's own grid ------------------------

@pytest.mark.parametrize("which", [0, 1, 2])
def test_atan2_forms_on_the_reference_grid(pkg, cuda, which):
    """tests/golden/atan2.npz was made by the unmodified common_sp.h:40-76: the integer grid the CIC output
    lives on, both diagonals (the 0.0083 rad branch discontinuity at |y| == |x|) and both axes."""
    g = np.load(os.path.join(GOLD, "atan2.npz"))
    ys, xs = np.meshgrid(g["ys"], g["xs"], indexing="ij")
    got = pkg.debug_atan2(ys, xs, which)
    assert np.abs(got - g["grid"]).max() <= 1e-6           # north_star: 1e-4 on audio; this is the phase itself
    d = g["diag"]
    z = np.zeros_like(d)
    for name, y, x in (("diag_pp", d, d), ("diag_pm", d, -d), ("axis_y0", z, d), ("axis_x0", d, z)):
        assert np.abs(pkg.debug_atan2(y, x, which) - g[name]).max() <= 1e-6, name
    assert float(pkg.debug_atan2([0], [0], which)[0]) == 0.0                       # common_sp.h:52-53
    assert abs(float(pkg.debug_atan2([5], [5], which)[0]) - (np.pi / 2 - 1 / 1.28)) < 1e-6
    assert abs(float(pkg.debug_atan2([-5], [-5], which)[0]) - (np.pi / 2 - 1 / 1.28 - np.pi)) < 1e-6


# ---- b200_fm_exec_cs32 ----------------------------------------------------------------------------------

def test_fm_exec_cs32_matches_oracle_with_state_carry(pkg, cuda, po, synth):
    torch = cuda
    n_streams = 3
    # every block leaves >= 10 first-stage outputs: below that resample.c:66 reads in front of its input buffer
    # (undefined in the reference and in its port); shorter blocks are covered by the chunking test below
    blocks = [20480, 40, 1024 + 8, 20480, 44, 4096]
    decs = [_decimated(po, synth, 10 * sum(blocks), seed=300 + s) for s in range(n_streams)]
    state = torch.zeros((n_streams, pkg.FM_STATE_FLOATS), dtype=torch.float32, device="cuda")
    sts = [po.FmState() for _ in range(n_streams)]
    pos = 0
    for n in blocks:
        d = torch.as_tensor(np.stack([x[pos:pos + n] for x in decs])).cuda()
        out = pkg.fm_exec_cs32(d, state, demod=True, phase=True)
        torch.cuda.synchronize()
        for s in range(n_streams):
            demod, _, audio, sts[s] = po.fm_demodulate(decs[s][pos:pos + n], sts[s])
            assert np.abs(out["demod"][s].cpu().numpy() - demod).max() <= 2e-6
            assert np.abs(out["audio"][s].cpu().numpy() - audio).max() <= 1e-5      # contract: 1e-4
            ph = po.atan2_approx(decs[s][pos:pos + n, 1].astype(np.float32), decs[s][pos:pos + n, 0].astype(np.float32))
            assert np.abs(out["phase"][s].cpu().numpy() - ph).max() <= 1e-6
        pos += n
    # the carried state is the reference's three statics (audio_main.c:77-79)
    st = state.cpu().numpy()
    for s in range(n_streams):
        assert abs(st[s, 0] - sts[s].prev_sample) <= 1e-6
        assert np.abs(st[s, 1:11] - np.array(sts[s].delay_line_1[:])).max() <= 2e-6
        assert np.abs(st[s, 11:21] - np.array(sts[s].delay_line_2[:])).max() <= 1e-5


def test_fm_exec_cs32_does_not_depend_on_chunking(pkg, cuda, po, synth):
    """Blocks of any multiple of 4 -- also shorter than the delay lines, where the reference itself reads out of
    bounds (resample.c:66) -- continue the stream exactly: same audio as one long block, bit for bit."""
    torch = cuda
    dec = _decimated(po, synth, 10 * 4096, seed=41)
    d_all = torch.as_tensor(dec[None]).cuda()
    state = torch.zeros((1, pkg.FM_STATE_FLOATS), dtype=torch.float32, device="cuda")
    whole = pkg.fm_exec_cs32(d_all, state)["audio"][0].cpu().numpy()
    state.zero_()
    parts, pos = [], 0
    for n in [4, 8, 4, 12, 1024, 4, 2048 - 32, 20, 4, 4, 4096 - 2048 - 1024 - 28]:
        parts.append(pkg.fm_exec_cs32(d_all[:, pos:pos + n].contiguous(), state)["audio"][0].cpu().numpy())
        pos += n
    assert pos == 4096
    assert np.array_equal(np.concatenate(parts), whole)
    _, _, want, _ = po.fm_demodulate(dec)
    assert np.abs(whole - want).max() <= 1e-5


def test_fm_exec_cs32_large_inputs_and_argument_errors(pkg, cuda, po):
    torch = cuda
    rng = np.random.default_rng(5)
    sig = rng.integers(-2**31, 2**31 - 1, size=(1, 4096, 2), dtype=np.int64).astype(np.int32)     # any int32, not CIC sums
    sig[0, :64] = 0
    state = torch.zeros((1, pkg.FM_STATE_FLOATS), dtype=torch.float32, device="cuda")
    out = pkg.fm_exec_cs32(torch.as_tensor(sig).cuda(), state, demod=True)
    demod, _, audio, _ = po.fm_demodulate(sig[0])
    assert np.abs(out["demod"][0].cpu().numpy() - demod).max() <= 2e-6
    assert np.abs(out["audio"][0].cpu().numpy() - audio).max() <= 1e-5
    with pytest.raises(pkg.B200Error):
        pkg.fm_exec_cs32(torch.zeros((1, 6, 2), dtype=torch.int32, device="cuda"), state)        # not a multiple of 4


def test_fm_exec_cs32_dropped_block_keeps_second_delay_line(pkg, cuda, po, synth):
    """audio_main.c:137-143: with the pool full the block is dropped AFTER the discriminator and the first
    half-band ran, and delay_line_2 does not advance."""
    torch = cuda
    dec = _decimated(po, synth, 10 * 3 * 2048, seed=9)
    state = torch.zeros((1, pkg.FM_STATE_FLOATS), dtype=torch.float32, device="cuda")
    st = po.FmState()
    audios = []
    for b in range(3):
        blk = dec[2048 * b:2048 * (b + 1)]
        d = torch.as_tensor(blk[None]).cuda()
        if b == 1:
            pkg.fm_exec_cs32(d, state, flags=pkg.FM_SKIP_STAGE2)
            keep = np.array(st.delay_line_2[:], dtype=np.float32)
            _, _, _, st = po.fm_demodulate(blk, st)
            st.delay_line_2[:] = list(keep)
        else:
            out = pkg.fm_exec_cs32(d, state)
            _, _, audio, st = po.fm_demodulate(blk, st)
            audios.append((out["audio"][0].cpu().numpy(), audio))
    for got, want in audios:
        assert np.abs(got - want).max() <= 1e-5


def test_fm_demod_host_blocks_and_golden(pkg, cuda, po):
    g = np.load(os.path.join(GOLD, "fm_demod_block.npz"))        # the unmodified audio_fm_demodulator on one block
    d = pkg.FmDemod()
    audio, demod = d.block(g["signal"], want_demod=True)
    assert np.abs(demod - g["demod"]).max() <= 2e-6
    assert np.abs(audio - g["audio"]).max() <= 1e-5
    # a second block continues the stream; reset goes back to its start
    a2, _ = d.block(g["signal"])
    _, _, want1, st = po.fm_demodulate(g["signal"])
    _, _, want2, _ = po.fm_demodulate(g["signal"], st)
    assert np.abs(a2 - want2).max() <= 1e-5
    d.reset()
    a3, _ = d.block(g["signal"])
    assert np.abs(a3 - want1).max() <= 1e-5
    d.close()


# ---- libb200audio.so: audio_main.h over the GPU demodulator -------------------------------------------------

def test_audio_compat_pool_and_reference_drain_order(pkg, cuda, po, synth):
    """audio_init / audio_fm_demodulator / audio_get_audio_payload: the pool of 50 buffers, the drop when it is
    full, and the drain order of audio_main.c:40-72 (b200_wire_reference_drain_index models the same thing)."""
    A = pkg.audio
    L = A.lib()
    L.audio_init()
    L.b200_audio_reset_stream()
    n_blocks, blk = 6, 20480
    dec = _decimated(po, synth, 10 * n_blocks * blk, seed=21)
    st = po.FmState()
    want = []
    for b in range(n_blocks):
        A.demodulate(dec[blk * b:blk * (b + 1)])
        _, _, audio, st = po.fm_demodulate(dec[blk * b:blk * (b + 1)], st)
        want.append(audio)
    want = np.concatenate(want)
    assert L.audio_new_audio_available() == 1 and L.b200_audio_buffer_len() == blk // 4
    # main.c:96: 2048-byte reads until nothing is left
    got = []
    for _ in range(4 * n_blocks * (blk // 4) // 512):
        chunk = A.get_payload(2048)
        if len(chunk) == 0:
            break
        got.append(chunk)
    got = np.concatenate(got)
    idx = np.array([pkg.lib().b200_wire_reference_drain_index(w, blk // 4) for w in range(len(got))])
    # after the last buffer one more call re-reads its first 512 samples (it is still the list head, audio_main.c:49-56)
    assert len(got) == n_blocks * (blk // 4) + 512
    assert np.abs(got - want[idx]).max() <= 1e-5
    # pool exhaustion: 50 buffers, then blocks are dropped and counted
    L.b200_audio_reset_stream()
    for b in range(52):
        A.demodulate(dec[:blk])
    assert L.b200_audio_dropped_blocks() == 2
    n = 0
    while A.take_buffer() is not None:
        n += 1
    assert n == 50
    L.audio_close()


@pytest.mark.skipif(not _po.have_dropin_audio(), reason="oracle/_ref/libdropin_audio_rtlws.so not built")
def test_unmodified_driver_with_gpu_demodulator(pkg, cuda, po, synth):
    """The reference's unmodified cbb_main.c + signal_source.c with audio_main.o replaced by libb200audio.so:
    main.c:205's registration puts atan2, limiter and both half-bands on the GPU (row f2)."""
    g = np.load(os.path.join(GOLD, "cbb_gain17.npz"))
    iq = synth.s2_tones(int(g["n"]), N=1024, seed=int(g["seed"]))
    before = pkg.launch_count()
    out = po.DropInAudio().cbb_run(iq, gain_db=17)
    assert pkg.launch_count() - before >= 18 + 5 + 2 * 5          # spectra, decimator blocks, demodulator (2 launches per block)
    dec_want, audio_want = po.chain_run(iq)
    assert np.array_equal(out["decimated"], dec_want)
    assert out["audio"].shape == audio_want.shape
    assert np.abs(out["audio"] - audio_want).max() <= 1e-5
    assert np.abs(out["audio"][:2048] - g["audio_head"]).max() <= 1e-5


@pytest.mark.skipif(not (_po.have_dropin_audio() and _po.have_ref()), reason="oracle/_ref not built")
def test_unmodified_main_c_with_gpu_demodulator_on_the_wire(pkg, cuda, po, synth):
    """main.c's websocket callback, unmodified, draining libb200audio.so: the socket sees what it sees with
    the reference's own audio_main.c underneath (message order, fragment sizes, audio within 1e-4)."""
    iq = synth.s3_fm(131072 * 7, seed=81)
    cmds = ("spectrumgain 17", "freq 99900", "start")
    want = po.Ref().ws_run(iq, commands=cmds)
    got = po.DropInAudio().ws_run(iq, commands=cmds)
    assert [(m, len(b)) for m, b in got] == [(m, len(b)) for m, b in want]
    n_audio = 0
    for (m, a), (_, b) in zip(got, want):
        if b.startswith(b"t s;"):
            continue
        skip = 8 if a.startswith(b"FF;t a;d") else 0
        assert a[:skip] == b[:skip]
        assert np.abs(np.frombuffer(a[skip:], dtype="<f4") - np.frombuffer(b[skip:], dtype="<f4")).max() <= 1e-4
        n_audio += 1
    assert n_audio > 0


# ---- opt-in extensions: de-emphasis and the 15/16 resampler ---------------------------------------------------

@pytest.mark.parametrize("flags_name,rate", [pytest.param(f, 51200.0, id=f) for f in
                                               ("AUDIO_DEEMPH_50US", "AUDIO_DEEMPH_75US", "AUDIO_RESAMPLE_48K", "both")] +
                         [pytest.param(f, r, id=f"{f}-{r:.0f}") for r in (128000.0, 512000.0, 800000.0)
                          for f in ("AUDIO_DEEMPH_50US", "AUDIO_DEEMPH_75US", "both")])
def test_audio_post_matches_definition_across_batches(pkg, cuda, po, flags_name, rate):
    """rate: the audio rate fs / (4R) the de-emphasis is designed for (51.2 kHz at the reference's R = 10)."""
    torch = cuda
    flags = pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K if flags_name == "both" else getattr(pkg, flags_name)
    rng = np.random.default_rng(11)
    n_streams = 3
    batches = [5120, 16, 2048 + 16, 5120, 128]
    x = rng.uniform(-1, 1, size=(n_streams, sum(batches))).astype(np.float32)
    state = torch.zeros((n_streams, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    y_state = [np.zeros(1, np.float32) for _ in range(n_streams)]
    hist = [np.zeros(15, np.float32) for _ in range(n_streams)]
    tau = 50e-6 if flags & pkg.AUDIO_DEEMPH_50US else 75e-6
    pos = 0
    for n in batches:
        got = pkg.audio_post(torch.as_tensor(x[:, pos:pos + n]).cuda().contiguous(), state, flags, rate).cpu().numpy()
        for s in range(n_streams):
            want = x[s, pos:pos + n]
            if flags & (pkg.AUDIO_DEEMPH_50US | pkg.AUDIO_DEEMPH_75US):
                want, y_state[s] = po.deemphasis(want, rate, tau, y_state[s])
            if flags & pkg.AUDIO_RESAMPLE_48K:
                want, hist[s] = po.resample_15_16(want, hist[s])
            assert got[s].shape == want.shape
            assert np.abs(got[s] - want).max() <= 2e-6
        pos += n


def test_audio_post_resampler_is_a_resampler(pkg, cuda):
    """A 1 kHz tone at 51.2 kHz comes out as a 1 kHz tone at 48 kHz (unity gain, fixed delay of 7.97 input samples)."""
    torch = cuda
    n = 51200
    t = np.arange(n) / 51200.0
    x = np.sin(2 * np.pi * 1000.0 * t).astype(np.float32)
    state = torch.zeros((1, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    y = pkg.audio_post(torch.as_tensor(x[None]).cuda(), state, pkg.AUDIO_RESAMPLE_48K).cpu().numpy()[0]
    assert len(y) == 48000
    delay = (239 / 2) / 15 / 51200.0
    want = np.sin(2 * np.pi * 1000.0 * (np.arange(48000) / 48000.0 - delay))
    assert np.abs(y[100:] - want[100:]).max() < 2e-3
    with pytest.raises(pkg.B200Error):
        pkg.audio_post(torch.zeros((1, 24), dtype=torch.float32, device="cuda"), state, pkg.AUDIO_RESAMPLE_48K)


# ---- multi-GPU gather through the C ABI ------------------------------------------------------------------------

def test_comm_gather_single_rank_and_sharding_helpers(pkg, cuda):
    torch = cuda
    assert [pkg.shard_count(10, 4, r) for r in range(4)] == [3, 3, 2, 2]
    assert [pkg.shard_stream(10, 4, 1, i) for i in range(3)] == [1, 5, 9]
    assert pkg.lib().b200_comm_nccl_version() > 20000
    comm = pkg.Comm(pkg.Comm.unique_id(), 1, 0)
    assert pkg.lib().b200_comm_world(comm.h) == 1 and pkg.lib().b200_comm_rank(comm.h) == 0
    assert pkg.lib().b200_comm_world(None) < 0 and pkg.lib().b200_shard_count(10, 4, 4) < 0 and pkg.lib().b200_shard_stream(10, 4, 1, 3) < 0
    send = torch.randint(0, 256, (7, 1024), dtype=torch.uint8, device="cuda")
    recv = torch.zeros_like(send)
    comm.gather_rows(send, 7, recv)
    torch.cuda.synchronize()
    assert torch.equal(send, recv)
    comm.close()


def test_comm_gather_all_devices_of_one_process(pkg, cuda):
    """b200_comm_create_all + b200_comm_gather_rows_all: one host thread, G devices (skipped on a 1-GPU box)."""
    import ctypes as C
    torch = cuda
    G = torch.cuda.device_count()
    if G < 2:
        pytest.skip("needs at least two GPUs")
    G = min(G, 4)
    L = pkg.lib()
    comms = (C.c_void_p * G)()
    assert L.b200_comm_create_all(G, comms) == 0, pkg.binding.last_error()
    n_total, row = 37, 1024
    rows = torch.randint(0, 256, (n_total, row), dtype=torch.uint8)
    sends = [rows[r::G].contiguous().to(f"cuda:{r}") for r in range(G)]
    recv = torch.zeros((n_total, row), dtype=torch.uint8, device="cuda:0")
    ptrs = (C.c_void_p * G)(*[s.data_ptr() for s in sends])
    assert L.b200_comm_gather_rows_all(comms, G, ptrs, n_total, row, C.c_void_p(recv.data_ptr()), 0, None) == 0, \
        pkg.binding.last_error()
    for r in range(G):
        torch.cuda.synchronize(r)
    assert torch.equal(recv.cpu(), rows)
    for r in range(G):
        L.b200_comm_destroy(comms[r])
    torch.cuda.set_device(0)


@pytest.mark.parametrize("n_gpus", [1, 2, 8])
def test_multi_host_buffers_sharded_over_the_devices_of_one_process(pkg, cuda, po, synth, n_gpus):
    """b200_multi_chain: global host arrays in, stream s on device s mod G, payload rows gathered on device 0
    (NCCL when G > 1) -- against the single-GPU device-resident path on the same bytes."""
    torch = cuda
    if torch.cuda.device_count() < n_gpus:
        pytest.skip(f"needs {n_gpus} GPUs")
    n_streams, n = 11, 5120 * 3
    iq = np.stack([synth.s3_fm(n, seed=700 + s) for s in range(n_streams)])
    m = pkg.Multi(n_gpus, n_streams, n, gain_db=20, K_avg=6)
    for batch in range(2):                       # the second batch continues every stream (history carried per device)
        db, audio, avg = m.chain(iq, n)
        if batch == 0:
            ring = pkg.StreamRing(n_streams, n)
        ring.load(iq)
        avg_want = torch.zeros((n_streams, 1024), dtype=torch.uint8, device="cuda")
        db_want, audio_want = pkg.chain_exec(ring, gain_db=20, avg_u8=avg_want, K_avg=6)
        ring.carry()
        torch.cuda.synchronize()
        assert np.array_equal(db, db_want.cpu().numpy())
        assert np.array_equal(audio, audio_want.cpu().numpy())
        assert np.array_equal(avg, avg_want.cpu().numpy())
    m.close()
    torch.cuda.set_device(0)
