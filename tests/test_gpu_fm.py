"""GPU parity: the FM branch and the fused chain (through the C ABI) against the CPU oracle
and the golden vectors of the unmodified reference.

Tolerances (BASELINE.json north_star): CIC output bit-exact (int32); demodulated audio
within 1e-4 absolute (audio is bounded by the +-1 limiter)."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
AUDIO_TOL = 1e-4


def oracle_stream(po, iq, R=10):
    """CIC + demodulation of a whole stream in one block (state semantics are block-size independent)."""
    n = (len(iq) // (4 * R)) * 4 * R
    _, dec, _ = po.cic_decimate(R, iq[:n])
    _, _, audio, _ = po.fm_demodulate(dec)
    return dec, audio


@pytest.mark.parametrize("R", [10, 5, 12, 16, 1, 7, 64, 3, 4, 6, 8, 9, 11, 13, 14, 15, 2, 17, 103, 171, 255, 256])
def test_fm_exec_matches_oracle(pkg, cuda, po, synth, R):
    torch = cuda
    n = 4 * R * 8 * 61              # whole audio samples, multiple of 8, not a multiple of the tile
    iqs = np.stack([synth.s3_fm(n, seed=50 + s, deviation=(25e3, 75e3, 5e3)[s]) for s in range(3)])
    ring = pkg.StreamRing(3, n, R=R)
    ring.load(iqs)
    audio, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    audio, dec = audio.cpu().numpy(), dec.cpu().numpy()
    for s in range(3):
        want_dec, want_audio = oracle_stream(po, iqs[s], R)
        assert np.array_equal(dec[s], want_dec), "CIC output must be bit-exact"
        assert np.abs(audio[s] - want_audio).max() <= AUDIO_TOL


def test_fm_worst_case_bytes_and_silence(pkg, cuda, po, synth):
    torch = cuda
    n = 5120 * 7
    iqs = np.stack([synth.s1_noise(n, seed=1),                       # white bytes: every atan2 branch
                    np.full((n, 2), 128, np.uint8),                 # silence: atan2(0, 0) = 0 everywhere
                    np.full((n, 2), 255, np.uint8),                 # the |y| == |x| branch boundary
                    np.tile(np.array([[0, 255], [255, 0]], np.uint8), (n // 2, 1))])
    ring = pkg.StreamRing(4, n)
    ring.load(iqs)
    audio, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    audio, dec = audio.cpu().numpy(), dec.cpu().numpy()
    for s in range(4):
        want_dec, want_audio = oracle_stream(po, iqs[s])
        assert np.array_equal(dec[s], want_dec)
        assert np.abs(audio[s] - want_audio).max() <= AUDIO_TOL
    assert not audio[1].any()


def test_fm_state_carries_across_batches(pkg, cuda, po, synth):
    """Three consecutive batches with history carry == one long stream == the reference's
    block-by-block run with its delay structs (rf_decimator.c:28, audio_main.c:77-79)."""
    torch = cuda
    n, batches = 5120 * 4, 3
    iq = synth.s3_fm(n * batches, seed=60)
    ring = pkg.StreamRing(1, n)
    got = []
    for b in range(batches):
        ring.load(iq[None, b * n:(b + 1) * n])
        audio, _ = pkg.fm_exec(ring)
        got.append(audio.cpu().numpy()[0].copy())
        ring.carry()
    got = np.concatenate(got)
    _, want = oracle_stream(po, iq)
    assert np.abs(got - want).max() <= AUDIO_TOL
    # and reset really goes back to stream start
    ring.reset()
    ring.load(iq[None, :n])
    audio, _ = pkg.fm_exec(ring)
    assert np.abs(audio.cpu().numpy()[0] - want[:n // 40]).max() <= AUDIO_TOL


@pytest.mark.parametrize("name", ["fm_chain_25k.npz", "fm_chain_75k.npz"])
def test_fm_goldens_default_rate(pkg, cuda, synth, name):
    torch = cuda
    g = np.load(os.path.join(GOLD, name))
    iq = synth.s3_fm(int(g["n"]), deviation=float(g["deviation"]), seed=int(g["seed"]))
    assert hashlib.sha256(iq.tobytes()).hexdigest() == str(g["iq_sha"])
    n = 2 * 204800                   # the two whole 100 ms blocks the reference emitted
    ring = pkg.StreamRing(1, n)
    ring.load(iq[None, :n])
    audio, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    dec = dec.cpu().numpy()[0]
    assert hashlib.sha256(dec.tobytes()).hexdigest() == str(g["dec_sha"])
    assert np.abs(audio.cpu().numpy()[0] - g["audio"]).max() <= AUDIO_TOL


def test_fm_golden_small_custom_rate(pkg, cuda):
    g = np.load(os.path.join(GOLD, "fm_chain_small.npz"))
    n = len(g["dec"]) * 10
    ring = pkg.StreamRing(1, n)
    ring.load(g["iq"][None, :n])
    audio, dec = pkg.fm_exec(ring, decimated=True)
    assert np.array_equal(dec.cpu().numpy()[0], g["dec"])
    assert np.abs(audio.cpu().numpy()[0] - g["audio"]).max() <= AUDIO_TOL


def test_fm_argument_errors(pkg, cuda):
    ring = pkg.StreamRing(1, 5120)
    ring.n_samples = 5100                      # not a multiple of 4*R
    with pytest.raises(pkg.B200Error):
        pkg.fm_exec(ring)
    with pytest.raises(pkg.B200Error):
        pkg.StreamRing(1, 5120, R=0)


def check_chain_exec(pkg, torch, po, synth, R, K_avg, gain_db):
    """b200_chain_exec_r on 7 streams against the oracle: per-frame dB, audio and the K_avg-frame payload bytes.
    K_avg None: every frame of the batch (n / 1024, the most the argument check admits)."""
    tile = int(pkg.lib().b200_chain_tile_samples(R))
    n = tile * -(-5120 * 9 // tile)
    K_avg = n // 1024 if K_avg is None else K_avg
    n_streams = 7
    iqs = np.stack([synth.s3_fm(n, seed=70 + s, carrier=(0.0, 50e3)[s % 2]) for s in range(n_streams)])
    ring = pkg.StreamRing(n_streams, n, R=R)
    ring.load(iqs)
    avg = torch.zeros((n_streams, 1024), dtype=torch.uint8, device="cuda")
    before = pkg.launch_count()
    db, audio = pkg.chain_exec(ring, gain_db=gain_db, avg_u8=avg, K_avg=K_avg)
    torch.cuda.synchronize()
    assert pkg.launch_count() > before
    db, audio, avg = db.cpu().numpy(), audio.cpu().numpy(), avg.cpu().numpy()
    gain = 10.0 ** int(gain_db / 10)
    for s in range(n_streams):
        rows = po.Spectrum(1024).rows(iqs[s])
        with np.errstate(divide="ignore"):
            want_db = 10 * np.log10(gain * rows)
        ok = rows > 1e-6 * rows.mean(axis=1, keepdims=True)
        assert np.abs(db[s][ok] - want_db[ok]).max() <= 0.01
        _, want_audio = oracle_stream(po, iqs[s], R)
        assert np.abs(audio[s] - want_audio).max() <= AUDIO_TOL
        rows_k = po.Spectrum(1024).rows(iqs[s], K=K_avg)[0]
        want_u8, dbf = po.db_payload(rows_k, K_avg, gain_db)
        diff = avg[s] != want_u8
        assert diff.mean() < 0.01 and (np.abs(dbf[diff] - np.rint(dbf[diff])) <= 0.01).all()


def test_chain_exec_matches_oracle(pkg, cuda, po, synth):
    check_chain_exec(pkg, cuda, po, synth, R=10, K_avg=6, gain_db=20)


@pytest.mark.parametrize("R,K_avg,gain_db", [(R, K, g) for R in (10, 1, 7, 100, 256)
                                             for K, g in ((6, 20), (1, -15), (None, 20)) if (R, K, g) != (10, 6, 20)])
def test_chain_exec_r_matches_oracle(pkg, cuda, po, synth, R, K_avg, gain_db):
    """The fused kernel at R = 10, spectrum + b200_fm_exec otherwise; one frame and every frame per payload row;
    gain_db = -15 scales by 10^-1, C's integer division (cbb_main.c:112)."""
    check_chain_exec(pkg, cuda, po, synth, R, K_avg, gain_db)


def test_chain_full_size_properties(pkg, cuda):
    """BASELINE config 3/5 scale through properties: 64 streams x 4 Mi samples.
    (a) streams are independent: stream s of the batch == the same bytes run alone;
    (b) time-shift covariance of the FM branch: a stream delayed by one tile (5120 samples)
        produces the same audio delayed by 128 samples;
    (c) silence in -> silence out, bit for bit."""
    torch = cuda
    n_streams, n = 64, 5120 * 800
    g = torch.Generator(device="cuda").manual_seed(3)
    ring = pkg.StreamRing(n_streams, n)
    ring.batch.copy_(torch.randint(0, 256, (n_streams, n, 2), dtype=torch.uint8, device="cuda", generator=g))
    ring.batch[1, 5120:] = ring.batch[0, :n - 5120]
    ring.batch[1, :5120] = 128
    ring.batch[2] = 128
    db, audio = pkg.chain_exec(ring)
    torch.cuda.synchronize()
    assert torch.equal(audio[1, 128:], audio[0, :n // 40 - 128])
    assert torch.equal(db[1, 5:], db[0, :n // 1024 - 5])
    assert not audio[2].any() and torch.isneginf(db[2]).all()
    solo = pkg.StreamRing(1, n)
    solo.batch.copy_(ring.batch[37:38])
    db1, audio1 = pkg.chain_exec(solo)
    assert torch.equal(db1[0], db[37]) and torch.equal(audio1[0], audio[37])
    # |audio| <= (sum |h|)^2 of the two half-bands on a +-1 limited input
    assert audio.abs().max().item() <= 1.46404 ** 2 + 1e-6


def test_fm_full_size_properties(pkg, cuda):
    """BASELINE config 3 at its full size (2^30 samples of FM chain, R = 10) through properties:
    (a) the CIC output is exact integer arithmetic: per stream, sum over decimated samples == sum over all bytes
        - 128 per sample (int64 on the device);
    (b) the standalone FM kernel and the fused chain kernel produce the same audio from the same bytes;
    (c) |audio| is bounded by the limiter and the two half-bands."""
    torch = cuda
    n_streams, n = 256, 5120 * 820                     # 256 x 4 198 400 = 1.07e9 samples
    assert n_streams * n >= 1 << 30
    g = torch.Generator(device="cuda").manual_seed(11)
    ring = pkg.StreamRing(n_streams, n)
    ring.batch.copy_(torch.randint(0, 256, (n_streams, n, 2), dtype=torch.uint8, device="cuda", generator=g))
    audio, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    want = torch.empty((n_streams, 2), dtype=torch.int64, device="cuda")
    for s0 in range(0, n_streams, 32):
        want[s0:s0 + 32] = ring.batch[s0:s0 + 32].to(torch.int32).sum(dim=1, dtype=torch.int64) - 128 * n
    assert torch.equal(dec.sum(dim=1, dtype=torch.int64), want)
    del dec
    db = torch.empty((n_streams, n // 1024, 1024), dtype=torch.float32, device="cuda")
    _, audio2 = pkg.chain_exec(ring, db=db)
    torch.cuda.synchronize()
    assert (audio - audio2).abs().max().item() <= 1e-6
    assert audio.abs().max().item() <= 1.46404 ** 2 + 1e-6


@pytest.mark.parametrize("n_streams,n_tiles", [(1, 1), (1, 2), (1, 3), (1, 4), (1, 5), (2, 7), (3, 13), (1, 31), (5, 1)])
def test_chain_pipeline_edges(pkg, cuda, po, synth, n_streams, n_tiles):
    """Few tiles per CTA / per group: ring prologue shorter than its depth, groups with no work,
    the last tile's audio job after the loop, history at the very start of every stream."""
    torch = cuda
    n = 5120 * n_tiles
    iqs = np.stack([synth.s1_noise(n, seed=400 + s) if s % 2 else synth.s3_fm(n, seed=400 + s)
                    for s in range(n_streams)])
    ring = pkg.StreamRing(n_streams, n)
    ring.load(iqs)
    db, audio = pkg.chain_exec(ring)
    audio_only, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    db, audio, audio_only, dec = db.cpu().numpy(), audio.cpu().numpy(), audio_only.cpu().numpy(), dec.cpu().numpy()
    for s in range(n_streams):
        want_dec, want_audio = oracle_stream(po, iqs[s])
        assert np.array_equal(dec[s], want_dec)
        assert np.abs(audio[s] - want_audio).max() <= AUDIO_TOL
        assert np.abs(audio_only[s] - want_audio).max() <= AUDIO_TOL
        rows = po.Spectrum(1024).rows(iqs[s])
        ok = rows > 1e-6 * rows.mean(axis=1, keepdims=True)
        assert np.abs(db[s][ok] - 10 * np.log10(rows[ok])).max() <= 0.01


def test_fm_tile_boundaries_r10(pkg, cuda, po, synth):
    """Audio lengths around the 62-sample tile of the R = 10 kernel (n_samples only has to be a
    multiple of 40): whole tiles, one short tile, a single audio sample."""
    torch = cuda
    for n_audio in (1, 2, 61, 62, 63, 124, 125, 1000):
        n = 40 * n_audio
        if n % 8:
            n_audio += 1          # n_samples must also be a multiple of 8
            n = 40 * n_audio
        iq = synth.s3_fm(n, seed=n_audio)
        ring = pkg.StreamRing(1, n)
        ring.load(iq[None])
        audio, dec = pkg.fm_exec(ring, decimated=True)
        torch.cuda.synchronize()
        want_dec, want_audio = oracle_stream(po, iq)
        assert np.array_equal(dec.cpu().numpy()[0], want_dec)
        assert np.abs(audio.cpu().numpy()[0] - want_audio).max() <= AUDIO_TOL
