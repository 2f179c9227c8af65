"""The fused chain kernel (chain_jobs_kernel: b200_chain_exec at R = 10) when every CTA walks many tiles, against
the float64 oracle, and chain_exec's checks on the output tensors it is given.

The kernel is persistent: it launches min(SM count, tiles) CTAs and CTA b walks tiles b, b + G, b + 2G, ... through a
four-stage TMA ring and four demod / work buffers.  Only from a CTA's fifth tile on does it refill a stage it has
used before, wait for a demod buffer to drain before reusing it, wait on the flipped parity of full[] / demod_full[]
and run a tile's audio job inside its loop rather than after it.  So each case sizes its batch from b200_sm_count()
so that every CTA walks q or q + 1 tiles (q = 9..12: walks end at every phase of the ring and the demod buffers),
with 1 tile per stream (the divisor 1 of the tile -> stream division), a power of two and primes per stream.

One oracle run checks every tile: stream s is the window X[5120 s : 5120 (s + P)] of one signal X, with the 320
samples before it as its history (stream 0 keeps the reset history, the oracle's zero state), so its dB rows and
audio are X's from frame 5 s and audio sample 128 s on.  X mixes an FM station, a full-scale station, white bytes,
silence and alternating 0 / 255 bytes in segments that are not whole tiles.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_fm import AUDIO_TOL, oracle_stream
from test_gpu_fm_rates import fm_segment, sm_count

pytestmark = pytest.mark.gpu

TILE, FRAMES, AUDIO = 5120, 5, 128          # samples, dB rows and audio samples per tile of the fused kernel
SEGMENTS = (("fm", 31_013), ("loud", 17_389), ("noise", 9_001), ("silence", 7_777), ("alt", 4_099))


def walk_streams(pkg, q, P):
    """Stream count S for P tiles per stream such that the fused grid (G = SM count CTAs) walks q or q + 1 tiles
    per CTA: floor(S P / G) = q and S P mod G != 0."""
    G = sm_count(pkg)
    S = q * G // P + 1
    total = S * P
    assert total // G == q and total % G != 0, dict(G=G, q=q, P=P, S=S, total=total, r=total % G)
    walks = {-(-(total - b) // G) for b in range(G)}          # tiles CTA b walks
    assert walks == {q, q + 1}, (G, q, P, S, walks)
    return S


def walk_signal(n):
    """n samples of IQ bytes: the SEGMENTS in turn, repeated."""
    src = {"fm": np.resize(fm_segment("fm", 1_000_003, 1), (n, 2)),
           "loud": np.resize(fm_segment("loud", 999_983, 2), (n, 2)),
           "noise": np.random.default_rng(5).integers(0, 256, size=(n, 2), dtype=np.uint8),
           "alt": np.resize(np.array([[0, 255], [255, 0]], np.uint8), (n, 2))}
    x = np.full((n, 2), 128, np.uint8)
    pos = 0
    while pos < n:
        for kind, m in SEGMENTS:
            if kind in src:
                x[pos:pos + m] = src[kind][pos:pos + m]
            pos += m
    return x


def windows(torch, x, S, start, n):
    """[S, n, 2]: row s = x[TILE s + start : TILE s + start + n] of a cuda tensor x [samples, 2]."""
    base = torch.arange(S, device=x.device)[:, None] * TILE + start
    return x[base + torch.arange(n, device=x.device)]


def walk_ring(pkg, torch, X, S, P):
    """A ring whose stream s holds the window X[TILE s : TILE (s + P)] with the samples before it as history."""
    ring = pkg.StreamRing(S, P * TILE)
    h = ring.hist
    x = torch.as_tensor(X).cuda()
    ring.batch.copy_(windows(torch, x, S, 0, P * TILE))
    ring.buf[1:, :h] = windows(torch, x, S - 1, TILE - h, h)
    return ring


@pytest.mark.parametrize("q,P,gain_db", [(9, 41, 17), (10, 1, -15), (11, 64, 30), (12, 131, 0)])
def test_chain_walk_matches_oracle(pkg, cuda, po, q, P, gain_db):
    """Every dB row and audio sample of every stream against the oracle, and tile t of stream s == tile t + 1 of
    stream s - 1 bit for bit (the same bytes, history included, reach different CTAs at different walk steps)."""
    torch = cuda
    G = sm_count(pkg)
    S = walk_streams(pkg, q, P)
    X = walk_signal((P + S - 1) * TILE)
    assert len(X) < 8_000_000
    ring = walk_ring(pkg, torch, X, S, P)
    db, audio = pkg.chain_exec(ring, gain_db=gain_db)
    torch.cuda.synchronize()
    if P >= 2:
        assert torch.equal(db[1:, :FRAMES * (P - 1)], db[:-1, FRAMES:]), (q, P, S, G)
        assert torch.equal(audio[1:, :AUDIO * (P - 1)], audio[:-1, AUDIO:]), (q, P, S, G)
    db, audio = db.cpu().numpy(), audio.cpu().numpy()

    rows = po.Spectrum(1024).rows(X)
    assert rows.shape == (FRAMES * (P + S - 1), 1024)
    frame = FRAMES * np.arange(S)[:, None] + np.arange(FRAMES * P)          # [S, 5P]: X's frame of each dB row
    with np.errstate(divide="ignore"):
        want_db = 10 * np.log10(10.0 ** int(gain_db / 10) * rows)              # C's integer gain_db / 10
    ok = (rows > 1e-6 * rows.mean(axis=1, keepdims=True))[frame]
    err = np.abs(db[ok] - want_db[frame][ok])
    assert ok.mean() > 0.5 and err.max() <= 0.01, (q, P, S, G, float(err.max()))
    silent = (rows == 0).all(axis=1)[frame]
    assert silent.any() and np.isneginf(db[silent]).all(), (q, P, S, G)

    _, want_audio = oracle_stream(po, X)
    sample = AUDIO * np.arange(S)[:, None] + np.arange(AUDIO * P)
    err = np.abs(audio - want_audio[sample])
    assert err.max() <= AUDIO_TOL, (q, P, S, G, np.unravel_index(err.argmax(), err.shape), float(err.max()))


WALK_Q, WALK_P = 9, 41


def test_chain_walk_padded_layouts(pkg, cuda):
    """Through the C ABI at walk size: IQ rows 48 bytes longer than the ring's, the padding 0xFF; audio rows the first
    n_audio floats of NaN rows n_audio + 5 long; the dB rows between two NaN guard rows.  Every padding and guard
    value stays NaN and the outputs equal the packed run bit for bit."""
    torch = cuda
    S, P, gain_db = walk_streams(pkg, WALK_Q, WALK_P), WALK_P, 17
    n, n_rows, n_audio = P * TILE, FRAMES * P, AUDIO * P
    ring = walk_ring(pkg, torch, walk_signal((P + S - 1) * TILE), S, P)
    want_db, want_audio = pkg.chain_exec(ring, gain_db=gain_db)

    row = ring.stride_bytes
    iq = torch.full((S, row + 48), 0xFF, dtype=torch.uint8, device="cuda")
    iq[:, :row] = ring.buf.reshape(S, row)
    a_full = torch.full((S, n_audio + 5), float("nan"), dtype=torch.float32, device="cuda")
    d_full = torch.full((S * n_rows + 2, 1024), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    before = pkg.launch_count()
    rc = pkg.lib().b200_chain_exec_r(C.c_void_p(iq.data_ptr() + 2 * ring.hist), row + 48, S, n, 10, gain_db,
                                     C.c_void_p(d_full[1].data_ptr()), C.c_void_p(a_full.data_ptr()), n_audio + 5,
                                     None, 6, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert rc == 0, pkg.last_error()
    assert pkg.launch_count() > before
    assert torch.isnan(a_full[:, n_audio:]).all()
    assert torch.isnan(d_full[0]).all() and torch.isnan(d_full[-1]).all()
    assert torch.equal(a_full[:, :n_audio], want_audio)
    assert torch.equal(d_full[1:-1].view(S, n_rows, 1024), want_db)


def test_chain_walk_carry(pkg, cuda):
    """At walk size, three batches joined by ring.carry() == one batch of three times the samples, bit for bit."""
    torch = cuda
    S, P, gain_db = walk_streams(pkg, WALK_Q, WALK_P), WALK_P, 30
    n = P * TILE
    x = torch.as_tensor(walk_signal((3 * P + S - 1) * TILE)).cuda()
    whole = pkg.StreamRing(S, 3 * n)
    whole.batch.copy_(windows(torch, x, S, 0, 3 * n))
    want_db, want_audio = pkg.chain_exec(whole, gain_db=gain_db)
    ring = pkg.StreamRing(S, n)
    dbs, audios = [], []
    for b in range(3):
        ring.batch.copy_(windows(torch, x, S, b * n, n))
        db, audio = pkg.chain_exec(ring, gain_db=gain_db)
        dbs.append(db)
        audios.append(audio)
        ring.carry()
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(dbs, dim=1), want_db)
    assert torch.equal(torch.cat(audios, dim=1), want_audio)


def test_chain_exec_refuses_bad_outputs(pkg, cuda):
    """db, audio and avg_u8 of the wrong dtype, shape, layout or device are refused before any launch.  Every bad
    tensor has storage for at least what the kernels would write, so a call that got through could not write past
    it (a CPU tensor is pinned, so the device can reach it)."""
    torch = cuda
    S, n = 3, 2 * TILE
    ring = pkg.StreamRing(S, n)
    rows, n_audio = n // 1024, n // 40
    f32 = dict(dtype=torch.float32, device="cuda")
    bad = {
        "db": [torch.zeros((S, rows, 1024), dtype=torch.float64, device="cuda"),
               torch.zeros((S, rows + 1, 1024), **f32),
               torch.zeros((S, 1024, rows), **f32).transpose(1, 2),
               torch.zeros((S, rows, 1024), dtype=torch.float32).pin_memory()],
        "audio": [torch.zeros((S, n_audio), dtype=torch.float64, device="cuda"),
                  torch.zeros((S, n_audio + 1), **f32),
                  torch.zeros((n_audio, S), **f32).t(),
                  torch.zeros((S, n_audio), dtype=torch.float32).pin_memory()],
        "avg_u8": [torch.zeros((S, 1024), dtype=torch.int16, device="cuda"),
                   torch.zeros((S, 2048), dtype=torch.uint8, device="cuda"),
                   torch.zeros((1024, S), dtype=torch.uint8, device="cuda").t(),
                   torch.zeros((S, 1024), dtype=torch.uint8).pin_memory()],
    }
    torch.cuda.synchronize()
    before = pkg.launch_count()
    for name, tensors in bad.items():
        for t in tensors:
            with pytest.raises(pkg.B200Error):
                pkg.chain_exec(ring, **{name: t})
    assert pkg.launch_count() == before
    # audio rows may be slices of wider rows
    a_full = torch.full((S, n_audio + 3), float("nan"), **f32)
    avg = torch.zeros((S, 1024), dtype=torch.uint8, device="cuda")
    db, audio = pkg.chain_exec(ring, db=torch.empty((S, rows, 1024), **f32), audio=a_full[:, :n_audio], avg_u8=avg)
    want_db, want_audio = pkg.chain_exec(ring)
    torch.cuda.synchronize()
    assert pkg.launch_count() > before
    assert torch.isnan(a_full[:, n_audio:]).all()
    assert torch.equal(db, want_db) and torch.equal(audio, want_audio)
