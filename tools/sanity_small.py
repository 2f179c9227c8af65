"""Tiny run of every kernel (for compute-sanitizer): small shapes, no timing."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as g

pkg = g.load_package()
pkg.init(0)
n = 5120 * 3
iq = np.stack([pkg.synth.s3_fm(n, seed=s) for s in range(3)])
ring = pkg.StreamRing(3, n)
ring.load(iq)
db, audio = pkg.chain_exec(ring)
a2, dec = pkg.fm_exec(ring, decimated=True)
ring.carry()
for N, K, hop, win in ((1024, 1, None, 0), (1024, 6, None, 0), (1024, 2, 512, 1), (2048, 1, None, 0), (4096, 2, None, 1),
                       (8192, 1, None, 0), (512, 1, None, 0)):
    pkg.SpectrumPlan(N, hop=hop, K=K, window=win).exec(ring.batch, db=True, power=True, db_u8=True)
big = pkg.StreamRing(1, 65536 * 2)
big.load(pkg.synth.s2_tones(65536 * 2, N=65536)[None])
pkg.SpectrumPlan(65536, hop=32768, window=1).exec(big.batch, db=True)
pkg.SpectrumPlan(65536, K=2).exec(big.batch, power=True)
# round 2: the four-step kernel at 16 / 32 branches, the cs32 demodulator, the audio extensions
pkg.SpectrumPlan(16384, hop=8192, window=1).exec(big.batch, db=True, power=True, db_u8=True)
pkg.SpectrumPlan(32768, K=2).exec(big.batch, db=True)
dm = pkg.FmDemod()
dm.block(dec[0][:4096].cpu().numpy(), want_demod=True)
dm.block(dec[0][4096:8192].cpu().numpy(), want_audio=False)
dm.close()
st = torch.zeros((3, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
pkg.audio_post(audio[:, :368], st, pkg.AUDIO_DEEMPH_50US | pkg.AUDIO_RESAMPLE_48K)
r7 = pkg.StreamRing(2, 4 * 7 * 8 * 9, R=7)
r7.load(np.stack([pkg.synth.s1_noise(4 * 7 * 8 * 9, seed=s) for s in range(2)]))
pkg.fm_exec(r7, decimated=True)
# FM channels at offsets: the R = 10 kernel and the general one (R = 7)
inc = torch.tensor([[0, pkg.fm_channel_tune(200e3, 2.048e6), pkg.fm_channel_tune(-1.024e6, 2.048e6) - 2**32]] * 3,
                   dtype=torch.int32, device="cuda")
pkg.fm_channels_exec(ring, inc, 0, baseband=True)
pkg.fm_channels_exec(r7, inc[:2, :2].contiguous(), 4 * 7 * 10, baseband=True)
# the runs-table form (boxcar and FIR) and channels on the push stream
pkg.fm_channels_exec_runs(ring, [(0, 0, [1, 2, 3]), (2, 40 * 9, [5])])
fr = pkg.StreamRing(2, 5120, history=pkg.fm_channels_fir_history_samples(10, 40))
pkg.fm_channels_exec_runs(fr, [(1, 0, [7, 8])], taps=torch.ones(40, dtype=torch.float32, device="cuda"))
sess = pkg.Session(3, n)
hdb = np.empty((3, n // 1024, 1024), np.float32)
hau = np.empty((3, n // 40), np.float32)
sess.chain(np.ascontiguousarray(iq), n, hdb, hau)
ps = pkg.PushStream(2, 5120 * 2, channel_capacity=2)
ps.set_channels(1, [0, pkg.fm_channel_tune(200e3, 2.048e6)], [4, 5])
for s in range(2):
    ps.push(s, iq[s])
ps.flush()
# audio post-processing over a row table, and on the push stream's centre and channel audio
pkg.audio_post_rows(audio[:, :368], [(2, 0, 1, 0), (0, 1, 0, 1)], st, pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K)
pp = pkg.PushStream(2, 5120 * 2, channel_capacity=2)
pp.set_audio_post(pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K)
pp.set_channels(0, [pkg.fm_channel_tune(-200e3, 2.048e6)], [9])
for s in range(2):
    pp.push(s, iq[s])
pp.flush()
torch.cuda.synchronize()
print("sanity ok", float(db.abs().max()) > 0, float(audio.abs().max()) >= 0)
