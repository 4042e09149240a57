"""TEST INFRASTRUCTURE ONLY: the wavelet oracle (oracle/wavelet.py) for the other banks of the reference's pad table
(triplane_encoder.py:174-180): haar, bior2.2, bior2.6, bior4.4.  Importing this module adds them to `oracle.wavelet.WAVELETS`
(new keys only; bior6.8 stays as it is), so every oracle function that takes `wave` accepts them.  `train_step` is
oracle/pipeline.train_step with the wavelet as an argument.

Filter banks in PyWavelets order, as oracle/wavelet.py lists bior6.8: rec_lo centred at L/2 - 1, dec_lo at L/2 with one
leading zero (the same residual assumption as there: PyWavelets cannot be run here).  bior2.2 / bior2.6 are the spline CDF
pairs in closed form, bior4.4 is CDF 9/7.  Every bank has 4*pad == L - 2, so a padded level maps n -> 2n for all of them;
tests/test_wavelet_banks.py anchors the constants."""
from oracle import pipeline
from oracle import wavelet as W


def _bank(dec_lo, rec_lo, pad):
    """PyWavelets' quadrature-mirror relations: rec_hi[k] = (-1)^k dec_lo[k], dec_hi[k] = (-1)^(k+1) rec_lo[k]
    (the bior6.8 constants of oracle/wavelet.py satisfy both)."""
    return dict(rec_lo=list(rec_lo), rec_hi=[(-1) ** k * v for k, v in enumerate(dec_lo)], dec_lo=list(dec_lo),
                dec_hi=[(-1) ** (k + 1) * v for k, v in enumerate(rec_lo)], pad=pad)


_S = 0.3535533905932738   # sqrt(2) / 4
HAAR_LO = [0.7071067811865476, 0.7071067811865476]
BIOR22_DEC_LO = [0.0, -0.1767766952966369, 0.3535533905932738, 1.0606601717798214, 0.3535533905932738, -0.1767766952966369]
BIOR22_REC_LO = [0.0, _S, 0.7071067811865476, _S, 0.0, 0.0]
BIOR26_DEC_LO = [0.0, -0.006905339660024878, 0.013810679320049757, 0.046956309688169176, -0.10772329869638811,
                 -0.16987135563661201, 0.4474660099696121, 0.966747552403483, 0.4474660099696121, -0.16987135563661201,
                 -0.10772329869638811, 0.046956309688169176, 0.013810679320049757, -0.006905339660024878]
BIOR26_REC_LO = [0.0] * 5 + [_S, 0.7071067811865476, _S] + [0.0] * 6
BIOR44_DEC_LO = [0.0, 0.03782845550726404, -0.023849465019556843, -0.11062440441843718, 0.37740285561283066,
                 0.8526986790088938, 0.37740285561283066, -0.11062440441843718, -0.023849465019556843, 0.03782845550726404]
BIOR44_REC_LO = [0.0, -0.06453888262869706, -0.04068941760916406, 0.41809227322161724, 0.7884856164055829,
                 0.41809227322161724, -0.04068941760916406, -0.06453888262869706, 0.0, 0.0]

BANKS = {   # pad: triplane_encoder.py:174-180
    "bior2.6": _bank(BIOR26_DEC_LO, BIOR26_REC_LO, 3),
    "bior4.4": _bank(BIOR44_DEC_LO, BIOR44_REC_LO, 2),
    "bior2.2": _bank(BIOR22_DEC_LO, BIOR22_REC_LO, 1),
    "haar": _bank(HAAR_LO, HAAR_LO, 0),
}
for _name, _b in BANKS.items():
    W.WAVELETS.setdefault(_name, _b)


def train_step(pf, coefs, weights, rays_o, rays_d, target, bitfield, noises, wave, lam=0.2, loss_scale=1.0, **kw):
    """oracle/pipeline.train_step with the planes reconstructed by wavelet `wave` -> (loss, M)"""
    planes = W.build_planes(pf, coefs, wave)
    image, ws, depth, M = pipeline.render_train(planes, weights, rays_o, rays_d, bitfield, noises, **kw)
    loss = ((image - target) ** 2).mean(-1).mean() + pipeline.wavelet_regulariser(coefs, lam)
    (loss * loss_scale).backward()
    return float(loss.detach()), M
