"""CPU: known-answer anchors of the wavelet banks of the reference's pad table that tests/wavelet_oracle.py adds to the
oracle: haar, bior2.2, bior2.6, bior4.4, next to bior6.8 (tests/test_oracle_wavelet.py pins that one).  PyWavelets cannot
be run here, so these properties are what anchors the constants: length and padding, zero placement, symmetry, sums, the vanishing
moments their names promise, perfect reconstruction, the n -> 2n level contract, the DC gain, and the embedding into the
18-tap frame the IDWT kernels use for every wavelet."""
import numpy as np
import pytest
import torch

from oracle import wavelet as W
from tests import wavelet_oracle  # noqa: F401  (adds the four banks to W.WAVELETS)

NEW = ["haar", "bior2.2", "bior2.6", "bior4.4"]
# (length, pad, vanishing moments of rec_hi, of dec_hi): bior Nr.Nd -> rec_hi Nd, dec_hi Nr
SPEC = {"haar": (2, 0, 1, 1), "bior2.2": (6, 1, 2, 2), "bior2.6": (14, 3, 6, 2), "bior4.4": (10, 2, 4, 4), "bior6.8": (18, 4, 8, 6)}


def embed18(taps):
    """a bank of length L placed in the 18-tap frame of bior6.8: G[k + 9 - L/2] = g[k], zeros elsewhere (the IDWT kernels' taps,
    trinerflet_b200/csrc/idwt_core.cuh)"""
    off = 9 - len(taps) // 2
    return [0.0] * off + list(taps) + [0.0] * (18 - off - len(taps))


def _support(f):
    nz = np.flatnonzero(f)
    return nz[0], nz[-1]


def _moments(f):
    """number of vanishing moments of filter f: the first p whose moment sum k^p f[k] is not zero (relative to the taps)"""
    f = np.asarray(f, np.float64)
    k = np.arange(f.size) - (f.size - 1) / 2
    scale = np.abs(f).sum()
    c = max(np.abs(k).max(), 1.0)
    for p in range(20):
        if abs((k ** p * f).sum()) > 1e-9 * scale * c ** p:
            return p
    return 20


@pytest.mark.parametrize("wave", NEW + ["bior6.8"])
def test_bank_shape_placement_symmetry_sums_moments(wave):
    w = W.WAVELETS[wave]
    L, pad, m_rec, m_dec = SPEC[wave]
    assert all(len(w[k]) == L for k in ("rec_lo", "rec_hi", "dec_lo", "dec_hi"))
    assert w["pad"] == pad and 4 * pad == L - 2
    rec_lo, dec_lo = np.array(w["rec_lo"]), np.array(w["dec_lo"])
    rec_hi, dec_hi = np.array(w["rec_hi"]), np.array(w["dec_hi"])
    k = np.arange(L)
    assert np.array_equal(rec_hi, (-1.0) ** k * dec_lo) and np.array_equal(dec_hi, (-1.0) ** (k + 1) * rec_lo)
    if wave == "haar":
        assert np.count_nonzero(rec_lo) == 2 and np.count_nonzero(dec_lo) == 2
    else:   # PyWavelets placement: rec_lo centred at L/2 - 1, dec_lo at L/2 with one leading zero
        assert dec_lo[0] == 0.0 and dec_lo[1] != 0.0
        a, b = _support(rec_lo)
        assert a + b == 2 * (L // 2 - 1)
        a, b = _support(dec_lo)
        assert a + b == 2 * (L // 2)
    seg = lambda f: f[_support(f)[0]:_support(f)[1] + 1]
    for f in (rec_lo, dec_lo):                        # linear phase: symmetric low-pass filters ...
        assert np.array_equal(seg(f), seg(f)[::-1])
    for f in (rec_hi, dec_hi):                        # ... and high-pass filters symmetric up to sign (haar: antisymmetric)
        assert np.array_equal(np.abs(seg(f)), np.abs(seg(f))[::-1])
    # (the 16-digit CDF 9/7 taps of bior4.4 carry ~1e-12 of rounding)
    assert abs(rec_lo.sum() - np.sqrt(2)) < 1e-11 and abs(dec_lo.sum() - np.sqrt(2)) < 1e-11
    assert abs(rec_hi.sum()) < 1e-11 and abs(dec_hi.sum()) < 1e-11
    assert _moments(rec_hi) == m_rec and _moments(dec_hi) == m_dec


@pytest.mark.parametrize("wave", NEW)
def test_perfect_reconstruction_level_contract_and_dc_gain(wave):
    g = torch.Generator().manual_seed(len(wave))
    x = torch.randn(2, 3, 40, 36, dtype=torch.float64, generator=g)
    ll, yh = W.afb2d(x, wave)
    y = W.sfb2d(ll, yh, wave)
    assert y.shape == x.shape and (y - x).abs().max().item() < 1e-10
    n = 24
    pf = torch.randn(3, 2, n, n, dtype=torch.float64, generator=g)
    c = [torch.randn(3, 2, 3, n, n, dtype=torch.float64, generator=g), torch.randn(3, 2, 3, 2 * n, 2 * n, dtype=torch.float64, generator=g)]
    assert W.build_planes(pf, c, wave).shape == (3, 2, 4 * n, 4 * n)
    val = 0.7
    p = W.build_planes(torch.full((3, 1, n, n), val, dtype=torch.float64), [torch.zeros(3, 1, 3, n, n, dtype=torch.float64)], wave)
    assert p.shape == (3, 1, 2 * n, 2 * n)
    assert (p[..., 8:-8, 8:-8] - val).abs().max().item() < 1e-11      # IDWT(pad(2c), 0) = c away from the zero-padded border


@pytest.mark.parametrize("wave", NEW + ["bior6.8"])
def test_embedding_into_the_18_tap_frame(wave):
    """G[k + 9 - L/2] = g[k] with pad 4 reconstructs what g with its own pad does: the frame of the IDWT kernels"""
    w = W.WAVELETS[wave]
    framed = {k: embed18(w[k]) for k in ("rec_lo", "rec_hi", "dec_lo", "dec_hi")}
    W.WAVELETS["_framed"] = dict(framed, pad=4)
    try:
        g = torch.Generator().manual_seed(3)
        pf = torch.randn(3, 2, 16, 16, dtype=torch.float64, generator=g)
        c = [torch.randn(3, 2, 3, 16 * 2 ** l, 16 * 2 ** l, dtype=torch.float64, generator=g) for l in range(2)]
        a, b = W.build_planes(pf, c, wave), W.build_planes(pf, c, "_framed")
        assert a.shape == b.shape and (a - b).abs().max().item() <= 1e-14 * a.abs().max().item()
        # ... which is the closed form of one padded 1-D level with the framed taps
        x, d = torch.randn(12, dtype=torch.float64, generator=g), torch.randn(12, dtype=torch.float64, generator=g)
        P = w["pad"]
        pad = torch.nn.functional.pad
        ref = W.sfb1d(pad((2 * x).view(1, 1, 12, 1), (0, 0, P, P)), pad(d.view(1, 1, 12, 1), (0, 0, P, P)), w["rec_lo"], w["rec_hi"], 2)
        cf = W.idwt_level_closed_form_1d(x.tolist(), d.tolist(), framed["rec_lo"], framed["rec_hi"])
        assert (ref.flatten() - torch.tensor(cf, dtype=torch.float64)).abs().max().item() < 1e-14
    finally:
        del W.WAVELETS["_framed"]
