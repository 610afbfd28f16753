"""CPU checks of the float64 encoder references (tests/enc_reference.py) against the oracle where it computes the same thing, so that the
GPU encoder stage tests (test_gpu_encode_stages.py) compare the kernels with references that are themselves pinned."""
import numpy as np
import pytest

import enc_reference as R
import icc_util
from spec_cases import OPSIN_INV


def test_opsin_constants_invert_the_spec_inverse_matrix():
    assert np.abs(R.OPSIN_ABSORBANCE @ OPSIN_INV - np.eye(3)).max() < 1e-6


def test_srgb8_to_xyb_matches_the_oracle(oracle):
    rng = np.random.default_rng(1)
    rgb = np.concatenate([np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, axis=1),          # every level, gray
                          np.stack([np.arange(256), np.zeros(256), np.full(256, 255)], axis=1).astype(np.uint8),
                          rng.integers(0, 256, (4096, 3), dtype=np.uint8)])
    n = len(rgb)
    x, y, b = (np.zeros(n, np.float32) for _ in range(3))
    oracle.lib().jxlo_srgb8_to_xyb(np.ascontiguousarray(rgb).ctypes.data, n, x.ctypes.data, y.ctypes.data, b.ctypes.data)
    want = R.linear_to_xyb(np.stack([R.srgb_to_linear(rgb[:, k]) for k in range(3)], axis=-1))
    got = np.stack([x, y, b]).astype(np.float64)
    err = np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)
    assert np.all(err < 2e-6), err                  # fp32 evaluation in the oracle


def test_bgra_to_xyb_takes_the_b_channel_for_gray_and_the_profile_for_icc():
    rng = np.random.default_rng(2)
    bgra = rng.integers(0, 256, (5, 7, 4), dtype=np.uint8)
    g = R.bgra_to_xyb(bgra, gray=True)
    assert np.allclose(g, R.bgra_to_xyb(np.repeat(bgra[..., :1], 4, axis=-1)))
    # sRGB primaries: the colorants map to the identity
    srgb_para = icc_util.make_matrix_icc(icc_util.SRGB_PRIMS, gamma=2.2)
    assert icc_util.parse_icc(srgb_para)["tags"][b"rTRC"][:4] == b"para"
    curves, m = R.icc_to_linear_srgb(srgb_para)
    assert np.abs(m - np.eye(3)).max() < 5e-4                        # s15Fixed16 colorants of sRGB -> identity
    v = np.linspace(0, 1, 11)
    assert np.allclose(curves[0](v), v ** 2.2, atol=2e-5)


@pytest.mark.parametrize("curve", ["para", "curv1", "table"])
def test_icc_curves_follow_the_tag(curve):
    icc = icc_util.make_matrix_icc(icc_util.P3_PRIMS, gamma=2.2, curve=curve)
    curves, m = R.icc_to_linear_srgb(icc)
    v = np.arange(256) / 255.0
    tol = {"para": 1e-4, "curv1": 1e-12, "table": 2e-4}[curve]       # s15Fixed16 gamma; u8.8 gamma 2.19921875 vs itself; 1024-entry table
    want = v ** (563 / 256.0 if curve == "curv1" else 2.2)
    assert np.abs(curves[1](v) - want).max() < tol
    # P3 -> sRGB: rows sum to 1 (white stays white), the red primary is out of sRGB gamut in green and blue
    assert np.abs(m.sum(axis=1) - 1).max() < 1e-3 and m[1, 0] < 0 and m[2, 0] < 0


def test_dct8_matches_the_oracle_transform_and_layout(oracle):
    rng = np.random.default_rng(3)
    plane = rng.standard_normal((16, 24)).astype(np.float32)
    S = R.dct8_blocks(plane.astype(np.float64))
    for by in range(2):
        for bx in range(3):
            px = np.ascontiguousarray(plane[8 * by:8 * by + 8, 8 * bx:8 * bx + 8])
            coef = np.zeros(64, np.float32)
            oracle.lib().jxlo_transform_from_pixels(0, px.ctypes.data, 8, coef.ctypes.data)
            assert np.abs(coef - S[by, bx]).max() < 2e-6 * np.abs(S[by, bx]).max()
            assert abs(S[by, bx, 0] - px.astype(np.float64).mean()) < 1e-12
    # the absolute transform bounds every coefficient
    assert np.all(np.abs(S) <= R.dct8_blocks(plane.astype(np.float64), absolute=True) + 1e-12)


def test_gaborish_matches_the_oracle_stage(oracle):
    """The same check as test_gaborish_stage_matches_fp64_convolution, with the reference's own filter: mirrored at the extent it is given."""
    w, h = 203, 141
    data = oracle.encode(oracle.synthetic_image(w, h, seed=4), effort=7, gab=1, epf=0)
    d = oracle.decode(data, keep_stages=True)
    idct = d.stages["idct"].reshape(3, d.ypad, d.xpad).astype(np.float64)[:, :h, :w]
    gab = d.stages["gab"].reshape(3, d.ypad, d.xpad)[:, :h, :w]
    want = R.gaborish(idct)
    err = np.abs(gab - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2))
    assert np.all(err < 1e-6), err


def test_inverse_gaborish_nearly_inverts_the_filter():
    rng = np.random.default_rng(5)
    smooth = np.cumsum(np.cumsum(rng.standard_normal((3, 64, 72)), axis=1), axis=2)
    smooth /= np.abs(smooth).max()
    back = R.gaborish(R.inverse_gaborish(smooth))
    one = R.gaborish(R.inverse_gaborish(smooth, steps=1))
    assert np.abs(back - smooth).max() < np.abs(one - smooth).max() < np.abs(R.gaborish(smooth) - smooth).max()


def test_dequant_table_and_order_come_from_the_oracle(oracle):
    dq = np.zeros(3 * 64, np.float32)
    assert oracle.lib().jxlo_dequant_table(0, dq.ctypes.data) == 192
    order = np.zeros(64, np.uint32)
    assert oracle.lib().jxlo_natural_order(0, order.ctypes.data) == 64
    assert sorted(order) == list(range(64)) and order[0] == 0
    assert np.all(dq > 0)


def test_quantiser_rules():
    qf = np.array([0.0, 0.55, -0.56, 0.56, 1.5, 2.5, -2.5, 40000.0, -40000.0])
    assert list(R.quantise(qf)) == [0, 0, -1, 1, 2, 2, -2, 32767, -32768]
    q = np.array([0, 1, -1, 2, -3])
    got = R.dequant_bias(q, 1)
    assert np.allclose(got, [0, R.QUANT_BIAS[1], -R.QUANT_BIAS[1], 2 - 0.145 / 2, -3 + 0.145 / 3])
    assert list(R.ambiguous_rounding(np.array([2.5, 2.4, 0.5601]), 1e-3, dead_zone=True)) == [True, False, True]


def test_aq_and_cfl_rules():
    act = np.array([0.0, 1e9, R.AQ_REF - 1e-4])
    hf, mulq = R.aq_hf_mul(act, 10)
    assert list(hf) == [14, 8, 10] and np.isclose(mulq[2], 1.0)           # 1.35 level (flat), 0.75 level (busy), 1.0
    stats = np.zeros((9, 17, 4))                                          # 2 x 3 tiles, the last ones partial
    stats[..., 3] = 1.0
    stats[..., 1] = 0.5
    stats[..., 2] = 3.0                                                   # kb = 3: ytob = 84 * 2, clamped
    fx, fb, rx, rb, syy = R.cfl_factors(stats, 2, 3)
    assert fx.shape == (2, 3) and np.all(fx == 42) and np.all(fb == 127) and syy[1, 2] == 1.0
    fx, fb, *_ = R.cfl_factors(np.zeros((9, 17, 4)), 2, 3)
    assert np.all(fx == 0) and np.all(fb == 0)
