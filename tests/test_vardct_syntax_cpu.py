"""CPU tests of the VarDCT syntax the in-house encoders never write, through files of the independent writer (vardct_syntax_cases.py):
the oracle must decode each file to exactly the writer's integers, and its LF and reconstruction to the float64 references of dec_reference.py.
Each context, order and LZ77 rule the files exercise is shown to matter: the writer can encode with that one rule wrong, and the oracle must
then fail or decode other coefficients. (The GPU never decodes such a file.)"""
import numpy as np
import pytest

import dec_reference as ref
import jxl_spec_writer as jw
import vardct_syntax_cases as vc
from test_gpu_stages import TF_SRGB, orient, xyb_to_output
from test_gpu_vardct_syntax import FILTER_F32_REL

FP32_REL = 2e-6        # the oracle computes in fp32: relative to each channel's range


def _decode(oracle, name, wrong=None):
    data, ints = vc.case(name, wrong)
    return oracle.decode(data, keep_stages=True), ints


def _rel(got, want):
    got, want = np.asarray(got, np.float64).reshape(3, -1), np.asarray(want, np.float64).reshape(3, -1)
    return np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)


@pytest.mark.parametrize("name", vc.NAMES)
def test_oracle_decodes_the_writers_integers(oracle, name):
    d, c = _decode(oracle, name)
    xb, yb = c["xb"], c["yb"]
    w, h = (c["h"], c["w"]) if c["kw"]["orientation"] >= 5 else (c["w"], c["h"])     # the oriented image's size
    assert (d.width, d.height, d.xpad, d.ypad) == (w, h, 8 * xb, 8 * yb)
    assert np.array_equal(d.stages["coeffs"].reshape(3, -1, 64), c["coeffs"])
    assert np.count_nonzero(c["coeffs"]) > 0
    assert np.array_equal(d.stages["lfq"], np.stack(c["lfq"]))
    hf = np.zeros((yb, xb), np.int64)
    for by, bx, s, hm in c["blocks"]:
        cy, cx = jw.VARBLOCK[s]
        hf[by:by + cy, bx:bx + cx] = hm
    assert np.array_equal(d.stages["hf_mul"], hf)
    assert np.array_equal(d.stages["ytox"], c["ytox"]) and np.array_equal(d.stages["ytob"], c["ytob"])
    kw = c["kw"]
    assert (d.global_scale, d.quant_lf, d.x_qm_scale, d.b_qm_scale) == (kw["global_scale"], kw["quant_lf"], kw["x_qm_scale"], kw["b_qm_scale"])


@pytest.mark.parametrize("name", vc.NAMES)
def test_oracle_lf_matches_float64(oracle, name):
    d, c = _decode(oracle, name)
    kw = c["kw"]
    want = ref.lf_planes(c["lfq"], kw["lf_dequant"], kw["global_scale"], kw["quant_lf"], kw["extra_precision"], kw["cfl"])
    if not kw["skip_smoothing"]:
        raw = want
        want = ref.lf_smoothing(raw, kw["lf_dequant"], kw["global_scale"], kw["quant_lf"])
        changed = np.abs(want - raw) > 1e-6 * np.abs(raw).max()
        assert changed[:, 1:-1, 1:-1].mean() > 0.2, "smoothing changes too few LF samples of %s" % name
    err = _rel(d.stages["lf"], want)
    assert np.all(err <= FP32_REL), err


@pytest.mark.parametrize("name", ["dct8_single_band", "dct8_bands"])
def test_oracle_reconstruction_matches_float64(oracle, name):
    d, c = _decode(oracle, name)
    qb = vc.OPSIN[2] if c["kw"]["opsin"] else None
    want = ref.dct8_reconstruction(c, ref.table0_of(c), qb)
    err = _rel(d.stages["idct"], want)
    assert np.all(err <= FP32_REL), err


# rule -> the case whose file it changes (one group has one preset; DCT8-only files have no multi-cell counts; pred 63 needs dense DCT8 pairs)
WRONG_CASE = {"preset_offset": "two_pass", "qf_ge": "two_pass", "lf_idx_xyb": "two_pass", "block_ctx_c": "two_pass", "perm_inverted": "two_pass",
              "perm_no_skip": "two_pass", "nz_bucket_63": "dct8_bands", "prev_lt": "two_pass", "lz77_multiplier": "lz77", "nz_floor": "two_pass"}


@pytest.mark.parametrize("rule", jw.WRONG_RULES)
def test_each_rule_matters(oracle, rule):
    assert set(WRONG_CASE) == set(jw.WRONG_RULES)
    data, c = vc.case(WRONG_CASE[rule], rule)
    assert data != vc.case(WRONG_CASE[rule])[0]
    try:
        d = oracle.decode(data, keep_stages=True)
    except oracle.OracleError:
        return
    assert not np.array_equal(d.stages["coeffs"].reshape(3, -1, 64), c["coeffs"]), "the oracle decodes the same coefficients with %s" % rule


def test_lz77_copies_reach_both_sides_of_the_special_distance_range(monkeypatch):
    """A Modular reader sends distance symbols < 120 through its special-distance table and subtracts 119 from the others; the AC rule is
    symbol + 1. The lz77 case must carry symbols on both sides of 120 (and symbol 0) for a reader that mixes the rules up to decode it wrongly."""
    seen = []
    copies = jw.lz77_copies

    def spy(*a):
        out = copies(*a)
        seen.extend(it[3] for it in out if it[0] == "copy")
        return out

    monkeypatch.setattr(jw, "lz77_copies", spy)
    c = vc._ints("lz77")
    jw.vardct_frame(c["w"], c["h"], c["lfq"], c["blocks"], c["ytox"], c["ytob"], c["coeffs"], **c["kw"])
    assert 0 in seen and any(1 <= s < 120 for s in seen) and any(s >= 120 for s in seen)


def test_idct8_reference_matches_the_oracle_transform(oracle):
    rng = np.random.default_rng(5)
    for _ in range(4):
        coef = rng.normal(size=64).astype(np.float32)
        px = np.zeros(64, np.float32)
        oracle.lib().jxlo_transform_to_pixels(0, coef.ctypes.data, px.ctypes.data, 8)
        want = ref.idct8(coef.astype(np.float64).reshape(8, 8))
        assert np.abs(px.reshape(8, 8) - want).max() <= 1e-5 * np.abs(want).max()


def test_mode6_table_from_library_parameters_equals_the_library_table(oracle):
    dq = np.zeros(192, np.float32)
    assert oracle.lib().jxlo_dequant_table(0, dq.ctypes.data) == 192
    lib = [[3150.0, 0.0, -0.4, -0.4, -0.4, -2.0], [560.0, 0.0, -0.3, -0.3, -0.3, -0.3], [512.0, -2.0, -1.0, 0.0, -1.0, -2.0]]   # SURVEY A.8
    want = ref.dequant_table(8, 8, lib)
    assert np.abs(dq.reshape(3, 64) - want).max() <= 2e-6 * np.abs(want).max()


def test_raw_dequantisation_tables_are_refused(oracle):
    with pytest.raises(oracle.OracleError, match="RAW"):
        oracle.decode(vc.raw_table_file())


# ------------------------------------------------------------------------------------------------ restoration filters
def _restore(c, planes, switches=()):
    kw = c["kw"]
    return ref.restore(planes, c["w"], c["h"], kw["gab"], kw["epf_iters"], kw["restoration"], c["sharp"], c["blocks"], kw["global_scale"], switches)


@pytest.mark.parametrize("name", vc.FILTER_NAMES)
def test_oracle_filters_match_float64(oracle, name):
    """The oracle's gaborish and EPF stages, fed with its own reconstruction, against the float64 reference (each stage on its own)."""
    d, c = _decode(oracle, name)
    kw, w, h = c["kw"], c["w"], c["h"]
    st = {k: d.stages[k].reshape(3, d.ypad, d.xpad)[:, :h, :w] for k in ("idct", "gab", "epf")}
    gab = ref.gaborish(st["idct"], ref.restoration_params(kw["restoration"])["gab_w"]) if kw["gab"] else st["idct"].astype(np.float64)
    assert np.all(_rel(st["gab"], gab) <= FP32_REL), _rel(st["gab"], gab)
    epf = ref.restore(st["gab"], w, h, False, kw["epf_iters"], kw["restoration"], c["sharp"], c["blocks"], kw["global_scale"])
    assert np.all(_rel(st["epf"], epf) <= FP32_REL), _rel(st["epf"], epf)


def test_filter_cases_sit_away_from_the_skip_threshold():
    """EPF is continuous in its inputs except where a cell's inv_sigma crosses the skip threshold: no cell lies within 1e-4 of it, and every
    EPF case with more than one cell has both filtered and skipped cells (the single-cell frames are filtered)."""
    for name in vc.FILTER_NAMES:
        c = vc._ints(name)
        kw = c["kw"]
        if not kw["epf_iters"]:
            continue
        isg = ref.inv_sigma(c["sharp"], c["blocks"], kw["global_scale"], ref.restoration_params(kw["restoration"]))
        assert np.abs(isg / ref.MIN_INV_SIGMA - 1).min() > 1e-4, name
        skipped = int((isg < ref.MIN_INV_SIGMA).sum())
        assert 0 < skipped < isg.size if isg.size > 1 else skipped == 0, (name, skipped, isg.size)


def test_filter_cases_carry_custom_and_default_parameters():
    o = {n: vc.SPECS[n][2] for n in vc.FILTER_NAMES}
    r = vc.RESTORATION
    assert len(set(r["gab_w"][0::2])) == 3 and len(set(r["gab_w"][1::2])) == 3
    lut = list(r["sharp_lut"])
    assert 0.0 in lut and lut != sorted(lut) and any(r[k] != ref.DEFAULT_RESTORATION[k] for k in ("quant_mul", "border_sad_mul"))
    assert r["pass0_sigma_scale"] != ref.DEFAULT_RESTORATION["pass0_sigma_scale"] and r["pass2_sigma_scale"] != ref.DEFAULT_RESTORATION["pass2_sigma_scale"]
    assert [n for n in o if not o[n].get("restoration")] == ["gab_epf1"]
    assert [n for n in o if (o[n].get("restoration") or {}).get("all_default")] == ["all_default_224x100"]
    assert any(o[n].get("epf") == 3 and -(-vc.SPECS[n][1] // 256) >= 3 for n in o)


def _output(c, xyb):
    kw = c["kw"]
    inv, bias, _ = kw["opsin"]
    tf = (kw["color"] or {}).get("tf", TF_SRGB)
    return orient(xyb_to_output(xyb, tf=tf, opsin_inv=inv, opsin_bias=[-v for v in bias]), kw["orientation"])


@pytest.mark.parametrize("switch", ref.SWITCHES)
def test_each_filter_rule_matters(oracle, switch):
    """Each rule of the reference, applied differently, moves some case's output samples by at least 20x the bound the GPU's samples are held
    to (FILTER_F32_REL, relative to max(|sample|, 1e-3)): the cases can tell each rule from its alternative."""
    worst = 0.0
    for name in vc.FILTER_NAMES:
        d, c = _decode(oracle, name)
        idct = d.stages["idct"].reshape(3, d.ypad, d.xpad).astype(np.float64)
        real = _output(c, _restore(c, idct))
        moved = _output(c, _restore(c, idct, (switch,)))
        worst = max(worst, float((np.abs(moved - real) / np.maximum(np.abs(real), 1e-3)).max()))
    assert worst >= 20 * FILTER_F32_REL, "%s moves the output by %.3g at most" % (switch, worst)
