"""-m gpu tests of the VarDCT syntax the in-house encoders never write (custom LF dequantisation, block-context maps, CfL parameters,
dequantisation tables, HF presets, coefficient orders, two passes, prefix and LZ77 AC codes, a custom opsin matrix), through the files of
the independent writer (vardct_syntax_cases.py), stage by stage:
  * quantised coefficients (stage 4): exactly the writer's integers (a wrong lf_idx or block context changes them);
  * LF (stage 3): the float64 reference where smoothing is off, the oracle where it is on;
  * reconstruction (stage 0): the float64 reference on DCT8-only files, the oracle's on files with varblocks;
  * output samples: the float64 colour conversion of the oracle's planes under the file's own opsin matrix;
  * every entry point (LoadImage, a bundled batch with 16-lane AC warps, a band decode) gives the same pixels.
The CPU side (test_vardct_syntax_cpu.py) holds the oracle to the same integers and shows that each rule the files exercise matters."""
import numpy as np
import pytest

import dec_reference as ref
import vardct_syntax_cases as vc
from test_gpu_stages import _gpu_coeffs, _gpu_planes, _oracle_planes, _rel_err, render_branch, xyb_to_output

pytestmark = pytest.mark.gpu

# Relative to the channel's range, about 4x the worst value measured on a B200 (1000 W) over these files.
LF_REL_BOUND = 6e-7      # measured 1.35e-7 (X channel, two_lf_groups, against float64)
RECON_REL_BOUND = 1e-6   # measured 2.4e-7 (X channel, dct8_bands, against float64); 1.7e-7 against the oracle (multi_group_ans)
U8_DELTA = 4e-5          # |got - real| <= 0.5 + delta code units; measured 0.5 - 2.0e-5 (dct8_bands) and 0.5 - 4.5e-6 (gab_epf1)

# Which case carries which feature of the writer (a coverage guard, like test_every_reconstruction_kernel_is_exercised).
FEATURES = {
    "multi-group TOC, ragged last group row and column": "multi_group_ans",
    "single TOC entry": "single_group_prefix",
    "two LF groups": "two_lf_groups",
    "DCT16, DCT32, DCT16X8, DCT8X16": "multi_group_ans",
    "custom LfChannelDequantization": "multi_group_ans",
    "global_scale and quant_lf": "multi_group_ans",
    "extra_precision 1-3": "lz77",
    "custom BlockCtxMap": "multi_group_ans",
    "custom ColorCorrelation": "multi_group_ans",
    "hf_mul 1 .. 256 across the qf thresholds": "multi_group_ans",
    "CfL tiles -128 and 127": "multi_group_ans",
    "mode-6 tables, one with a single band": "multi_group_ans",
    "Library tables": "multi_group_ans",
    "several HF presets": "multi_group_ans",
    "coefficient-order permutations": "multi_group_ans",
    "two passes with a shift": "two_pass",
    "ANS AC code (k_ac_vardct<true>)": "multi_group_ans",
    "prefix AC code (k_ac_vardct<false>)": "single_group_prefix",
    "LZ77 AC code (k_ac_vardct<false>)": "lz77",
    "custom opsin matrix and quant biases": "dct8_single_band",
    "adaptive LF smoothing": "smoothing",
    "gaborish + EPF 1 render": "gab_epf1",
}
REQUIRED = {"multi-group TOC, ragged last group row and column", "single TOC entry", "two LF groups", "DCT16, DCT32, DCT16X8, DCT8X16",
            "custom LfChannelDequantization", "global_scale and quant_lf", "extra_precision 1-3", "custom BlockCtxMap", "custom ColorCorrelation",
            "hf_mul 1 .. 256 across the qf thresholds", "CfL tiles -128 and 127", "mode-6 tables, one with a single band", "Library tables",
            "several HF presets", "coefficient-order permutations", "two passes with a shift", "ANS AC code (k_ac_vardct<true>)",
            "prefix AC code (k_ac_vardct<false>)", "LZ77 AC code (k_ac_vardct<false>)", "custom opsin matrix and quant biases"}


def _staged_ac_bytes(kw):
    """Shared memory the staged AC tables of a single-pass ANS case take (RunLf's code_bytes + 64 in decode_engine.cu; 8 clusters, log_alpha 8):
    k_ac_vardct<true> runs when this is at most 96 KB and the code is neither prefix nor LZ77."""
    up = lambda n: (n + 15) & ~15
    num_ctx = 495 * (max(kw["presets"]) + 1 if kw["presets"] else 1) * (kw["bctx"].num_ctx if kw["bctx"] else 15)
    return up(8 * 4) + up(num_ctx) + up((8 << 8) * 8) + 64


def test_every_feature_has_a_case():
    """The table above names every feature, and each named case has the structure the name claims."""
    assert REQUIRED <= set(FEATURES) and set(FEATURES.values()) <= set(vc.NAMES)
    assert {k for k in FEATURES if "k_ac_vardct<true>" in k} and {k for k in FEATURES if "k_ac_vardct<false>" in k}
    o = {n: vc.SPECS[n][2] for n in vc.NAMES}
    i = {n: vc._ints(n) for n in ("multi_group_ans", "single_group_prefix", "two_lf_groups", "two_pass", "lz77")}
    m = i["multi_group_ans"]
    kw = m["kw"]
    assert -(-m["xb"] // 32) * -(-m["yb"] // 32) > 1 and m["w"] % 256 and m["h"] % 256 and -(-m["yb"] // 32) >= 3
    assert -(-i["single_group_prefix"]["xb"] // 32) * -(-i["single_group_prefix"]["yb"] // 32) == 1 and not i["single_group_prefix"]["kw"]["pass_shift"]
    assert -(-i["two_lf_groups"]["xb"] // 256) == 2
    assert {b[2] for b in m["blocks"]} == {0, 4, 5, 6, 7}
    assert kw["lf_dequant"] and kw["cfl"] and kw["bctx"] and kw["global_scale"] != 32768 and kw["quant_lf"] != 64
    assert all(kw["bctx"].lf_thr) and len(kw["bctx"].qf_thr) > 1
    assert {b[3] for b in m["blocks"]} >= {1, 256} and m["ytox"].min() == -128 and m["ytob"].max() == 127
    assert any(len(t[0]) == 1 for t in kw["tables"].values()) and len(kw["tables"]) < 17
    assert max(kw["presets"]) >= 1 and kw["orders"] and not kw["pass_shift"]
    assert i["two_pass"]["kw"]["pass_shift"] and i["two_pass"]["kw"]["orders"]
    assert {vc.SPECS[n][2].get("extra_precision", 0) for n in vc.NAMES} >= {1, 2, 3}
    assert i["single_group_prefix"]["kw"]["code"] == "prefix" and i["lz77"]["kw"]["code"] == "lz77" and kw["code"] == "ans"
    assert _staged_ac_bytes(kw) <= 96 * 1024                     # so multi_group_ans decodes through k_ac_vardct<true>
    assert vc.SPECS[FEATURES["custom opsin matrix and quant biases"]][2]["opsin"] and o["smoothing"]["smoothing"] and o["gab_epf1"]["gab"]


@pytest.mark.parametrize("name", vc.NAMES)
def test_coefficients_are_the_writers(gpu, name):
    data, c = vc.case(name)
    got, outside = _gpu_coeffs(gpu, data, c["w"], c["h"])
    assert outside == 0, "non-zero coefficients in cells outside the image"
    want = c["coeffs"].reshape(3, -1)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%d coefficients differ, first at %s: GPU %d, writer %d" % (len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])


@pytest.mark.parametrize("name", vc.NAMES)
def test_lf_planes(gpu, oracle, name):
    data, c = vc.case(name)
    kw = c["kw"]
    got = _gpu_planes(gpu, data, 3, c["w"], c["h"])
    if kw["skip_smoothing"]:
        want = ref.lf_planes(c["lfq"], kw["lf_dequant"], kw["global_scale"], kw["quant_lf"], kw["extra_precision"], kw["cfl"])
    else:
        want = oracle.decode(data, keep_stages=True).stages["lf"].reshape(3, c["yb"], c["xb"]).astype(np.float64)
    err = _rel_err(got, want)
    assert np.all(err <= LF_REL_BOUND), "LF planes differ by %s of the channel range" % err


@pytest.mark.parametrize("name", vc.NAMES)
def test_reconstruction(gpu, oracle, name):
    data, c = vc.case(name)
    got = _gpu_planes(gpu, data, 0, c["w"], c["h"]).astype(np.float64)
    if {b[2] for b in c["blocks"]} == {0} and c["kw"]["skip_smoothing"]:
        want = ref.dct8_reconstruction(c, ref.table0_of(c), vc.OPSIN[2] if c["kw"]["opsin"] else None)
    else:
        want = _oracle_planes(oracle.decode(data, keep_stages=True), "idct")
    err = _rel_err(got, want)
    assert np.all(err <= RECON_REL_BOUND), "reconstruction differs by %s of the channel range" % err


@pytest.mark.parametrize("name,branch", [("dct8_bands", "k_output"), ("gab_epf1", "k_render_wide_tma<1,false>")])
def test_rendered_samples_under_the_files_opsin_matrix(gpu, oracle, name, branch):
    data, c = vc.case(name)
    kw = c["kw"]
    assert kw["opsin"] is not None and render_branch(int(kw["gab"]), kw["epf_iters"], c["w"], c["h"]) == branch
    d = oracle.decode(data, keep_stages=True)
    planes = _oracle_planes(d, "epf")[:, :c["h"], :c["w"]]
    inv, bias, _ = kw["opsin"]
    real = np.clip(xyb_to_output(planes, opsin_inv=inv, opsin_bias=[-v for v in bias]), 0, 1) * 255.0
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(data, image)
    excess = np.abs(image.layer_data.color.astype(np.float64) - real) - 0.5
    assert float(excess.max()) <= U8_DELTA, "worst |got - real| = 0.5 + %.4g code units" % float(excess.max())


def _load(gpu, data):
    image = gpu.DecoderImage()
    gpu.JpegXLNative.LoadImage(data, image)
    return image.layer_data.color


def test_batch_and_band_decode_equal_load_image(gpu):
    files = [vc.case(n)[0] for n in vc.NAMES]
    singles = [_load(gpu, f) for f in files]
    # 70 files, 40 in flight: bundled entropy launches and 16-lane AC warps. Only single-pass multi-group files with ANS codes that fit the
    # staged tables are bundled into k_ac_vardct_multi (multi_group_ans, two_lf_groups, dct8_bands and smoothing here); the prefix, LZ77,
    # two-pass and single-group files take the per-frame AC path in the same batch
    batch = [files[i % len(files)] for i in range(70)]
    outs = [np.zeros_like(singles[i % len(files)]) for i in range(70)]
    assert gpu.decode_batch(batch, outs, max_in_flight=40) == [0] * 70
    for i, o in enumerate(outs):
        assert np.array_equal(o, singles[i % len(files)]), (i, vc.NAMES[i % len(files)])
    data = vc.case("multi_group_ans")[0]
    full = singles[vc.NAMES.index("multi_group_ans")]
    w, h, gdim, rows = gpu.band_layout(data)
    assert rows >= 3
    parts = [gpu.decode_band(data, a, b) for a, b in ((0, 1), (1, 2), (2, rows))]
    assert np.array_equal(np.concatenate(parts, axis=0), full)


def test_raw_dequantisation_tables_are_refused(gpu):
    with pytest.raises(gpu.FormatException, match="RAW") as e:
        _load(gpu, vc.raw_table_file())
    assert e.value.status == "DecodeError"
