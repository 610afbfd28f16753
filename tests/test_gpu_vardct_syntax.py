"""-m gpu tests of the VarDCT syntax the in-house encoders never write (custom LF dequantisation, block-context maps, CfL parameters,
dequantisation tables, HF presets, coefficient orders, two passes, prefix and LZ77 AC codes, a custom opsin matrix), through the files of
the independent writer (vardct_syntax_cases.py), stage by stage:
  * quantised coefficients (stage 4): exactly the writer's integers (a wrong lf_idx or block context changes them);
  * LF (stage 3): the float64 reference, with adaptive smoothing where the file asks for it;
  * reconstruction (stage 0): the float64 reference on DCT8-only files, the oracle's on files with varblocks;
  * output samples: the GPU's own stage-0 planes through the float64 restoration filters (gaborish, EPF with the file's parameters) and
    colour conversion under the file's own opsin matrix, on every render kernel; one DCT8-only file from the writer's integers alone;
  * every entry point (LoadImage, a bundled batch with 16-lane AC warps, a band decode) gives the same pixels.
The CPU side (test_vardct_syntax_cpu.py) holds the oracle to the same integers and shows that each rule the files exercise matters."""
import numpy as np
import pytest

import dec_reference as ref
import vardct_syntax_cases as vc
import jxl_spec_writer as jw
from test_gpu_stages import TF_LINEAR, TF_SRGB, _gpu_coeffs, _gpu_planes, _oracle_planes, _rel_err, orient, render_branch, xyb_to_output

pytestmark = pytest.mark.gpu

# Relative to the channel's range, about 4x the worst value measured on a B200 (1000 W) over these files.
LF_REL_BOUND = 6e-7      # measured 1.35e-7 (X channel, two_lf_groups, against float64)
LF_SMOOTH_REL_BOUND = 1.8e-6   # with adaptive smoothing, against float64; measured 4.4e-7 (B channel, all_default_224x100)
RECON_REL_BOUND = 1e-6   # measured 2.4e-7 (X channel, dct8_bands, against float64); 1.7e-7 against the oracle (multi_group_ans)
U8_DELTA = 4e-5          # |got - real| <= 0.5 + delta code units; measured 0.5 - 2.0e-5 (dct8_bands, k_output)
# Restored samples (GPU stage-0 planes -> float64 gaborish + EPF + colour) against the GPU's rendered output
# (k_output, no filters: U8_DELTA). Measured on a B200 (1000 W) over the filter cases:
FILTER_U8_DELTA = 1.2e-4   # code units over 0.5; measured 2.8e-5 (wide_193x161, k_render_wide_tma<1,false> and <1,true>)
FILTER_U16_DELTA = 0.07    # code units over 0.5; measured 0.016 (u16_orient6_200x136, k_render<1,1,false>)
FILTER_F32_REL = 1.3e-4    # relative to max(|real|, 1e-3); measured 3.1e-5 (dct8_f32_linear, k_render<1,1,false>)
INTEGERS_F32_REL = 4e-4    # the same file from the writer's integers (reconstruction included); measured 9.8e-5

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
    "custom restoration parameters": "epf3_132x67",
    "RestorationFilter all_default": "all_default_224x100",
}

# Every kernel render_branch() can return for a VarDCT frame with filters, and the case (and output) that selects it
RENDER_KERNEL = {
    "k_render<0,1,true>": "epf1_260x97", "k_render<0,1,false>": "epf1_95x63",
    "k_render<0,2,true>": "epf2_128x65", "k_render<0,2,false>": "epf2_161x33",
    "k_render<0,3,true>": "epf3_132x67", "k_render<0,3,false>": "tiny_1x1",
    "k_render<1,0,true>": "gab_192x129", "k_render<1,0,false>": "gab_127x95",
    "k_render<1,1,false>": "u16_orient6_200x136",
    "k_render<1,2,true>": "all_default_224x100", "k_render<1,2,false>": "tiny_5x3",
    "k_render<1,3,true>": "bands_300x530", "k_render<1,3,false>": "tiny_9x7",
    "k_render_wide_tma<1,false>": "wide_193x161", "k_render_wide_tma<1,true>": "wide_193x161",
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
def test_lf_planes(gpu, name):
    data, c = vc.case(name)
    kw = c["kw"]
    got = _gpu_planes(gpu, data, 3, c["w"], c["h"])
    want = ref.lf_planes(c["lfq"], kw["lf_dequant"], kw["global_scale"], kw["quant_lf"], kw["extra_precision"], kw["cfl"])
    if not kw["skip_smoothing"]:
        want = ref.lf_smoothing(want, kw["lf_dequant"], kw["global_scale"], kw["quant_lf"])
    err = _rel_err(got, want)
    bound = LF_REL_BOUND if kw["skip_smoothing"] else LF_SMOOTH_REL_BOUND
    assert np.all(err <= bound), "LF planes differ by %s of the channel range" % err


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


def _sample(kw):
    return {8: "u8", 16: "u16", 32: "f32"}[kw["bits"]]


def _outputs(name):
    """(bgra, kernel) of every output a case is decoded to: LoadImage, and the BGRA32 surface where that takes the wide render kernel."""
    w, h, _ = vc.SPECS[name]
    kw = vc._ints(name)["kw"]
    gab, epf, sample, orientation = int(kw["gab"]), kw["epf_iters"], _sample(kw), kw["orientation"]
    out = [(False, render_branch(gab, epf, w, h, sample=sample, orientation=orientation))]
    bgra = render_branch(gab, epf, w, h, sample=sample, orientation=orientation, bgra=True)
    if bgra.startswith("k_render_wide_tma"):
        out.append((True, bgra))
    return out


def _real(xyb, kw):
    """[h][w][3] (oriented) output samples of XYB planes under the file's opsin matrix, transfer function and orientation."""
    inv, bias, _ = kw["opsin"]
    tf = (kw["color"] or {}).get("tf", TF_SRGB)
    return orient(xyb_to_output(xyb, tf=tf, opsin_inv=inv, opsin_bias=[-v for v in bias]), kw["orientation"])


def _worst(got, real, sample):
    """The measure each bound applies to: code units over 0.5 (u8, u16), or the relative difference (f32)."""
    g = got.astype(np.float64)
    if sample == "f32":
        return float((np.abs(g - real) / np.maximum(np.abs(real), 1e-3)).max())
    scale = 255.0 if sample == "u8" else 65535.0
    return float((np.abs(g - np.clip(real, 0, 1) * scale) - 0.5).max())


FILTER_BOUND = {"u8": FILTER_U8_DELTA, "u16": FILTER_U16_DELTA, "f32": FILTER_F32_REL}


def _rendered(gpu, data, bgra):
    if bgra:
        got = gpu.load_image_bgra(data)
        assert np.all(got[..., 3] == 255)
        return got[..., 2::-1]
    return _load(gpu, data)


def test_every_render_kernel_is_exercised():
    """The 15 kernels render_branch() returns for VarDCT frames with filters, each selected by the case listed for it (and by no
    unlisted surprise): every fused-render instantiation has a case whose samples are held to float64."""
    want = {"k_render<%d,%d,%s>" % (g, e, f) for g, e in ((0, 1), (0, 2), (0, 3), (1, 0), (1, 2), (1, 3)) for f in ("true", "false")}
    want |= {"k_render<1,1,false>", "k_render_wide_tma<1,false>", "k_render_wide_tma<1,true>"}
    assert set(RENDER_KERNEL) == want and len(want) == 15
    reached = {k for n in vc.FILTER_NAMES for _, k in _outputs(n)}
    assert reached == want
    for kernel, name in RENDER_KERNEL.items():
        assert kernel in [k for _, k in _outputs(name)], (kernel, name)


@pytest.mark.parametrize("name", vc.FILTER_NAMES + ["dct8_bands"])
def test_filters_match_float64(gpu, name):
    """The GPU's own reconstruction (stage 0) through the float64 gaborish, EPF and colour conversion equals what it renders, to fp32
    level: only the render kernel's arithmetic is under test (dct8_bands: no filters, k_output under the file's opsin matrix)."""
    data, c = vc.case(name)
    kw, w, h = c["kw"], c["w"], c["h"]
    planes = _gpu_planes(gpu, data, 0, w, h).astype(np.float64)
    xyb = ref.restore(planes, w, h, kw["gab"], kw["epf_iters"], kw["restoration"], c["sharp"], c["blocks"], kw["global_scale"])
    real = _real(xyb, kw)
    sample = _sample(kw)
    for bgra, kernel in _outputs(name):
        got = _rendered(gpu, data, bgra)
        assert got.shape == real.shape, (kernel, got.shape, real.shape)
        worst = _worst(got, real, "u8" if bgra else sample)
        bound = U8_DELTA if kernel == "k_output" else FILTER_BOUND["u8" if bgra else sample]
        assert worst <= bound, "%s (%s): worst %.4g" % (name, kernel, worst)


def test_filtered_samples_from_the_writers_integers(gpu):
    """DCT8 only: dequantisation, CfL and IDCT (dct8_reconstruction), gaborish + EPF with custom parameters (restore) and the f32 linear
    colour conversion, all float64 from the integers the writer put in the file: neither the oracle nor a GPU stage is involved."""
    data, c = vc.case("dct8_f32_linear")
    kw, w, h = c["kw"], c["w"], c["h"]
    assert {b[2] for b in c["blocks"]} == {0} and kw["skip_smoothing"] and kw["restoration"] and _sample(kw) == "f32"
    planes = ref.dct8_reconstruction(c, ref.table0_of(c), kw["opsin"][2])
    xyb = ref.restore(planes, w, h, kw["gab"], kw["epf_iters"], kw["restoration"], c["sharp"], c["blocks"], kw["global_scale"])
    worst = _worst(_load(gpu, data), _real(xyb, kw), "f32")
    assert worst <= INTEGERS_F32_REL, "worst relative difference %.4g" % worst


def test_bands_of_a_gaborish_epf3_frame_equal_load_image(gpu):
    data = vc.case("bands_300x530")[0]
    full = _load(gpu, data)
    w, h, gdim, rows = gpu.band_layout(data)
    assert rows >= 3 and vc.SPECS["bands_300x530"][2]["epf"] == 3
    parts = [gpu.decode_band(data, a, b) for a, b in ((0, 1), (1, 2), (2, rows))]
    assert np.array_equal(np.concatenate(parts, axis=0), full)


def _modular_file(gab, epf_iters, restoration=None):
    rng = np.random.default_rng(9)
    channels = [rng.integers(0, 256, (24, 40)).tolist() for _ in range(3)]
    b = jw.Bits()
    b.u(16, 0x0AFF)
    jw.size_header(b, 40, 24)
    jw.image_metadata(b)
    b.pad_to_byte()
    return b.bytes() + jw.modular_frame(channels, 0, gab=gab, epf_iters=epf_iters, restoration=restoration)


@pytest.mark.parametrize("gab,epf_iters,restoration", [(True, 0, None), (False, 1, None), (True, 2, dict(sigma_for_modular=0.75))])
def test_modular_frames_with_restoration_filters_are_refused(gpu, gab, epf_iters, restoration):
    with pytest.raises(gpu.FormatException, match="restoration filters on Modular") as e:
        _load(gpu, _modular_file(gab, epf_iters, restoration))
    assert e.value.status == "DecodeError"
    _load(gpu, _modular_file(False, 0))     # the same file without filters decodes


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
