"""CPU: the oracle against the committed golden vectors (generated from the UNMODIFIED
reference by the scripts in tests/golden/)."""
import numpy as np
import pytest
import torch

from oracle import color_ref, lhn_ref, synth
from tests import util


def test_oracle_vs_golden_64(synth_sd):
    g = util.golden("lhn_64.npz")
    L, ab, m = g["L"], g["ab"], g["mask"]
    (reg, dist), inter = util.oracle_forward(synth_sd, L, ab, m, 0.5, dist=True, intermediates=True)
    for i in range(2):
        # golden holds the reference's quirky dist=True return: tanh*110*110 (model.py:166-168)
        assert util.maxabs(reg[i] * 110.0, g["reg_quirk_%d" % i]) < 5e-2
        assert util.maxabs(reg[i], g["reg_quirk_%d" % i] / 110.0) < 5e-4
        assert util.maxabs(dist[i], g["dist16_%d" % i]) < 1e-6
        names = {"model1": "conv1_2", "model2": "conv2_2", "model3": "conv3_3", "model4": "conv4_3",
                 "model5": "conv5_3", "model6": "conv6_3", "model7": "conv7_3", "model8": "conv8_3",
                 "model9": "conv9_3", "model10": "conv10_2"}
        for blk, nm in names.items():
            t = inter[nm][i]
            assert util.maxabs(t[:8], g["%s_%d_c8" % (blk, i)]) < 2e-4, blk
            assert util.maxabs(t.mean(dim=(1, 2)), g["%s_%d_chmean" % (blk, i)]) < 1e-4, blk


@pytest.mark.parametrize("case,mc", [("mc0_zero", 0.0), ("mc0_kat", 0.0), ("mc1_rand5", 0.5)])
def test_oracle_vs_golden_256(synth_sd, case, mc):
    g = util.golden("lhn_256.npz")
    L = g["img_l_mc"].astype(np.float32)[None]
    if case.endswith("zero"):
        ab, m = np.zeros((2, 256, 256)), np.zeros((1, 256, 256))
    elif case.endswith("kat"):
        ab, m = np.zeros((2, 256, 256)), np.zeros((1, 256, 256))
        synth.put_point(ab, m, [135, 160], 3, [23, -69])
        synth.put_point(ab, m, [100, 160], 3, [0, 0])
    else:
        ab, m = synth.synthetic_hints(256, 5, 0)
    out = util.oracle_forward(synth_sd, L, ab[None], m[None], mc)
    assert util.maxabs(out[0], g[case + "_ab_raw"]) < 2e-4


def test_golden_image_prep_and_post():
    """img_l_mc and the uint8 post-process of the reference wrapper are reproduced by
    oracle/color_ref.py from the stored resized RGB / raw ab (rows a10, a11)."""
    g = util.golden("lhn_256.npz")
    lab = color_ref.rgb2lab_transpose(g["img_rgb"])
    assert np.max(np.abs(lab[[0]] - 50.0 - g["img_l_mc"])) < 1e-9
    rgb = color_ref.lab2rgb_transpose(lab[[0]], g["mc0_kat_ab_raw"].astype(np.float64))
    assert np.array_equal(rgb, g["mc0_kat_rgb"])
    out_ab = color_ref.rgb2lab_transpose(rgb)[1:]
    assert np.max(np.abs(out_ab - g["mc0_kat_output_ab"])) < 1e-4


def test_color_known_answers():
    # published sRGB(D65) -> CIELAB values
    kat = {(255, 255, 255): (100.0, 0.0, 0.0), (0, 0, 0): (0.0, 0.0, 0.0),
           (255, 0, 0): (53.24, 80.09, 67.20), (0, 255, 0): (87.73, -86.18, 83.18),
           (0, 0, 255): (32.30, 79.19, -107.86), (128, 128, 128): (53.59, 0.0, 0.0)}
    for rgb, lab in kat.items():
        got = color_ref.rgb2lab(np.array([[rgb]], dtype=np.uint8))[0, 0]
        assert np.max(np.abs(got - np.array(lab))) < 0.03, (rgb, got)
    rs = np.random.RandomState(0)
    rgb = rs.randint(0, 256, (64, 64, 3)).astype(np.uint8)
    back = (np.clip(color_ref.lab2rgb(color_ref.rgb2lab(rgb)), 0, 1) * 255 + 0.5).astype(np.uint8)
    assert np.array_equal(back, rgb)                      # round trip is exact after rounding


def test_product_color_matches_oracle():
    from interactive_deep_colorization_b200 import color
    rs = np.random.RandomState(1)
    rgb = rs.randint(0, 256, (50, 40, 3)).astype(np.uint8)
    assert np.max(np.abs(color.rgb2lab(rgb) - color_ref.rgb2lab(rgb))) < 1e-10
    lab = np.stack([rs.uniform(0, 100, (50, 40)), rs.uniform(-110, 110, (50, 40)), rs.uniform(-110, 110, (50, 40))], -1)
    assert np.max(np.abs(color.lab2rgb(lab) - color_ref.lab2rgb(lab))) < 1e-10
    assert np.array_equal(color.lab2rgb_transpose(lab[..., :1].transpose(2, 0, 1), lab[..., 1:].transpose(2, 0, 1)),
                          color_ref.lab2rgb_transpose(lab[..., :1].transpose(2, 0, 1), lab[..., 1:].transpose(2, 0, 1)))


def test_oracle_vs_reference_forward(synth_sd):
    """The oracle against the reference's own SIGGRAPHGenerator(dist=True).forward, as recorded by
    tests/golden/make_ref_forward_golden.py (same weights, one 64x64 synthetic image)."""
    g = util.golden("ref_forward_64.npz")
    (oreg, odist) = lhn_ref.lhn_forward(synth_sd, g["L"], g["ab"], g["mask"], 0.5, dist=True, ref_quirks=True)
    assert util.maxabs(oreg, g["reg"]) < 1e-3                     # values are O(1e3) here (quirk q1)
    y, x = g["dist_yx"]
    assert util.maxabs(lhn_ref.upsample4(odist)[0][:, y, x], g["dist_at_yx"]) < 1e-7
    # state_dict key compatibility of the drop-in module
    from interactive_deep_colorization_b200.model import SIGGRAPHGeneratorB200
    assert set(SIGGRAPHGeneratorB200(dist=True).state_dict().keys()) == set(g["state_dict_keys"].tolist())


def test_global_stats_encode_pinned_to_reference_nnenc():
    """Row f3: the nearest-bin encode + global average of oracle/caffe_spec.global_stats against the output of the
    reference's own NNEncode(NN=1, sigma=5) class (caffe_files/color_quantization.py:6-38, what NNEncLayer wraps,
    caffe_traininglayers.py:161-196), stored by tests/golden/make_glob_golden.py."""
    from oracle import caffe_spec
    g = util.golden("glob_nnenc.npz")
    pts = np.load(util.os.path.join(util.GOLDEN, "pts_in_hull.npy"))
    for name in ("mortar", "rand"):
        got = caffe_spec.global_stats(g[name + "_rgb"], pts)
        cells = g[name + "_bin"].size
        near_boundary = int((g[name + "_margin"] < 1e-3).sum())          # FP32 vs FP64 distance ties
        assert np.abs(got[:313] - g[name + "_hist"]).sum() * cells / 2 <= near_boundary + 1e-3   # float32 storage of the histogram
        assert abs(got[:313].sum() - 1.0) < 1e-6 and got[313] == 1.0 and got[315] == 1.0
