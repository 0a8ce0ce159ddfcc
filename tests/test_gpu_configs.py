"""GPU: the BASELINE.json configurations and call paths that round 1 left untested -- rank != 0 weight adoption,
config 4 at its real size (512^2 x 16 with the global-hints vector), config 5 (20 accumulating clicks on the
graph-replayed path), the chunked host pipeline with the dist head / global hints / FAST_FP16, the plan-time
options (PDL, CTA pairs on the split-K path, halo tiles) against each other, and the pinned sub-oracles."""
import numpy as np
import pytest
import torch

from oracle import caffe_spec, color_ref, synth
from tests import util

pytestmark = pytest.mark.gpu
TOL_AB = 1e-3


def _glob_sd(synth_sd):
    gsd = caffe_spec.synthetic_glob_state_dict()
    sd = dict(synth_sd)
    sd.update({k: torch.from_numpy(v) for k, v in gsd.items()})
    return sd, gsd


def test_rank_nonzero_weight_adoption_is_bit_identical(synth_sd):
    """Multi-GPU weight path (parallel.ShardedColorizer, ranks != 0): reserve_weights -> receive the packed arena ->
    adopt_weights.  Emulated on ONE GPU with a device-to-device copy instead of the NCCL broadcast; the adopting
    context must produce bit-identical outputs (regression head, dist head, RGB)."""
    from interactive_deep_colorization_b200.engine import LhnContext
    from interactive_deep_colorization_b200.parallel import _DevBlob
    L, ab, m = util.small_batch(3, 64, seed=21)
    a = util.make_ctx(synth_sd, 64, 64, max_n=3, dist=True)
    b = LhnContext(device=0, max_n=3, H=64, W=64, dist=True)
    b.reserve_weights()
    (pa, na), (pb, nb) = a.weights_arena(), b.weights_arena()
    assert na == nb and na > 60e6
    ta = torch.as_tensor(_DevBlob(pa, na), device="cuda:0")
    tb = torch.as_tensor(_DevBlob(pb, nb), device="cuda:0")
    tb.copy_(ta)
    torch.cuda.synchronize()
    b.adopt_weights()
    ra = a.forward_host(L, ab, m, 0.5, want_dist=True, want_rgb=True)
    rb = b.forward_host(L, ab, m, 0.5, want_dist=True, want_rgb=True)
    for k in ("ab", "dist", "rgb"):
        assert np.array_equal(ra[k], rb[k]), k
    da = a.forward_device(util.dev(L), util.dev(ab), util.dev(m), 0.5)["ab"]
    db = b.forward_device(util.dev(L), util.dev(ab), util.dev(m), 0.5)["ab"]
    torch.cuda.synchronize()
    assert torch.equal(da, db)
    a.close(); b.close()


def test_config4_512_batch16_global_hints(synth_sd):
    """BASELINE config 4 at its real size: 16 x 512x512 with a global-hints histogram vector per image, through the
    host-pointer call (chunked pipeline + glob) and the device-pointer call; every image against the oracle."""
    sd, gsd = _glob_sd(synth_sd)
    N = 16
    L, ab, m = synth.synthetic_batch(N, 512, seed=40, max_hints=10)
    glob_ab, sat = synth.synthetic_glob(N, seed=3)
    glob = np.ascontiguousarray(np.concatenate([glob_ab, sat], axis=1).astype(np.float32))
    gvec = caffe_spec.global_hints_vector(gsd, glob)
    ctx = util.make_ctx(sd, 512, 512, max_n=N, global_hints=True)
    r = ctx.forward_host(L, ab, m, 0.5, glob=glob, want_rgb=True)
    d = ctx.forward_device(util.dev(L), util.dev(ab), util.dev(m), 0.5, glob=util.dev(glob))["ab"]
    torch.cuda.synchronize()
    assert np.array_equal(r["ab"], d.cpu().numpy())                    # host pipeline == single-shot device path
    worst = 0.0
    for i0 in range(0, N, 4):                                          # oracle in slices of 4 (CPU memory)
        ref = util.oracle_forward(synth_sd, L[i0:i0 + 4], ab[i0:i0 + 4], m[i0:i0 + 4], 0.5, glob_add=gvec[i0:i0 + 4])
        worst = max(worst, util.maxabs(r["ab"][i0:i0 + 4], ref))
    print("config 4 (16 x 512^2 + global hints): max|d ab| = %.3e" % worst)
    assert worst <= TOL_AB
    # the vector matters, and it is per image
    r0 = ctx.forward_host(L[:2], ab[:2], m[:2], 0.5, glob=np.ascontiguousarray(glob[[1, 0]]))
    assert util.maxabs(r0["ab"], r["ab"][:2]) > 0.1
    ctx.close()


def test_config5_sequential_clicks_parity(synth_sd):
    """BASELINE config 5: 20 sequential put_point -> net_forward calls (one new hint per step, accumulating;
    DemoInteractiveColorization.ipynb:131-139,178,222) on ONE graph-replaying context with the dist head resident.
    Every click is compared with the oracle: raw ab, the clicked pixel's 529-bin distribution, RGB and the quantised
    output_ab."""
    g = util.golden("lhn_256.npz")
    L = g["img_l_mc"].astype(np.float32)[None]
    ctx = util.make_ctx(synth_sd, 256, 256, max_n=1, dist=True)
    ctx.set_dist_resident(True)
    rs = np.random.RandomState(5)
    a1, m1 = np.zeros((1, 2, 256, 256), np.float32), np.zeros((1, 1, 256, 256), np.float32)
    worst_ab = worst_d = 0.0
    for step in range(20):
        loc = rs.randint(8, 248, 2)
        synth.put_point(a1[0], m1[0], loc, 3, rs.uniform(-80, 80, 2))
        r = ctx.forward_host(L, a1, m1, 0.5, want_rgb=True, want_abq=True)
        pix = ctx.fetch_dist(0, int(loc[0]) // 4, int(loc[1]) // 4)
        ref_ab, ref_dist = util.oracle_forward(synth_sd, L, a1, m1, 0.5, dist=True)
        worst_ab = max(worst_ab, util.maxabs(r["ab"], ref_ab))
        worst_d = max(worst_d, util.maxabs(pix, ref_dist[0, :, int(loc[0]) // 4, int(loc[1]) // 4]))
        rgb_ref = color_ref.lab2rgb_transpose(L[0].astype(np.float64) + 50.0, r["ab"][0].astype(np.float64))
        assert np.array_equal(r["rgb"][0], rgb_ref)                    # post-process of OUR ab is bit-exact
        assert np.max(np.abs(r["abq"][0] - color_ref.rgb2lab_transpose(r["rgb"][0])[1:])) < 1e-9
    print("config 5: 20 clicks, worst max|d ab| = %.3e, worst |d dist| = %.3e" % (worst_ab, worst_d))
    assert worst_ab <= TOL_AB and worst_d < 1e-5
    assert ctx.last_launch_count() >= 28
    ctx.close()


@pytest.mark.parametrize("n", [9, 33])
def test_forward_host_large_batch_with_dist_and_glob(synth_sd, n):
    """idc_forward_host, batches >= 8 (chunked copy/compute overlap) with want_dist, want_rgb, the quantised ab and a
    global-hints vector: bit-identical to the single-shot device-pointer call."""
    sd, _ = _glob_sd(synth_sd)
    L, ab, m = synth.synthetic_batch(n, 64, seed=9, max_hints=4)
    glob_ab, sat = synth.synthetic_glob(n, seed=2)
    glob = np.ascontiguousarray(np.concatenate([glob_ab, sat], axis=1).astype(np.float32))
    ctx = util.make_ctx(sd, 64, 64, max_n=n, dist=True, global_hints=True)
    ref = ctx.forward_device(util.dev(L), util.dev(ab), util.dev(m), 0.5, glob=util.dev(glob), want_dist=True, want_rgb=True)
    ref = {k: v.cpu().numpy() for k, v in ref.items() if v is not None}
    for _ in range(2):
        r = ctx.forward_host(L, ab, m, 0.5, glob=glob, want_dist=True, want_rgb=True, want_abq=True)
        for k in ("ab", "dist", "rgb"):
            assert np.array_equal(r[k], ref[k]), k
    for i in (0, n - 1):
        assert np.max(np.abs(r["abq"][i] - color_ref.rgb2lab_transpose(r["rgb"][i])[1:])) < 1e-9
    ctx.close()


def test_fast_fp16_forward_host_large_batch(synth_sd):
    """ADVICE r1: FAST_FP16 has no lo planes; the chunked host pipeline launches conv1_1 with img0 > 0 and must not
    turn the null lo pointer into a bogus address."""
    n = 12
    L, ab, m = synth.synthetic_batch(n, 64, seed=13, max_hints=4)
    ctx = util.make_ctx(synth_sd, 64, 64, max_n=n, fast_fp16=True)
    ref = ctx.forward_device(util.dev(L), util.dev(ab), util.dev(m), 0.5)["ab"].cpu().numpy()
    r = ctx.forward_host(L, ab, m, 0.5, want_rgb=True)
    assert np.array_equal(r["ab"], ref)
    oracle = util.oracle_forward(synth_sd, L, ab, m, 0.5)
    assert util.maxabs(r["ab"], oracle) < 0.5                          # single-pass FP16: NOT the parity configuration
    ctx.close()


def test_plan_options_agree(synth_sd):
    """PDL on/off and the side-stream dist head on/off must be bit-identical (same kernels, same order of arithmetic); CTA pairs on the split-K path and
    the halo-tile operand change the summation order only: each variant within tolerance of the oracle and within
    3e-4 of each other.  256^2, batch 1 (the interactive plan: split-K everywhere) and batch 4."""
    g = util.golden("lhn_256.npz")
    L1 = g["img_l_mc"].astype(np.float32)[None]
    a1, m1 = synth.synthetic_hints(256, 5, 0)
    a1, m1 = a1[None].astype(np.float32), m1[None].astype(np.float32)
    ref = g["mc1_rand5_ab_raw"]
    outs = {}
    for name, opts in (("default", {}), ("no_pdl", {"pdl": 0}), ("no_side_dist", {"side_dist": 0}),
                       ("conv1_1_fp32", {"conv1_1_umma": 0}),
                       ("no_split_pairs", {"split_pairs": 0}), ("split_bn256", {"split_bn128": 0}),
                       ("no_halo", {"halo": 0}), ("halo_all", {"halo": 3})):
        ctx = util.make_ctx(synth_sd, 256, 256, max_n=1, dist=True, options=opts)
        r = ctx.forward_host(L1, a1, m1, 0.5, want_dist=True, want_rgb=True)
        r2 = ctx.forward_host(L1, a1, m1, 0.5, want_dist=True, want_rgb=True)      # graph replay
        assert np.array_equal(r["ab"], r2["ab"]) and np.array_equal(r["dist"], r2["dist"])
        err = util.maxabs(r["ab"][0], ref)
        print("options %-15s max|d ab| vs reference golden = %.3e" % (name, err))
        assert err <= TOL_AB, (name, err)
        outs[name] = r
        ctx.close()
    for k in ("no_pdl", "no_side_dist"):    # scheduling only: bit-identical
        assert np.array_equal(outs["default"]["ab"], outs[k]["ab"]), k
        assert np.array_equal(outs["default"]["dist"], outs[k]["dist"]), k
        assert np.array_equal(outs["default"]["rgb"], outs[k]["rgb"]), k
    for k in ("no_split_pairs", "split_bn256", "no_halo", "halo_all", "conv1_1_fp32"):
        assert util.maxabs(outs[k]["ab"], outs["default"]["ab"]) < 3e-4, k
    # batch 4 on a max_n = 4 context (halo + pairs plans differ from the batch-1 context)
    L, ab, m = synth.synthetic_batch(4, 256, seed=77, max_hints=6)
    oracle = util.oracle_forward(synth_sd, L, ab, m, 0.5)
    got = {}
    for name, opts in (("default", {}), ("no_pdl", {"pdl": 0}), ("no_halo", {"halo": 0})):
        ctx = util.make_ctx(synth_sd, 256, 256, max_n=4, options=opts)
        got[name] = ctx.forward_host(L, ab, m, 0.5)["ab"]
        assert util.maxabs(got[name], oracle) <= TOL_AB, name
        ctx.close()
    assert np.array_equal(got["default"], got["no_pdl"])


def test_stream_launched_pdl_chain_matches_graph(synth_sd):
    """The device-pointer call (plain stream launches with the PDL attribute, no graph) and the graph-replayed host
    call run the same kernels: bit-identical, also when forwards are issued back to back without a sync."""
    L, ab, m = synth.synthetic_batch(1, 256, seed=3, max_hints=6)
    ctx = util.make_ctx(synth_sd, 256, 256, max_n=1, dist=True)
    h = ctx.forward_host(L, ab, m, 0.5, want_dist=True, want_rgb=True)
    dL, dab, dm = util.dev(L), util.dev(ab), util.dev(m)
    outs = [ctx.forward_device(dL, dab, dm, 0.5, want_dist=True, want_rgb=True) for _ in range(1)]
    for _ in range(5):                                                 # back-to-back, no sync in between
        last = ctx.forward_device(dL, dab, dm, 0.5, want_dist=True, want_rgb=True)
    torch.cuda.synchronize()
    for r in (outs[0], last):
        assert np.array_equal(r["ab"].cpu().numpy(), h["ab"])
        assert np.array_equal(r["dist"].cpu().numpy(), h["dist"])
        assert np.array_equal(r["rgb"].cpu().numpy(), h["rgb"])
    ctx.close()


def test_wrapper_fused_quantised_ab_and_globdist_fullres(synth_sd):
    """net_forward is one C-ABI call: output_ab (the reference's quantised `_set_out_ab_`) comes back with the RGB.
    ADVICE r1: ColorizeImageB200GlobDist.get_img_fullres / get_img_gray_fullres (the histogram-transfer notebook calls
    them) must work although that class has no `self.net`."""
    from interactive_deep_colorization_b200 import colorize_image as CI
    g = util.golden("lhn_256.npz")
    cm = CI.ColorizeImageB200(Xd=256)
    cm.prep_net(state_dict=synth_sd)
    cm.set_image(g["img_rgb"])
    ab, m = np.zeros((2, 256, 256)), np.zeros((1, 256, 256))
    CI.put_point(ab, m, [135, 160], 3, [23, -69])
    rgb = cm.net_forward(ab, m)
    ref_q = color_ref.rgb2lab_transpose(rgb)
    assert cm.output_ab.dtype == np.float64 and cm.output_ab.shape == (2, 256, 256)
    assert np.max(np.abs(cm.output_ab - ref_q[1:])) < 1e-9
    assert np.max(np.abs(cm.output_lab - ref_q)) < 1e-9                # lazily derived, same values
    assert np.max(np.abs(cm.output_ab - g["mc0_kat_output_ab"] * 0 - ref_q[1:])) < 1e-9
    sd, _ = _glob_sd(synth_sd)
    cid = CI.ColorizeImageB200GlobDist(Xd=256)
    cid.prep_net(state_dict=sd)
    cid.set_image(g["img_rgb"])
    cid.net_forward(ab, m)
    full = cid.get_img_fullres()
    assert full.shape == (256, 256, 3) and full.dtype == np.uint8
    d = np.abs(full.astype(int) - color_ref.lab2rgb_transpose(cid.img_l_fullres, cid.output_ab).astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 1e-3
    assert cid.get_img_gray_fullres().shape == (256, 256, 3)


def test_get_ab_reccs_sampled_reproduces_reference_answer(synth_sd):
    """Row a16: method='sampled' is the reference's own procedure (np.random + sklearn KMeans on 25 000 inverse-CDF
    samples, data/colorize_image.py:322-354).  With np.random.seed(0) it must reproduce the reference's stored answer
    for the same image / hints (tests/golden/lhn_dist_256.npz: reccs_128_128_K9, generated by the unmodified
    reference with the same seed) up to the few samples that a 1e-6 difference in the pmf can move."""
    from interactive_deep_colorization_b200 import colorize_image as CI
    g, gd = util.golden("lhn_256.npz"), util.golden("lhn_dist_256.npz")
    cd = CI.ColorizeImageB200Dist(Xd=256, maskcent=True)
    cd.prep_net(state_dict=synth_sd)
    cd.set_image(g["img_rgb"])
    a5, m5 = synth.synthetic_hints(256, 5, 0)
    cd.net_forward(a5, m5)
    np.random.seed(0)
    got = cd.get_ab_reccs(128, 128, K=9, N=25000, method='sampled')
    ref = gd["reccs_128_128_K9"]
    err = np.abs(got - ref).max()
    print("get_ab_reccs(method='sampled', seed 0) vs the reference's stored answer: max|d| = %.4f ab units" % err)
    # measured 0.32: a handful of the 25 000 samples sit within the 1e-6 pmf difference of a CDF edge and land in the
    # neighbouring bin (10 ab units away); a cluster holds ~2 800 samples, so its centre moves by ~10 * k / 2800
    assert got.shape == (9, 2) and err < 0.6


def test_global_stats_kernel_vs_reference_nnenc():
    """Row f3 pinned: global_stats_kernel's histogram against the reference's own NNEncode(NN=1) output (fixture from
    tests/golden/make_glob_golden.py); only cells within 1e-3 ab units of a bin boundary may land in the other bin."""
    from interactive_deep_colorization_b200 import prepost
    g = util.golden("glob_nnenc.npz")
    for name in ("mortar", "rand"):
        got = prepost.global_stats_gpu(g[name + "_rgb"])
        cells = g[name + "_bin"].size
        near = int((g[name + "_margin"] < 1e-3).sum())
        moved = np.abs(got[:313].astype(np.float64) - g[name + "_hist"]).sum() * cells / 2
        print("global_stats %s: %.1f of %d cells differ from NNEncode (%d within 1e-3 of a boundary)" % (name, moved, cells, near))
        assert moved <= near + 0.01


def _caffe_scaled(sd):
    """A synthetic 'Caffe-scaled' weight set: conv1_1 expects raw L-50 / ab / mask*110 (SURVEY q4)."""
    out = dict(sd)
    s = torch.tensor([100.0, 110.0, 110.0, 110.0]).reshape(1, 4, 1, 1)
    out["model1.0.weight"] = (sd["model1.0.weight"].double() / s.double()).float()
    return out


def test_caffe_named_wrappers(synth_sd):
    """Rows a14 / wrapper surface: ColorizeImageB200Caffe / ...CaffeDist / ...CaffeGlobDist keep the reference's Caffe
    class semantics (data/colorize_image.py:375-561): mask x 110, tanh x 100, 313-bin dist_ab, get_ab_reccs on
    pts_in_hull.  Spec-only oracle (oracle/caffe_spec.py), parity unpinned."""
    from interactive_deep_colorization_b200 import colorize_image as CI
    g = util.golden("lhn_256.npz")
    img = np.ascontiguousarray(g["img_rgb"][::4, ::4])                 # 64 x 64
    ab, m = np.zeros((2, 64, 64)), np.zeros((1, 64, 64))
    CI.put_point(ab, m, [30, 40], 3, [23, -69])
    cc = CI.ColorizeImageB200Caffe(Xd=64)
    assert cc.mask_mult == 110. and cc.pts_in_hull.shape == (313, 2)
    assert cc.net_forward(ab, m) == -1                                 # "I need to have an image!"
    cc.prep_net(0, state_dict=_caffe_scaled(synth_sd))
    cc.set_image(img)
    rgb = cc.net_forward(ab, m)
    assert np.array_equal(cc.input_mask_mult, m * 110.)                # the reference attribute keeps the x110
    L = cc.img_l_mc.astype(np.float32)[None]
    ref = util.oracle_forward(synth_sd, L, ab[None].astype(np.float32), m[None].astype(np.float32), 0.0)[0] * (100.0 / 110.0)
    assert util.maxabs(cc.output_ab_raw, ref) <= TOL_AB
    assert np.array_equal(rgb, color_ref.lab2rgb_transpose(cc.img_l, cc.output_ab_raw.astype(np.float64)))
    assert np.max(np.abs(cc.output_ab - color_ref.rgb2lab_transpose(rgb)[1:])) < 1e-9
    # global-hints variant: zero vector == plain call; a histogram changes the result
    sdg, gsd = _glob_sd(synth_sd)
    cg = CI.ColorizeImageB200CaffeGlobDist(Xd=64)
    cg.prep_net(0, state_dict=_caffe_scaled(sdg))
    cg.set_image(img)
    cg.net_forward(ab, m)
    gv0 = caffe_spec.global_hints_vector(gsd, np.zeros((1, 316), np.float32))
    ref0 = util.oracle_forward(synth_sd, L, ab[None].astype(np.float32), m[None].astype(np.float32), 0.0, glob_add=gv0)[0] * (100.0 / 110.0)
    assert util.maxabs(cg.output_ab_raw, ref0) <= TOL_AB
    hist = cg.get_global_histogram(np.random.RandomState(4).randint(0, 256, (120, 160, 3)).astype(np.uint8))
    raw0 = cg.output_ab_raw.copy()
    cg.net_forward(ab, m, hist)
    assert util.maxabs(cg.output_ab_raw, raw0) > 0.05
    # 313-bin distribution model
    pts = np.load(util.os.path.join(util.GOLDEN, "pts_in_hull.npy"))
    csd = caffe_spec.synthetic_caffe313_state_dict(pts_in_hull=pts)
    sd313 = _caffe_scaled(synth_sd)
    sd313.update({k: torch.from_numpy(v) for k, v in csd.items() if k != "caffe.pts_in_hull"})
    cd = CI.ColorizeImageB200CaffeDist(Xd=64)
    assert np.array_equal(cd.pts_grid[cd.in_hull], cd.pts_in_hull) and cd.in_hull.sum() == 313
    cd.prep_net(0, state_dict=sd313, S=.2)
    cd.set_image(img)
    out = cd.net_forward(ab, m)
    assert out.shape == (64, 64, 3) and out.dtype == np.uint8
    _, inter = util.oracle_forward(synth_sd, L, ab[None].astype(np.float32), m[None].astype(np.float32), 0.0, intermediates=True)
    with torch.no_grad():
        pred64, distS64 = caffe_spec.caffe313_head(csd, inter, dtype=torch.float64)
    assert util.maxabs(cd.output_ab_raw, pred64[0]) <= 2e-3            # spec-only head, see test_caffe313_head
    assert np.array_equal(out, color_ref.lab2rgb_transpose(cd.img_l, cd.output_ab_raw.astype(np.float64)))
    for (y, x) in ((0, 0), (17, 33), (63, 63)):
        assert util.maxabs(np.asarray(cd.dist_ab[:, y, x]), distS64[0, :, y, x]) < 1e-5
    full = cd.dist_ab_full
    assert full.shape == (529, 64, 64) and abs(full[:, 5, 6].sum() - 1.0) < 1e-4 and full[~cd.in_hull].max() == 0.0
    assert cd.dist_ab_grid.shape == (23, 23, 64, 64)
    rec, conf = cd.get_ab_reccs(17, 33, K=6, return_conf=True)
    assert rec.shape == (6, 2) and abs(conf.sum() - 1.0) < 1e-4 and np.all(np.diff(conf) <= 1e-9)
    np.random.seed(1)
    rec_s = cd.get_ab_reccs(17, 33, K=6, method='sampled')
    assert rec_s.shape == (6, 2) and np.abs(rec_s).max() <= 110


@pytest.mark.parametrize("sh,sw,dh,dw", [(507, 600, 256, 256), (864, 1296, 256, 256), (512, 512, 256, 256),
                                         (100, 80, 256, 256), (64, 96, 128, 192), (257, 511, 128, 128), (300, 300, 64, 64)])
def test_resize_u8_linear_is_bit_identical_to_cv2(sh, sw, dh, dw):
    """Row f1: `cv2.resize(im, (Xd, Xd))` of load_image (data/colorize_image.py:52-66) restated for the GPU.  OpenCV's
    8-bit INTER_LINEAR is fixed-point; the kernel must reproduce it bit for bit (down- and up-scaling, the exact-2x
    area shortcut, border rows / columns)."""
    import cv2
    from interactive_deep_colorization_b200 import prepost
    src = np.random.RandomState(sh * 7 + sw).randint(0, 256, (sh, sw, 3)).astype(np.uint8)
    assert np.array_equal(prepost.resize_u8_linear_gpu(src, dh, dw), cv2.resize(src, (dw, dh)))


def test_load_image_on_gpu_matches_host_path(synth_sd, tmp_path):
    """Row f1: ColorizeImageB200.load_image with a net set runs rgb2lab (full resolution + net size) and the resize on
    the GPU; every attribute the reference sets must equal the host (numpy / cv2) path of the same class."""
    import cv2
    from scipy.ndimage import zoom
    from interactive_deep_colorization_b200 import colorize_image as CI
    from interactive_deep_colorization_b200.prepost import DeviceLab
    rgb = np.random.RandomState(11).randint(0, 256, (507, 600, 3)).astype(np.uint8)
    path = str(tmp_path / "im.png")
    cv2.imwrite(path, np.ascontiguousarray(rgb[:, :, ::-1]))
    gpu = CI.ColorizeImageB200(Xd=256)
    gpu.prep_net(state_dict=synth_sd)
    gpu.load_image(path)
    host = CI.ColorizeImageB200(Xd=256, gpu_prepost=False)
    host.load_image(path)                                             # no net set, gpu_prepost off: cv2 + numpy
    assert isinstance(gpu.img_lab_fullres, DeviceLab) and gpu.img_l_fullres.shape == (1, 507, 600)
    assert np.array_equal(gpu.img_rgb, host.img_rgb) and np.array_equal(gpu.img_rgb_fullres, host.img_rgb_fullres)
    for name in ("img_lab", "img_l", "img_ab", "img_l_mc", "img_lab_mc", "img_lab_fullres", "img_l_fullres", "img_ab_fullres"):
        a, b = np.asarray(getattr(gpu, name)), np.asarray(getattr(host, name))
        assert a.shape == b.shape and np.max(np.abs(a - b)) < 1e-10, name
    ab, m = np.zeros((2, 256, 256)), np.zeros((1, 256, 256))
    CI.put_point(ab, m, [135, 160], 3, [23, -69])
    gpu.net_forward(ab, m)
    full = gpu.get_img_fullres()                                      # L stays on the device for the full-res render
    ref = color_ref.lab2rgb_transpose(np.asarray(host.img_l_fullres),
                                      zoom(gpu.output_ab, (1, 507 / 256., 600 / 256.), order=1))
    d = np.abs(full.astype(int) - ref.astype(int))
    assert full.shape == (507, 600, 3) and d.max() <= 1 and (d > 0).mean() < 1e-3
    assert gpu.get_img_gray_fullres().shape == (507, 600, 3)


def test_display_step_cubic_resize_lab2rgb():
    """Row f1: the GUI's display step (ui/gui_draw.py:280-283) -- cv2 INTER_CUBIC resize of the float64 ab planes to the
    window size + lab2rgb -- as one kernel, against cv2 + the colour oracle."""
    import cv2
    from interactive_deep_colorization_b200 import prepost
    rs = np.random.RandomState(8)
    ab = rs.uniform(-60, 60, (2, 256, 256))
    for (H, W) in ((512, 512), (384, 600), (200, 256)):
        l_win = rs.uniform(5, 95, (H, W))
        got = prepost.display_rgb_gpu(ab, l_win)
        ab_win = cv2.resize(ab.transpose((1, 2, 0)), (W, H), interpolation=cv2.INTER_CUBIC)
        pred_lab = np.concatenate((l_win[..., np.newaxis], ab_win), axis=2)
        ref = (np.clip(color_ref.lab2rgb(pred_lab), 0, 1) * 255).astype('uint8')
        d = np.abs(got.astype(int) - ref.astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, (H, W, d.max(), (d > 0).mean())
