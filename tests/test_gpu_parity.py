"""GPU parity tests (-m gpu): every CUDA entry point, called through the C ABI via the host API,
against (a) the CPU oracle, (b) the committed golden vectors and (c) the outputs of the reference's
own CUDA kernels (compiled for sm_100a) on the same inputs, stored in tests/golden/reference_kernels.npz
by tests/golden/make_reference_kernels.py.
Tolerances: bit-exact for NMS indices / panoptic label maps / FPN levels; fp32 outputs within 1e-3
(BASELINE.json north_star), in practice ~1e-5 for the fp32 tiles."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-3


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kernels.npz"))


REF_SAMPLE = 2048


def ref_sample(n):
    """Fixed subset of a flattened output of n elements: large reference-kernel outputs are stored at these indices."""
    if n <= REF_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(n).choice(n, REF_SAMPLE, replace=False))


def t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def rand_rois(rng, n, B, extent, smin, smax):
    c = rng.uniform(0, extent, (n, 2)); s = np.exp(rng.uniform(np.log(smin), np.log(smax), (n, 2)))
    r = np.concatenate([rng.integers(0, B, (n, 1)), np.clip(c - s / 2, 0, extent - 1),
                        np.clip(c + s / 2, 0, extent - 1)], 1)
    return r.astype(np.float32)


# ----------------------------------------------------------------------------------------------
def test_native_library_is_loaded(dev):
    from upsnet_b200 import _lib
    n_sm = __import__("ctypes").c_int(0)
    assert _lib.lib().upsnet_version(__import__("ctypes").byref(n_sm)) == 100
    assert n_sm.value > 0
    maps = open("/proc/self/maps").read()
    assert "libupsnet_b200.so" in maps


# ------------------------------- ROIAlign -----------------------------------------------------
def test_roi_align_golden(dev, golden_ops, ref):
    import upsnet_b200 as U
    g = golden_ops
    out = U.roi_align(t(g["ra_feat"], dev), t(g["ra_rois"], dev), 7, 7, 0.25).cpu().numpy()
    assert np.abs(out - g["ra_out"]).max() < 1e-4
    assert np.abs(out - ref["roi_align_golden"]).max() < 1e-4


def roi_align_config1_case():
    torch.manual_seed(0)
    rng = np.random.default_rng(0)
    return torch.randn(1, 256, 256, 256), rand_rois(rng, 32, 1, 1024, 16, 512)


@pytest.mark.parametrize("ph", [7, 14])
def test_roi_align_config1_nchw_and_nhwc(dev, ph, ref):
    """BASELINE config #1: 1x256x256x256 feature map, 32 boxes, scale 1/4, sampling_ratio 2."""
    import upsnet_b200 as U
    feat, rois = roi_align_config1_case()
    want = O.roi_align(feat.numpy(), rois, ph, ph, 0.25)
    f = feat.to(dev); r = t(rois, dev)
    got = U.RoIAlign(ph, ph, 0.25)(f, r).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4  # FMA contraction moves sample coords by 1 ulp
    got_nhwc = U.roi_align(f.permute(0, 2, 3, 1).contiguous(), r, ph, ph, 0.25, layout="nhwc")
    assert np.abs(got_nhwc.permute(0, 3, 1, 2).cpu().numpy() - want).max() < 1e-4
    assert np.abs(ref["roi_align_config1_ph%d" % ph] - got.reshape(-1)[ref_sample(got.size)]).max() < 1e-4


def test_roi_align_edge_cases(dev):
    import upsnet_b200 as U
    f = torch.randn(2, 5, 9, 11)
    rois = np.array([[0, -50, -50, -10, -10], [1, 0, 0, 0, 0], [0, 30, 20, 500, 400], [1, 3.3, 2.2, 17.9, 30.1]],
                    np.float32)
    want = O.roi_align(f.numpy(), rois, 3, 5, 0.5)
    got = U.roi_align(f.to(dev), t(rois, dev), 3, 5, 0.5).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4  # FMA contraction moves sample coords by 1 ulp
    got2 = U.roi_align(f.to(dev).permute(0, 2, 3, 1).contiguous(), t(rois, dev), 3, 5, 0.5, layout="nhwc")
    assert np.abs(got2.permute(0, 3, 1, 2).cpu().numpy() - want).max() < 1e-4
    empty = U.roi_align(f.to(dev), torch.zeros(0, 5, device=dev), 3, 5, 0.5)
    assert empty.shape == (0, 5, 3, 5)


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_fpn_roi_align_matches_reference_bucketing(dev, layout):
    import upsnet_b200 as U
    rng = np.random.default_rng(4)
    C = 32
    feats = [torch.randn(1, C, 128 >> l, 192 >> l) for l in range(4)]
    rois = rand_rois(rng, 300, 1, 512, 8, 700)
    rois[:, 3] = np.minimum(rois[:, 3], 767); rois[:, 1] *= 1.4
    rois[:, 3] = np.maximum(rois[:, 3], rois[:, 1])
    want = O.fpn_roi_align([f.numpy() for f in feats], rois, 7, 7)
    fd = [f.to(dev) for f in feats]
    if layout == "nhwc":
        fd = [f.permute(0, 2, 3, 1).contiguous() for f in fd]
    got, lv = U.fpn_roi_align(fd, t(rois, dev), 7, 7, [1 / 4., 1 / 8., 1 / 16., 1 / 32.], layout=layout,
                              return_levels=True)
    if layout == "nhwc":
        got = got.permute(0, 3, 1, 2)
    assert np.array_equal(lv.cpu().numpy(), O.fpn_level_numpy(rois))  # bit-exact level assignment
    assert len(set(lv.cpu().numpy().tolist())) == 4
    assert np.abs(got.cpu().numpy() - want).max() < 1e-4
    if layout == "nchw":
        mod = U.FPNRoIAlign(7, 7, [1 / 4., 1 / 8., 1 / 16., 1 / 32.])
        assert np.abs(mod(fd, t(rois, dev)).cpu().numpy() - want).max() < 1e-4


# ------------------------------- NMS ----------------------------------------------------------
def test_nms_golden_reference_py_cpu_nms(dev, golden_ref, ref):
    import upsnet_b200 as U
    g = golden_ref
    for i in range(int(g["nms_cases"])):
        d = g["nms%d_dets" % i]; thr = float(g["nms%d_thresh" % i])
        keep = U.gpu_nms_wrapper(thr, 0)(d)
        assert keep == g["nms%d_keep" % i].tolist(), "case %d" % i
        assert ref["nms_golden_%d" % i].tolist() == keep


def nms_dense_cases():
    rng = np.random.default_rng(11)
    for n, extent in [(1, 50), (64, 80), (65, 80), (129, 100), (1000, 250), (4097, 600), (8000, 1200)]:
        c = rng.uniform(0, extent, (n, 2)); s = np.exp(rng.uniform(np.log(16), np.log(128), (n, 2)))
        scores = (rng.permutation(n) + 1.0) / (n + 1)
        yield n, np.concatenate([c - s / 2, c + s / 2, scores[:, None]], 1).astype(np.float32)


def test_nms_dense_random_bit_exact(dev, ref):
    import upsnet_b200 as U
    for n, d in nms_dense_cases():
        for thr in (0.3, 0.5, 0.7):
            want = O.nms(d, thr)
            got = U.nms(t(d[:, :4], dev), t(d[:, 4], dev), thr).cpu().tolist()
            assert got == want, (n, thr)
            assert len(want) < n or n == 1
        if n <= 4097:
            assert ref["nms_dense_%d" % n].tolist() == O.nms(d, 0.5)


def test_nms_segmented_levels_one_launch(dev):
    """Five independent problems (the five RPN levels) in one launch pair, no host round trip."""
    import upsnet_b200 as U
    rng = np.random.default_rng(12)
    lens = [1000, 1000, 777, 64, 0]
    segs, wants = [], []
    for n in lens:
        c = rng.uniform(0, 300, (n, 2)); s = np.exp(rng.uniform(np.log(16), np.log(128), (n, 2)))
        sc = np.sort((rng.permutation(n) + 1.0) / (n + 1))[::-1]
        d = np.concatenate([c - s / 2, c + s / 2, sc[:, None]], 1).astype(np.float32)
        segs.append(d); wants.append(O.nms(d, 0.7))
    boxes = t(np.concatenate(segs)[:, :4], dev)
    off = torch.tensor(np.concatenate([[0], np.cumsum(lens)]), dtype=torch.int32, device=dev)
    keep, cnt = U.nms_segmented(boxes, off, 1000, 0.7)
    for s_, w in enumerate(wants):
        assert keep[s_, :int(cnt[s_])].cpu().tolist() == w


def test_nms_host_dropin_entry(dev):
    """upsnet_nms_host has the reference `_nms` signature (host pointers, sorted boxes)."""
    import ctypes as C
    from upsnet_b200 import _lib
    rng = np.random.default_rng(13)
    n = 500
    c = rng.uniform(0, 200, (n, 2)); s = np.exp(rng.uniform(np.log(16), np.log(100), (n, 2)))
    sc = np.sort((rng.permutation(n) + 1.0) / (n + 1))[::-1]
    d = np.ascontiguousarray(np.concatenate([c - s / 2, c + s / 2, sc[:, None]], 1).astype(np.float32))
    keep = np.zeros(n, np.int32); num = np.zeros(1, np.int32)
    rc = _lib.lib().upsnet_nms_host(keep.ctypes.data_as(C.c_void_p), num.ctypes.data_as(C.c_void_p),
                                    d.ctypes.data_as(C.c_void_p), n, 5, 0.5, 0)
    assert rc == 0 and keep[:num[0]].tolist() == O.nms(d, 0.5)


# ------------------------------- DCN / conv ---------------------------------------------------
def test_dcn_golden(dev, golden_ops, ref):
    import upsnet_b200 as U
    g = golden_ops
    x, w, b = t(g["dcn_x"], dev), t(g["dcn_w"], dev), t(g["dcn_b"], dev)
    y = U.deform_conv(x, t(g["dcn_off"], dev), w, b, padding=1, deformable_groups=2).cpu().numpy()
    assert np.abs(y - g["dcn_y"]).max() < 1e-4
    m = U.ModulatedDeformConv(8, 12, 3, padding=1).to(dev)
    m.weight.data.copy_(w); m.bias.data.copy_(b)
    y2 = m(x, t(g["dcn2_om"], dev)).detach().cpu().numpy()      # module call = autograd path (parameters require grad), like the reference
    assert np.abs(y2 - g["dcn2_y"]).max() < 1e-4
    assert np.abs(y - ref["dcn_golden"]).max() < 1e-4


DCN_CFGS = [
    dict(N=1, Cin=256, Cout=128, H=32, W=48, stride=1, pad=1, dil=1, dg=1),   # semantic-head layer shape (a12)
    dict(N=2, Cin=64, Cout=96, H=25, W=42, stride=1, pad=1, dil=1, dg=1),     # ragged spatial size (B: 25x42)
    dict(N=2, Cin=32, Cout=40, H=17, W=19, stride=2, pad=1, dil=1, dg=2),
    dict(N=1, Cin=16, Cout=16, H=20, W=20, stride=1, pad=2, dil=2, dg=4),
]


def dcn_case(cfg, modulated):
    """(x, offset, weight, bias, mask or None) of one test_dcn_vs_oracle case."""
    rng = np.random.default_rng(21)
    N, Cin, Cout, H, W = cfg["N"], cfg["Cin"], cfg["Cout"], cfg["H"], cfg["W"]
    Ho = O.conv_out(H, cfg["pad"], cfg["dil"], 3, cfg["stride"]); Wo = O.conv_out(W, cfg["pad"], cfg["dil"], 3, cfg["stride"])
    x = rng.standard_normal((N, Cin, H, W)).astype(np.float32)
    w = (rng.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9)).astype(np.float32)
    b = rng.standard_normal(Cout).astype(np.float32)
    off = (rng.standard_normal((N, 18 * cfg["dg"], Ho, Wo)) * 2.5).astype(np.float32)
    mask = (rng.uniform(0, 2, (N, 9 * cfg["dg"], Ho, Wo))).astype(np.float32) if modulated else None
    return x, off, w, b, mask


@pytest.mark.parametrize("cfg", DCN_CFGS)
@pytest.mark.parametrize("modulated", [False, True])
def test_dcn_vs_oracle(dev, cfg, modulated, ref):
    import upsnet_b200 as U
    x, off, w, b, mask = dcn_case(cfg, modulated)
    want = O.deform_conv(x, off, w, b, mask, cfg["stride"], cfg["pad"], cfg["dil"], cfg["dg"])
    got = U.deform_conv(t(x, dev), t(off, dev), t(w, dev), t(b, dev), cfg["stride"], cfg["pad"], cfg["dil"],
                        cfg["dg"], mask=None if mask is None else t(mask, dev)).cpu().numpy()
    assert np.abs(got - want).max() < TOL, np.abs(got - want).max()
    assert np.abs(got - want).max() < 1e-4  # fp32 tiles are far inside the 1e-3 contract
    r = ref["dcn_cfg%d_mod%d" % (DCN_CFGS.index(cfg), modulated)]
    assert np.abs(got.reshape(-1)[ref_sample(got.size)] - r).max() < TOL


def test_deform_conv_with_offset_module_and_state_dict_names(dev):
    import upsnet_b200 as U
    m = U.DeformConvWithOffset(16, 24, 3, padding=1).to(dev)
    assert set(m.state_dict().keys()) == {"conv_offset.weight", "conv_offset.bias", "conv.weight", "conv.bias"}
    assert m.conv.weight.shape == (24, 16, 3, 3)
    torch.manual_seed(3)
    m.conv_offset.weight.data.normal_(0, 0.3)
    x = torch.randn(1, 16, 12, 14, device=dev)
    y = m(x).detach().cpu().numpy()      # module call = autograd path (parameters require grad), like the reference
    off = O.conv2d(x.cpu().numpy(), m.conv_offset.weight.detach().cpu().numpy(), m.conv_offset.bias.detach().cpu().numpy(), pad=1)
    want = O.deform_conv(x.cpu().numpy(), off, m.conv.weight.detach().cpu().numpy(), m.conv.bias.detach().cpu().numpy(), pad=1)
    assert np.abs(y - want).max() < 1e-4


@pytest.mark.parametrize("cfg", [
    dict(N=1, Cin=64, Cout=64, H=24, W=40, k=3, stride=1, pad=1, dil=1),
    dict(N=2, Cin=256, Cout=128, H=16, W=20, k=1, stride=2, pad=0, dil=1),    # Caffe-style strided 1x1
    dict(N=1, Cin=3, Cout=64, H=64, W=96, k=7, stride=2, pad=3, dil=1),       # stem (a1)
    dict(N=3, Cin=32, Cout=70, H=14, W=14, k=3, stride=1, pad=2, dil=2),
    dict(N=37, Cin=392, Cout=100, H=1, W=1, k=1, stride=1, pad=0, dil=1),     # fully connected (a9)
])
def test_conv2d_vs_oracle_with_epilogue(dev, cfg):
    import upsnet_b200 as U
    rng = np.random.default_rng(31)
    x = rng.standard_normal((cfg["N"], cfg["Cin"], cfg["H"], cfg["W"])).astype(np.float32)
    w = (rng.standard_normal((cfg["Cout"], cfg["Cin"], cfg["k"], cfg["k"])) / np.sqrt(cfg["Cin"] * cfg["k"] ** 2)).astype(np.float32)
    b = rng.standard_normal(cfg["Cout"]).astype(np.float32)
    want = O.conv2d(x, w, b, cfg["stride"], cfg["pad"], cfg["dil"])
    res = rng.standard_normal(want.shape).astype(np.float32)
    got = U.conv2d(t(x, dev), t(w, dev), t(b, dev), cfg["stride"], cfg["pad"], cfg["dil"]).cpu().numpy()
    assert np.abs(got - want).max() < 1e-4
    got2 = U.conv2d(t(x, dev), t(w, dev), t(b, dev), cfg["stride"], cfg["pad"], cfg["dil"], residual=t(res, dev),
                    relu=True).cpu().numpy()
    assert np.abs(got2 - np.maximum(want + res, 0)).max() < 1e-4


# ------------------------------- panoptic head -------------------------------------------------
def pan_case(n, H, W, seed, S=19, nthing=8, smax=None):
    rng = np.random.default_rng(seed)
    fcn = (rng.standard_normal((S, H, W)) * 3).astype(np.float32)
    c = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n)], 1)
    s = np.exp(rng.uniform(np.log(8), np.log(smax or min(H, W) / 2), (n, 2)))
    b = np.concatenate([c - s / 2, c + s / 2], 1).astype(np.float32)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, W - 1); b[:, 1::2] = np.clip(b[:, 1::2], 0, H - 1)
    prob = (0.6 + 0.4 * (rng.permutation(n) + 1) / (n + 1)).astype(np.float32)
    ml = (rng.standard_normal((n, 28, 28)) * 2 + 0.5).astype(np.float32)
    cls = rng.integers(1, nthing + 1, n).astype(np.int64)
    return fcn, b, prob, ml, cls


def run_pan(dev, fcn, b, prob, ml, cls, num_stuff=11, want_sem=False):
    import upsnet_b200 as U
    return U.panoptic_fuse(t(fcn[None], dev), t(b, dev), t(prob, dev), t(ml[:, None], dev), t(cls, dev), num_stuff,
                           want_sem=want_sem)


def test_panoptic_golden_bit_exact(dev, golden_ops):
    g = golden_ops
    keep, labels = run_pan(dev, g["pan_fcn"], g["pan_boxes"], g["pan_prob"], g["pan_ml"], g["pan_cls"])
    assert keep.cpu().tolist() == g["pan_keep"].tolist()
    assert np.array_equal(labels[0].cpu().numpy(), g["pan_labels"])


@pytest.mark.parametrize("n,H,W", [(1, 40, 56), (7, 64, 100), (40, 128, 160), (100, 256, 512), (300, 250, 333)])
def test_panoptic_vs_oracle_bit_exact(dev, n, H, W):
    fcn, b, prob, ml, cls = pan_case(n, H, W, seed=100 + n)
    want_keep, want_labels, want_sem = O.panoptic_head(fcn, b, prob, ml, cls, 11, want_sem=True)
    keep, labels, sem = run_pan(dev, fcn, b, prob, ml, cls, want_sem=True)
    assert keep.cpu().tolist() == want_keep.tolist()
    assert np.array_equal(labels[0].cpu().numpy(), want_labels)
    assert np.array_equal(sem[0].cpu().numpy(), want_sem)


def test_panoptic_edge_cases(dev):
    fcn, b, prob, ml, cls = pan_case(3, 40, 56, seed=5)
    for mlv, bv, cv in [(-np.abs(ml) - 1, b, cls),                                             # nothing kept
                        (np.stack([ml[0], ml[0], ml[1]]), np.stack([b[0], b[0], b[1]]), np.array([3, 3, 5])),
                        (ml[:1], np.zeros((1, 4), np.float32), np.array([0]))]:                   # MaskROI dummy
        pv = prob[:len(cv)]
        wk, wl = O.panoptic_head(fcn, bv, pv, mlv, cv.astype(np.int64), 11)
        k, l = run_pan(dev, fcn, bv, pv, mlv, cv.astype(np.int64))
        assert k.cpu().tolist() == wk.tolist() and np.array_equal(l[0].cpu().numpy(), wl)


def test_panoptic_coco_shape_classes(dev):
    """133 seg classes / 80 things (config B): exercises the generic channel loops."""
    fcn, b, prob, ml, cls = pan_case(60, 100, 168, seed=7, S=133, nthing=80)
    wk, wl = O.panoptic_head(fcn, b, prob, ml, cls, 53)
    k, l = run_pan(dev, fcn, b, prob, ml, cls, num_stuff=53)
    assert k.cpu().tolist() == wk.tolist() and np.array_equal(l[0].cpu().numpy(), wl)


def test_panoptic_full_size_properties_and_oracle(dev):
    """BASELINE full size (1024x2048, 100 instances): bit-exact against the oracle (the fused C oracle
    finishes in ~1 s) plus size-independent properties: labels in range, idempotent re-run, void/stuff
    pixels agree with a pure semantic argmax wherever no instance window covers them."""
    H, W, n = 1024, 2048, 100
    fcn, b, prob, ml, cls = pan_case(n, H, W, seed=42, smax=512)
    wk, wl = O.panoptic_head(fcn, b, prob, ml, cls, 11)
    k, l = run_pan(dev, fcn, b, prob, ml, cls)
    l = l[0].cpu().numpy()
    assert k.cpu().tolist() == wk.tolist()
    assert np.array_equal(l, wl)
    k2, l2 = run_pan(dev, fcn, b, prob, ml, cls)
    assert np.array_equal(l2[0].cpu().numpy(), l) and k2.cpu().tolist() == k.cpu().tolist()
    kk = len(wk)
    assert ((l < 11 + kk) | (l == 255)).all() and l.min() >= 0


def test_panoptic_head_module(dev):
    import upsnet_b200 as U
    fcn, b, prob, ml, cls = pan_case(12, 64, 96, seed=77)
    head = U.PanopticHead(num_seg_classes=19, num_classes=9)
    rois5 = np.concatenate([np.zeros((12, 1), np.float32), b], 1)
    out = head(t(fcn[None], dev), t(rois5, dev), t(prob, dev), t(ml[:, None], dev), t(cls, dev), want_sem=True)
    wk, wl, ws = O.panoptic_head(fcn, b, prob, ml, cls, 11, want_sem=True)
    assert out["keep_inds"].cpu().tolist() == wk.tolist()
    assert np.array_equal(out["panoptic_outputs"][0].cpu().numpy(), wl)
    assert np.array_equal(out["fcn_outputs"][0].cpu().numpy(), ws)


# ------------------------------- whole engine ---------------------------------------------------
def test_engine_forward_matches_cpu_path(dev):
    """resnet_upsnet on the GPU (C ABI kernels) vs the same host logic on the CPU path (torch-CPU convs +
    oracle ops), same weights.  Dense tensors within 1e-3 of their scale.  Discrete stages are checked
    where they are well defined: the random-init heads emit near-tied scores, so top-k / NMS orderings may
    legitimately differ between two fp32 implementations; the panoptic head is therefore verified
    bit-exactly by feeding the oracle the GPU engine's OWN head inputs."""
    from oracle.cpu_model import cpu_ops
    from upsnet_b200.model import UPSNetConfig
    from upsnet_b200.synthetic import synthetic_input, synthetic_model
    cfg = UPSNetConfig.cityscapes_r50()
    m_cpu = synthetic_model(cfg, depth=(1, 1, 1, 1), seed=3)
    m_gpu = synthetic_model(cfg, depth=(1, 1, 1, 1), seed=3, device=dev)
    m_gpu.load_state_dict({k: v.to(dev) for k, v in m_cpu.state_dict().items()})   # identical weights by construction
    m_cpu = m_cpu.to("cpu"); m_cpu.prepare(); m_gpu.prepare()
    m_gpu.keep_intermediates = True
    Hh, Ww = 256, 384
    inp = synthetic_input(Hh, Ww, seed=4)
    with cpu_ops(), torch.no_grad():
        r2, r3, r4, r5 = m_cpu.resnet_backbone(inp["data"])
        p_cpu = m_cpu.fpn(r2, r3, r4, r5)
        fcn_cpu = m_cpu.fcn_head(*p_cpu[:4])["fcn_output"]
        out_cpu = m_cpu(inp)
    gin = {"data": inp["data"].to(dev), "im_info": inp["im_info"]}
    with torch.no_grad():
        g2, g3, g4, g5 = m_gpu.resnet_backbone(gin["data"])
        p_gpu = m_gpu.fpn(g2, g3, g4, g5)
        out_gpu = m_gpu(gin)
    for a, b in zip(p_gpu, p_cpu):
        assert (a.cpu() - b).abs().max() <= TOL * max(1.0, float(b.abs().max()))
    it = out_gpu["_intermediates"]
    fcn_gpu = it["fcn_output"]
    assert (fcn_gpu.cpu() - fcn_cpu).abs().max() <= TOL * max(1.0, float(fcn_cpu.abs().max()))
    sem_agree = (out_gpu["fcn_outputs"].cpu() == out_cpu["fcn_outputs"]).float().mean().item()
    assert sem_agree > 0.999, sem_agree
    # semantic argmax and panoptic head: exact, on the engine's own inputs
    wk, wl, ws = O.panoptic_head(fcn_gpu[0].cpu().numpy(), it["pmask_rois"][:, 1:].cpu().numpy(),
                                 it["pcls_prob"].cpu().numpy(), it["pmask_score"].cpu().numpy().reshape(-1, 28, 28),
                                 it["pcls_idx"].cpu().numpy(), 11, want_sem=True)
    assert it["keep_inds"].cpu().tolist() == wk.tolist()
    assert np.array_equal(out_gpu["panoptic_outputs"][0].cpu().numpy(), wl)
    assert np.array_equal(out_gpu["fcn_outputs"][0].cpu().numpy(), ws)
    assert out_gpu["panoptic_outputs"].dtype == torch.int64 and out_gpu["panoptic_outputs"].shape == (1, Hh, Ww)
    assert out_gpu["pred_boxes"].shape[1] == 5 and out_gpu["mask_probs"].shape[1:] == (9, 28, 28)


def test_mask_removal_and_segterm_modules_match_reference_composition(dev):
    """The stand-alone MaskRemoval / SegTerm modules (reference signatures) composed exactly like
    models/resnet_upsnet.py:223-240 in plain torch must reproduce the fused head bit for bit."""
    import upsnet_b200 as U
    fcn, b, prob, ml, cls = pan_case(20, 96, 128, seed=31)
    fcn_t = t(fcn[None], dev); b_t = t(b, dev); cls_t = t(cls, dev)
    keep, energy = U.MaskRemoval(0.3)(b_t, t(prob, dev), t(ml[:, None], dev), cls_t, (96, 128))
    rois5 = torch.cat([torch.zeros(len(keep), 1, device=dev), b_t[keep]], 1)
    seg_logits, seg_inst = U.SegTerm(19, num_classes=9)(cls_t[keep], fcn_t, rois5 * 4.0)
    void = fcn_t[:, 11:].max(dim=1, keepdim=True)[0] - seg_inst.max(dim=1, keepdim=True)[0]
    logits = torch.cat([seg_logits, seg_inst + energy, void], dim=1)
    out = logits.max(dim=1)[1]
    out[out == logits.shape[1] - 1] = 255
    wk, wl = O.panoptic_head(fcn, b, prob, ml, cls, 11)
    assert keep.cpu().tolist() == wk.tolist()
    assert np.array_equal(out[0].cpu().numpy(), wl)
    fk, fl = run_pan(dev, fcn, b, prob, ml, cls)
    assert fk.cpu().tolist() == wk.tolist() and np.array_equal(fl[0].cpu().numpy(), wl)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("shape", [(1, 64, 62, 90), (2, 8, 17, 5), (1, 64, 128, 256)])
def test_maxpool_nhwc_matches_torch(dev, dtype, shape):
    """Stem max-pool (models/resnet.py:163) on NHWC storage: exact (max of the same values)."""
    import upsnet_b200 as U
    g = torch.Generator().manual_seed(4)
    x = torch.randn(shape, generator=g).to(dev).to(dtype).contiguous(memory_format=torch.channels_last)
    got = U.operators.max_pool2d(x, 3, 2, 1)
    want = torch.nn.functional.max_pool2d(x.float(), 3, 2, 1)
    assert got.dtype == dtype and got.shape == want.shape
    assert torch.equal(got.float(), want)


@pytest.mark.parametrize("shape,f", [((1, 19, 64, 96), 4), ((2, 3, 17, 5), 4), ((1, 19, 33, 50), 2), ((1, 1, 8, 8), 8)])
def test_upsample_bilinear_matches_torch(dev, shape, f):
    """Semantic-logit up-sampling (models/fcn.py:88-101): same source-index rule as ATen's upsample_bilinear2d."""
    import upsnet_b200 as U
    g = torch.Generator().manual_seed(6)
    x = torch.randn(shape, generator=g).to(dev)
    got = U.operators.upsample_bilinear(x, f)
    want = torch.nn.functional.interpolate(x, None, f, mode="bilinear", align_corners=False)
    assert got.shape == want.shape
    assert (got - want).abs().max().item() < 2e-6 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("hs,ws,n", [(16, 24, 6), (64, 128, 40), (33, 17, 3)])
def test_panoptic_head_fused_upsample_is_bit_identical(dev, hs, ws, n):
    """upsnet_panoptic_head_up4 (x4 bilinear up-sampling of the semantic score map evaluated inside the fusion kernel,
    models/fcn.py:88-101 + resnet_upsnet.py:217-247) against upsnet_panoptic_head on the materialised logits, and both
    against the CPU oracle on those logits: labels, semantic argmax and keep list bit for bit."""
    import upsnet_b200 as U
    from upsnet_b200 import operators as ops
    from oracle import oracle as O
    rng = np.random.default_rng(31 + hs)
    H, W = 4 * hs, 4 * ws
    score = (rng.standard_normal((1, 19, hs, ws)) * 3).astype(np.float32)
    c = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n)], 1); s = rng.uniform(6, 0.6 * min(H, W), (n, 2))
    b = np.concatenate([c - s / 2, c + s / 2], 1).astype(np.float32)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, W - 1); b[:, 1::2] = np.clip(b[:, 1::2], 0, H - 1)
    prob = rng.uniform(0.3, 1.0, n).astype(np.float32)
    ml = (rng.standard_normal((n, 28, 28)) * 2 + 0.5).astype(np.float32)
    cls = rng.integers(1, 9, n).astype(np.int64)
    ts = torch.from_numpy(score).to(dev)
    full = ops.upsample_bilinear(ts, 4)
    args = [torch.from_numpy(a).to(dev) for a in (b, prob, ml[:, None], cls)]
    k0, l0, s0 = U.panoptic_fuse(full, *args, 11, want_sem=True)
    k1, l1, s1 = U.panoptic_fuse(ts, *args, 11, want_sem=True, up4=True)
    assert torch.equal(k0, k1) and torch.equal(l0, l1) and torch.equal(s0, s1)
    wk, wl = O.panoptic_head(full[0].cpu().numpy(), b, prob, ml, cls, 11)
    assert k1.cpu().tolist() == wk.tolist() and np.array_equal(l1[0].cpu().numpy(), wl)
