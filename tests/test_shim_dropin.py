"""Drop-in proof for the `upsnet/` overlay (VERDICT r1 next-round item 8, SURVEY section 8b / Appendix B).

Stand-alone: this repository alone on sys.path -- the lines of `upsnet_end2end_test.py` that bind the script to the
model code (:36-37 config, :43-44 `from upsnet.models import *`, :162 `eval(config.symbol)()`, :190-193
`load_state_dict(..., resume=True)` with DataParallel's `module.` prefix, and the backbone-only torchvision key
remapping of models/resnet.py:213-222), then a forward through the engine (CPU ops plugged in: no GPU here)."""
import os
import textwrap

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_standalone_script_lines_and_state_dict(tmp_path):
    yaml_path = tmp_path / "exp.yaml"
    yaml_path.write_text(textwrap.dedent("""
        symbol: resnet_50_upsnet
        gpus: '0'
        dataset:
          num_classes: 9
          num_seg_classes: 19
        network:
          has_fcn_head: true
          fcn_num_layers: 2
          has_panoptic_head: true
        test:
          max_det: 100
    """))
    from upsnet.config.config import config, update_config          # upsnet_end2end_test.py:36
    update_config(str(yaml_path))                                   # parse_args.py:27
    assert config.network.fcn_num_layers == 2 and config.dataset.num_seg_classes == 19
    from upsnet.models import resnet_50_upsnet, resnet_101_upsnet   # noqa: F401  upsnet_end2end_test.py:44 (`import *`)
    test_model = eval(config.symbol)()                              # upsnet_end2end_test.py:162
    assert test_model.cfg.fcn_num_layers == 2 and test_model.num_classes == 9
    assert len(test_model.resnet_backbone.res4.layers) == 6

    # a checkpoint of this model saved through DataParallel: reference key names + `module.` prefix (resume=True)
    from upsnet_b200.synthetic import synthetic_model
    src = synthetic_model(test_model.cfg, seed=21)
    ckpt = {"module." + k: v.clone() for k, v in src.state_dict().items()}
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("error")                              # no unexpected / missing / shape warnings
        test_model.load_state_dict(ckpt, resume=True)               # upsnet_end2end_test.py:190-193
    for k, v in src.state_dict().items():      # .cpu(): DeformConv creates its parameters on CUDA when there is a GPU
        assert torch.equal(test_model.state_dict()[k].cpu(), v), k

    # backbone-only torchvision / caffe checkpoint (resume=False): conv1/bn1/layerN names (models/resnet.py:216-222)
    tv = {}
    for k, v in src.state_dict().items():
        if k.startswith("resnet_backbone.conv1."):
            tv[k[len("resnet_backbone.conv1."):]] = v + 1
        elif k.startswith("resnet_backbone.res"):
            n = int(k[len("resnet_backbone.res")])
            tv[k.replace("resnet_backbone.res%d.layers" % n, "layer%d" % (n - 1))] = v + 1
    fresh = eval(config.symbol)()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        fresh.load_state_dict(tv, resume=False)
    assert any("missing keys" in str(x.message) for x in w)        # heads are not in a backbone checkpoint
    assert torch.equal(fresh.state_dict()["resnet_backbone.res3.layers.1.conv2.weight"].cpu(),
                       src.state_dict()["resnet_backbone.res3.layers.1.conv2.weight"] + 1)
    assert torch.equal(fresh.state_dict()["resnet_backbone.conv1.bn1.running_var"].cpu(),
                       src.state_dict()["resnet_backbone.conv1.bn1.running_var"] + 1)

    # the forward the script's loop performs (upsnet_end2end_test.py:228): model(data) -> the reference's result dict
    from oracle.cpu_model import cpu_ops, synthetic_input
    small = synthetic_model(test_model.cfg, depth=(1, 1, 1, 1), seed=22)
    dst = type(small)([1, 1, 1, 1], test_model.cfg).to("cpu")
    dst.load_state_dict({"module." + k: v for k, v in small.state_dict().items()}, resume=True)
    inp = synthetic_input(96, 128, seed=23)
    with cpu_ops():
        a, b = small(inp), dst(inp)
    assert set(b.keys()) == {"cls_probs", "pred_boxes", "mask_probs", "fcn_outputs", "cls_inds", "panoptic_cls_inds",
                             "panoptic_cls_probs", "panoptic_outputs"}
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_reference_operator_module_paths():
    """The module paths models/resnet_upsnet.py:25-32 imports from, with the reference's constructor signatures."""
    from upsnet.operators.modules.deform_conv import DeformConv, DeformConvWithOffset             # noqa: F401
    from upsnet.operators.modules.fpn_roi_align import FPNRoIAlign                                # noqa: F401
    from upsnet.operators.modules.mask_matching import MaskMatching
    from upsnet.operators.modules.mask_removal import MaskRemoval
    from upsnet.operators.modules.mask_roi import MaskROI
    from upsnet.operators.modules.mod_deform_conv import ModDeformConv, ModulatedDeformConv       # noqa: F401
    from upsnet.operators.modules.pyramid_proposal import PyramidProposal
    from upsnet.operators.modules.roialign import RoIAlign                                        # noqa: F401
    from upsnet.operators.modules.unary_logits import MaskTerm, SegTerm
    from upsnet.nms.nms import gpu_nms_wrapper, py_nms_wrapper, cpu_nms_wrapper                    # noqa: F401
    MaskROI(clip_boxes=True, bbox_class_agnostic=False, top_n=100, num_classes=9, score_thresh=0.05)
    MaskROI(clip_boxes=True, bbox_class_agnostic=False, top_n=100, num_classes=9, nms_thresh=0.5, class_agnostic=True, score_thresh=0.6)
    PyramidProposal(feat_stride=np.array([4, 8, 16, 32, 64]), scales=np.array([8]), ratios=np.array([0.5, 1, 2]),
                    rpn_pre_nms_top_n=1000, rpn_post_nms_top_n=1000, threshold=0.7, rpn_min_size=0, individual_proposals=True)
    MaskRemoval(fraction_threshold=0.3); SegTerm(19); MaskTerm(19, box_scale=1 / 4.0); MaskMatching(19, enable_void=True)
    with pytest.raises(NotImplementedError):
        cpu_nms_wrapper(0.5)          # IoU >= thresh rule (SURVEY F10): not silently mapped onto the > kernel


def test_shim_modules_vs_reference_fixtures():
    """PyramidProposal / MaskROI through the reference module paths and signatures reproduce the reference's outputs."""
    from oracle.cpu_model import cpu_ops
    from upsnet.operators.modules.mask_roi import MaskROI
    from upsnet.operators.modules.pyramid_proposal import PyramidProposal
    from test_reference_fixtures import _check_mroi, mroi_case, pp_case
    ref = np.load(os.path.join(ROOT, "tests", "golden", "reference_modules.npz"))
    probs, deltas, info, pre, post, want_rois, want_sc = pp_case(ref, 2)
    with cpu_ops():
        m = PyramidProposal(np.array([4, 8, 16, 32, 64]), np.array([8]), np.array([0.5, 1, 2]), pre, post, 0.7, 0, individual_proposals=True)
        rois, sc = m([torch.from_numpy(p) for p in probs], [torch.from_numpy(d) for d in deltas], info[None])
        assert np.array_equal(sc.numpy(), want_sc)
        np.testing.assert_allclose(rois.numpy(), want_rois, rtol=0, atol=2e-3)
        c = mroi_case(ref, 1)
        mr = MaskROI(clip_boxes=True, bbox_class_agnostic=False, top_n=100, num_classes=9, nms_thresh=0.5,
                     class_agnostic=bool(c["agnostic"]), score_thresh=float(c["score_thresh"]))
        s, b, ci = mr(torch.from_numpy(c["rois"]), torch.from_numpy(c["delta"]), torch.from_numpy(c["prob"]), ref["mroi_im_info"])
        _check_mroi(c, s.numpy(), b.numpy(), ci.numpy())

