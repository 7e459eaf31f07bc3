"""Generates tests/golden/reference_kernels.npz: the outputs of the reference's own CUDA kernels (ROIAlign, deformable
im2col v1 / v2 + GEMM, NMS) on the inputs of tests/test_gpu_parity.py, which compares the product's kernels against them.
Outputs larger than test_gpu_parity.REF_SAMPLE elements are stored at the fixed indices of test_gpu_parity.ref_sample.

Needs a GPU and oracle/_ref/libupsnet_ref.so (oracle.build() compiles it from the reference's sources when they are
present).  Run:  python tests/golden/make_reference_kernels.py [out.npz]"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

from oracle import oracle as O  # noqa: E402
from test_gpu_parity import DCN_CFGS, dcn_case, nms_dense_cases, ref_sample, roi_align_config1_case  # noqa: E402


def main(path):
    dev = torch.device("cuda", 0)
    ref = O.RefKernels()

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def sampled(y):
        y = y.cpu().numpy().reshape(-1)
        return y[ref_sample(y.size)]
    ops = np.load(os.path.join(HERE, "oracle_ops.npz"))
    gref = np.load(os.path.join(HERE, "reference_numpy.npz"))
    out = {"roi_align_golden": ref.roi_align(t(ops["ra_feat"]), t(ops["ra_rois"]), 7, 7, 0.25).cpu().numpy()}
    feat, rois = roi_align_config1_case()
    for ph in (7, 14):
        out["roi_align_config1_ph%d" % ph] = sampled(ref.roi_align(feat.to(dev), t(rois), ph, ph, 0.25))
    for i in range(int(gref["nms_cases"])):
        keep = ref.nms(gref["nms%d_dets" % i], float(gref["nms%d_thresh" % i]))
        out["nms_golden_%d" % i] = np.asarray(keep, np.int32)
    for n, d in nms_dense_cases():
        if n <= 4097:
            out["nms_dense_%d" % n] = np.asarray(ref.nms(d, 0.5), np.int32)
    out["dcn_golden"] = ref.deform_conv(t(ops["dcn_x"]), t(ops["dcn_off"]), t(ops["dcn_w"]), t(ops["dcn_b"]),
                                        pad=1, dg=2).cpu().numpy()
    for ci, cfg in enumerate(DCN_CFGS):
        for modulated in (False, True):
            x, off, w, b, mask = dcn_case(cfg, modulated)
            y = ref.deform_conv(t(x), t(off), t(w), t(b), None if mask is None else t(mask),
                                cfg["stride"], cfg["pad"], cfg["dil"], cfg["dg"])
            out["dcn_cfg%d_mod%d" % (ci, modulated)] = sampled(y)
    torch.cuda.synchronize()
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_kernels.npz"))
