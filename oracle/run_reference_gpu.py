#!/usr/bin/env python
"""oracle/run_reference_gpu.py -- TEST INFRASTRUCTURE (drop-in test of the operator boundary, SURVEY 8b).

Runs the UNMODIFIED reference Python (network.py, proposal_layer.py, pth_nms.py, roi_pool.py, ... from the reference tree
at $SIS3D_REFERENCE) on the GPU in a process of its own -- the reference's package is called `lib`, like ours -- with its
two cffi extension modules replaced by the ctypes stubs of INTEGRATION.md section 2 bound to libsis3d.so
(oracle/ref_harness.py install(gpu=True)).  Writes the reference's _predictions for one named synthetic case;
oracle/make_golden_reference_gpu.py stores them as tests/golden/reference_gpu.npz.

    SIS3D_REFERENCE=<reference tree> python oracle/run_reference_gpu.py --case odd_45x27x41 --out ref_gpu.npz
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
SYNTH = os.path.join(ROOT, "3d-sis_b200", "sis3d_synth.py")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default="odd_45x27x41")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import importlib.util
    spec = importlib.util.spec_from_file_location("sis3d_synth", SYNTH)  # by path: our package dir must NOT be on sys.path
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    import ref_harness as rh
    c = synth.CASES[a.case]
    yml = ("SUNCG" if c["cfgname"] == "suncg" else "ScanNet") + "/rpn_class_mask_5.yml"
    cfg = rh.load_cfg(yml, gpu=True, USE_IMAGES=c["use_images"], USE_IMAGES_GT=True, USE_MASK=c["use_mask"])
    w = synth.make_weights(seed=0, net=cfg.NET, use_images=c["use_images"], num_classes=cfg.NUM_CLASSES,
                           a1=cfg.NUM_ANCHORS_LEVEL1, a2=cfg.NUM_ANCHORS_LEVEL2, use_mask=c["use_mask"])
    net = rh.build_net(cfg, w)
    data, boxes = synth.make_scene(c["seed"], c["dims"])
    views = None
    if c["use_images"]:
        views = synth.make_views(c["seed"], c["dims"], c["n_img"], boxes, intrinsic=np.array(cfg.INTRINSIC, dtype=np.float32))
    with torch.no_grad():
        P = rh.reference_forward(net, cfg, data, views)
    torch.cuda.synchronize()
    out = dict(rois=P["rois"][0].detach().cpu().numpy(), roi_scores=P["roi_scores"][0].detach().cpu().numpy(),
               level_inds=np.asarray(P["level_inds"][0].detach().cpu().numpy() if torch.is_tensor(P["level_inds"][0]) else P["level_inds"][0]),
               cls_pred=P["cls_pred"].detach().cpu().numpy(), cls_prob=P["cls_prob"].detach().cpu().numpy(),
               bbox_pred=P["bbox_pred"].detach().cpu().numpy(), gpu_nms_calls=rh.EXT_CALLS["gpu_nms"],
               roi_cuda_calls=rh.EXT_CALLS["roi_pooling_forward_cuda"],
               convs_on_cuda=int(next(net.parameters()).is_cuda))
    if c["use_mask"]:
        masks = P["mask_pred"][0]
        out["n_masks"] = len(masks)
        for j, m in enumerate(masks):
            out[f"mask_{j}"] = m.detach().cpu().numpy()
    np.savez_compressed(a.out, **out)
    print(f"reference on GPU over libsis3d _ext stubs: {out['rois'].shape[0]} rois, {out.get('n_masks', 0)} masks, "
          f"gpu_nms x{out['gpu_nms_calls']}, roi_pooling_forward_cuda x{out['roi_cuda_calls']}")


if __name__ == "__main__":
    main()
