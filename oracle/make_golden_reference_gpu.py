#!/usr/bin/env python
"""oracle/make_golden_reference_gpu.py -- TEST INFRASTRUCTURE ONLY; run once on a B200 after `make -C oracle ref` has
compiled the reference's CUDA kernels into oracle/_ref/, with the reference tree at $SIS3D_REFERENCE:

    SIS3D_REFERENCE=<reference tree> python oracle/make_golden_reference_gpu.py   # writes tests/golden/reference_gpu.npz

Stores what the reference's own GPU code computes on the seeded inputs of the GPU tests, so that they compare libsis3d
with it on any machine:
  * nms_cuda_keep_<seed>: keep list of the reference's NMS kernel (oracle/_ref/libref_nms_cuda.so), its suppression
    bitmask reduced on the host as lib/layer_utils/nms/src/nms_cuda.c:41-59 does (tests/test_gpu_ops.py);
  * roi_cuda_top / roi_cuda_argmax: the reference's RoI-pooling kernel (oracle/_ref/libref_roi_cuda.so) on the inputs of
    tests/golden/operators.npz (tests/test_gpu_ops.py);
  * dropin_<case>_*: the predictions of the reference's unmodified Python on the GPU with its two extension modules bound
    to libsis3d.so (oracle/run_reference_gpu.py; tests/test_gpu_dropin_reference.py).
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-sis_b200"))
import sis3d_synth as synth  # noqa: E402

NMS_CASES = ((0, 400, 0.1), (7, 777, 0.25))
DROPIN_CASES = ("odd_45x27x41", "cfg1_32")


def nms_keep(ref, seed, n, thr):
    b = torch.from_numpy(synth.make_nms_boxes(seed, n)).cuda()
    cb = (n + 63) // 64
    mask = torch.zeros(n, cb, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ref._nms(C.c_int(n), C.c_void_p(b.data_ptr()), C.c_void_p(mask.data_ptr()), C.c_float(thr))
    torch.cuda.synchronize()
    m = mask.cpu().numpy().view(np.uint64)
    remv = np.zeros(cb, np.uint64)
    keep = []
    for i in range(n):
        if not (remv[i // 64] >> np.uint64(i % 64)) & np.uint64(1):
            keep.append(i)
            remv[i // 64:] |= m[i, i // 64:]
    return np.array(keep, dtype=np.int64)


def roi_pool(ref):
    rois = np.load(os.path.join(ROOT, "tests", "golden", "operators.npz"))["roi_rois"]
    feat = np.random.default_rng(11).standard_normal((1, 16, 24, 12, 24)).astype(np.float32)
    fd, rd = torch.from_numpy(feat).cuda(), torch.from_numpy(rois).cuda()
    top = torch.zeros(rd.shape[0], 16, 4, 4, 4, device="cuda")
    arg = torch.zeros(top.shape, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ref.ROIPoolForwardLaucher(C.c_void_p(fd.data_ptr()), C.c_float(0.25), rd.shape[0], 24, 12, 24, 16, 4, 4, 4,
                              C.c_void_p(rd.data_ptr()), C.c_void_p(top.data_ptr()), C.c_void_p(arg.data_ptr()), C.c_void_p(0))
    torch.cuda.synchronize()
    return top.cpu().numpy(), arg.cpu().numpy()


def dropin(tag, tmp):
    out = os.path.join(tmp, f"{tag}.npz")
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "run_reference_gpu.py"), "--case", tag, "--out", out],
                          env=env, cwd=tmp)
    return {f"dropin_{tag}_{k}": v for k, v in np.load(out).items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "reference_gpu.npz"))
    a = ap.parse_args()
    assert os.path.isdir(os.path.join(os.environ.get("SIS3D_REFERENCE", ""), "lib")), "set SIS3D_REFERENCE to the reference tree"
    g = {}
    nms = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_nms_cuda.so"))
    for seed, n, thr in NMS_CASES:
        g[f"nms_cuda_cfg_{seed}"] = np.array([seed, n, thr])
        g[f"nms_cuda_keep_{seed}"] = nms_keep(nms, seed, n, thr)
    g["roi_cuda_top"], g["roi_cuda_argmax"] = roi_pool(C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_roi_cuda.so")))
    with tempfile.TemporaryDirectory() as tmp:
        for tag in DROPIN_CASES:
            g.update(dropin(tag, tmp))
    np.savez_compressed(a.out, **g)
    print(f"{a.out}: {len(g)} arrays, {os.path.getsize(a.out) / 1e3:.0f} kB on {torch.cuda.get_device_name()}")


if __name__ == "__main__":
    main()
