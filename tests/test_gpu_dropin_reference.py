"""Drop-in test of the operator boundary (SURVEY 8b, INTEGRATION.md section 2): the reference's OWN Python -- network.py,
proposal_layer.py, pth_nms.py, roi_pool.py, unmodified -- run on a B200 with its two cffi extension modules rebound to
libsis3d.so (`gpu_nms` -> sis3d_nms, `roi_pooling_forward_cuda` -> sis3d_roi_pool_fwd) by oracle/run_reference_gpu.py.
Its predictions are stored in tests/golden/reference_gpu.npz (generator: oracle/make_golden_reference_gpu.py) and must
equal (a) the CPU oracle, which is pinned to the all-CPU run of the same files, and (b) this repo's Network.forward on the
same inputs."""
import numpy as np
import pytest
import torch

import sis3d_synth as synth
from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("tag", ["odd_45x27x41", "cfg1_32"])
def test_reference_python_runs_over_libsis3d_extension_stubs(oracle, tag):
    g = load_golden("reference_gpu.npz")
    ref = {k[len(f"dropin_{tag}_"):]: v for k, v in g.items() if k.startswith(f"dropin_{tag}_")}
    c = synth.CASES[tag]
    assert ref["convs_on_cuda"] == 1 and ref["gpu_nms_calls"] >= 1 and ref["roi_cuda_calls"] >= 1, "the rebound kernels must have run"
    ocfg, w, data, views = synth.build_case(oracle, c)
    want = oracle.forward(ocfg, w, data, views, fma_mode=1)
    # (a) reference-on-GPU over our kernels == CPU oracle (pinned to the all-CPU reference run)
    assert ref["rois"].shape == tuple(want["rois"].shape)
    np.testing.assert_allclose(ref["rois"], want["rois"].numpy(), atol=2e-3)
    assert np.array_equal(ref["level_inds"].reshape(-1), want["level_inds"].numpy().reshape(-1))
    assert np.array_equal(ref["cls_pred"], want["cls_pred"].numpy())
    np.testing.assert_allclose(ref["cls_prob"], want["cls_prob"].numpy(), atol=1e-4)
    # (b) == this repo's forward (default math mode)
    net, cfg = synth.make_net(c, keep_debug=False, math="exact")
    P = net.forward(synth.make_blobs(c, data, views), "TEST", None)
    torch.cuda.synchronize()
    np.testing.assert_allclose(P["rois"][0].cpu().numpy(), ref["rois"], atol=2e-3)
    assert np.array_equal(P["cls_pred"].cpu().numpy(), ref["cls_pred"])
    if c["use_mask"]:
        assert int(ref["n_masks"]) == len(P["mask_pred"][0]) == len(want["mask_pred"])
        for j, m in enumerate(P["mask_pred"][0]):
            assert float(np.abs(m.cpu().numpy() - ref[f"mask_{j}"]).max()) < 1e-3
