"""Operator-level parity on the GPU (run with -m gpu on a B200): every call goes through the C ABI
(libsis3d.so via ctypes) and is compared with the CPU oracle on the same seeded inputs."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import sis3d_synth as synth
from conftest import ROOT, load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def S():
    from lib import _sis3d
    return _sis3d


# ---------------------------------------------------------------- NMS
@pytest.mark.parametrize("seed,n,thr", [(0, 400, 0.1), (1, 400, 0.35), (2, 1000, 0.5), (3, 64, 0.1), (4, 65, 0.7),
                                        (5, 1, 0.1), (6, 2500, 0.3)])
def test_nms_bit_exact(oracle, seed, n, thr):
    from lib.layer_utils.nms_wrapper import nms
    b = synth.make_nms_boxes(seed, n)
    keep = nms(torch.from_numpy(b).to(DEV), thr).cpu().numpy()
    want = oracle.nms3d(b, thr, fma_mode=1)  # the reference's CUDA arithmetic
    assert np.array_equal(keep, want)
    # the numpy (CPU-reference) arithmetic may differ by one ulp at the threshold only
    want_cpu = oracle.nms3d(b, thr, fma_mode=0)
    iou = oracle.iou_matrix(b, 0)
    if np.abs(iou - np.float32(thr)).min() > 1e-6:
        assert np.array_equal(keep, want_cpu)


def test_nms_matches_golden_reference_cpu_nms(oracle):
    from lib.layer_utils.nms_wrapper import nms
    g = load_golden("operators.npz")
    for seed in range(6):
        s, n, thr = g[f"nms_cfg_{seed}"]
        b = synth.make_nms_boxes(int(s), int(n))
        keep = nms(torch.from_numpy(b).to(DEV), float(thr)).cpu().numpy()
        assert np.array_equal(keep, g[f"nms_keep_{seed}"])


def test_nms_edge_cases(oracle):
    from lib.layer_utils.nms_wrapper import nms
    assert nms(torch.zeros(0, 6, device=DEV), 0.5).numel() == 0
    same = np.tile(np.array([[1, 2, 3, 9, 9, 9]], np.float32), (130, 1))
    assert nms(torch.from_numpy(same).to(DEV), 0.5).cpu().tolist() == [0]
    far = np.stack([np.array([i * 20, 0, 0, i * 20 + 5, 5, 5], np.float32) for i in range(70)])
    assert nms(torch.from_numpy(far).to(DEV), 0.1).cpu().tolist() == list(range(70))


def test_nms_mask_vs_reference_cuda_kernel(oracle):
    """Keep list of the reference's own kernel (its bitmask reduced as nms_cuda.c does; tests/golden/reference_gpu.npz,
    generator oracle/make_golden_reference_gpu.py) == ours."""
    from lib.layer_utils.nms_wrapper import nms
    g = load_golden("reference_gpu.npz")
    for seed in (0, 7):
        s, n, thr = g[f"nms_cuda_cfg_{seed}"]
        bd = torch.from_numpy(synth.make_nms_boxes(int(s), int(n))).to(DEV)
        assert nms(bd, float(thr)).cpu().tolist() == g[f"nms_cuda_keep_{seed}"].tolist()


# ---------------------------------------------------------------- RoI pooling
def _roi_inputs(seed=11, C_=16, dims=(24, 12, 24), n=40):
    rng = np.random.default_rng(seed)
    feat = rng.standard_normal((1, C_) + dims).astype(np.float32)
    rois = synth.make_nms_boxes(seed + 10, n)
    rois[0] = [5, 5, 5, 5, 5, 5]
    rois[1] = [90, 40, 90, 96, 48, 96]
    rois[2] = [0, 0, 0, 96, 48, 96]
    rois[3] = [10.5, 3.25, 7.75, 11.0, 3.5, 8.0]
    return feat, rois


@pytest.mark.parametrize("C_,pool", [(16, 4), (128, 4), (130, 2), (8, 3)])
def test_roi_pool_exact_both_layouts(oracle, S, C_, pool):
    from lib.layer_utils.roi_pooling.roi_pool import RoIPoolFunction
    feat, rois = _roi_inputs(C_=C_)
    want, warg = oracle.roi_pool3d(feat, rois, (pool,) * 3, 0.25)
    fn = RoIPoolFunction(pool, pool, pool, 0.25)
    out = fn(torch.from_numpy(feat).to(DEV), torch.from_numpy(rois).to(DEV))
    assert np.array_equal(out.cpu().numpy(), want)
    assert np.array_equal(fn.argmax.cpu().numpy(), warg)
    # VC layout, pyramid form (level 1 -> feat, level 2 -> -feat, id 0 -> zeros)
    fvc = torch.from_numpy(feat[0]).to(DEV).permute(1, 2, 3, 0).contiguous()
    n = rois.shape[0]
    lv = torch.ones(n, dtype=torch.int32, device=DEV)
    lv[1::3] = 2
    lv[2::5] = 0
    top = torch.empty(n, C_ * pool ** 3, device=DEV)
    arg = torch.empty(n, C_ * pool ** 3, dtype=torch.int32, device=DEV)
    rois_d, neg_fvc = torch.from_numpy(rois).to(DEV), (-fvc).contiguous()  # keep device buffers alive across the async launch
    S.check(S.lib.sis3d_roi_pool_levels(S.ptr(fvc), S.ptr(neg_fvc), None, S.ptr(lv), S.f32(0.25), n, 24, 12, 24,
                                        C_, pool, pool, pool, S.ptr(rois_d), S.ptr(top), S.ptr(arg),
                                        S.stream()))
    want2, warg2 = oracle.roi_pool3d(-feat, rois, (pool,) * 3, 0.25)
    lvh = lv.cpu().numpy()
    got = top.cpu().numpy().reshape(want.shape)
    garg = arg.cpu().numpy().reshape(want.shape)
    assert np.array_equal(got[lvh == 1], want[lvh == 1]) and np.array_equal(garg[lvh == 1], warg[lvh == 1])
    assert np.array_equal(got[lvh == 2], want2[lvh == 2]) and np.array_equal(garg[lvh == 2], warg2[lvh == 2])
    assert not got[lvh == 0].any()


def test_roi_pool_golden_and_reference_cuda(oracle):
    from lib.layer_utils.roi_pooling.roi_pool import RoIPoolFunction
    g = load_golden("operators.npz")
    feat = np.random.default_rng(11).standard_normal((1, 16, 24, 12, 24)).astype(np.float32)
    fd, rd = torch.from_numpy(feat).to(DEV), torch.from_numpy(g["roi_rois"]).to(DEV)
    fn = RoIPoolFunction(4, 4, 4, 0.25)
    out = fn(fd, rd)
    assert np.array_equal(out.cpu().numpy(), g["roi_out"])  # reference CPU C kernel
    ref = load_golden("reference_gpu.npz")  # reference CUDA kernel (generator: oracle/make_golden_reference_gpu.py)
    assert np.array_equal(out.cpu().numpy(), ref["roi_cuda_top"].reshape(out.shape))
    assert np.array_equal(fn.argmax.cpu().numpy(), ref["roi_cuda_argmax"].reshape(fn.argmax.shape))


# ---------------------------------------------------------------- convolution / pooling
CONV_CASES = [  # cin, cout, ks, stride, dims, bias, res, act
    (2, 32, 2, 2, (13, 9, 11), False, False, 1), (32, 32, 1, 1, (7, 5, 6), True, False, 1),
    (32, 32, 3, 1, (9, 6, 7), True, False, 1), (32, 64, 1, 1, (6, 5, 7), True, True, 1),
    (128, 64, 2, 2, (8, 6, 10), False, False, 1), (128, 128, 3, 1, (6, 5, 7), False, False, 1),
    (128, 256, 3, 1, (5, 4, 6), True, False, 1), (256, 22, 1, 1, (5, 4, 6), True, False, 0),
    (256, 66, 1, 1, (5, 4, 6), True, False, 0), (2, 64, 3, 1, (7, 9, 5), False, False, 1),
    (64, 19, 1, 1, (7, 3, 5), False, False, 2), (64, 64, 3, 1, (70, 3, 3), False, False, 1)]


@pytest.mark.parametrize("cin,cout,ks,stride,dims,bias,res,act", CONV_CASES)
def test_conv3d_vs_torch_fp32(S, cin, cout, ks, stride, dims, bias, res, act):
    rng = np.random.default_rng(cin * 1000 + cout + ks)
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w = (rng.standard_normal((cout, cin, ks, ks, ks)) / np.sqrt(cin * ks ** 3)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32) if bias else None
    pad = 1 if ks == 3 else 0
    ref = F.conv3d(torch.from_numpy(x), torch.from_numpy(w), None if b is None else torch.from_numpy(b), stride=stride,
                   padding=pad)
    r = rng.standard_normal(tuple(ref.shape)).astype(np.float32) if res else None
    if res:
        ref = ref + torch.from_numpy(r)
    ref = F.relu(ref) if act == 1 else (torch.sigmoid(ref) if act == 2 else ref)
    od = tuple(ref.shape[2:])
    xd = torch.from_numpy(x[0]).to(DEV).permute(1, 2, 3, 0).contiguous()  # VC
    wd = torch.from_numpy(w).to(DEV)
    ldw = (cout + 3) // 4 * 4
    packed = torch.empty(ks ** 3 * cin, ldw, device=DEV)
    S.check(S.lib.sis3d_pack_conv_weight(S.ptr(wd), cout, cin, ks, S.ptr(packed), S.stream()))
    out = torch.full(od + (cout + 4,), 7.0, device=DEV)  # write into a wider tensor at channel offset 4
    X, Y, Z = dims
    for layout in ("vc", "ncdhw"):
        if layout == "vc":
            inp, strides, sc = xd, (Y * Z * cin, Z * cin, cin), 1
        else:
            inp, strides, sc = torch.from_numpy(x[0]).to(DEV).contiguous(), (Y * Z, Z, 1), X * Y * Z
        regions, tiles = S.make_regions([dict(in_off=0, out_off=0, in_dim=dims, out_dim=od, in_stride=strides)], DEV)
        rd = torch.from_numpy(r[0]).to(DEV).permute(1, 2, 3, 0).contiguous() if res else None
        bd = torch.from_numpy(b).to(DEV) if bias else None
        S.check(S.lib.sis3d_conv3d(S.ptr(inp), C.c_int64(sc), S.ptr(packed), S.ptr(bd),
                                   S.ptr(rd), cout if res else 0, 0, S.ptr(out), cout + 4, 4, S.ptr(regions), 1, tiles, cin,
                                   cout, ks, stride, pad, act, S.stream()))
        got = out[..., 4:].permute(3, 0, 1, 2).cpu()
        assert torch.all(out[..., :4] == 7.0)
        torch.testing.assert_close(got, ref[0], atol=2e-5, rtol=1e-4)


def test_conv3d_regions_zero_pad_at_crop_border(S):
    """Two crops of one NCDHW scene in a single launch == conv of each crop with zero padding."""
    rng = np.random.default_rng(5)
    X, Y, Z = 20, 12, 16
    scene = rng.standard_normal((1, 2, X, Y, Z)).astype(np.float32)
    w = (rng.standard_normal((64, 2, 3, 3, 3)) / 7).astype(np.float32)
    crops = [(2, 1, 3, 9, 8, 10), (5, 0, 0, 20, 12, 7)]
    sd = torch.from_numpy(scene).to(DEV)
    packed = torch.empty(54, 64, device=DEV)
    wdev = torch.from_numpy(w).to(DEV)
    S.check(S.lib.sis3d_pack_conv_weight(S.ptr(wdev), 64, 2, 3, S.ptr(packed), S.stream()))
    sizes = [(c[3] - c[0], c[4] - c[1], c[5] - c[2]) for c in crops]
    offs = np.concatenate([[0], np.cumsum([a * b * c for a, b, c in sizes])])
    out = torch.empty(int(offs[-1]) * 64, device=DEV)
    regions, tiles = S.make_regions([dict(in_off=(c[0] * Y + c[1]) * Z + c[2], out_off=int(offs[j]) * 64, in_dim=s, out_dim=s,
                                          in_stride=(Y * Z, Z, 1)) for j, (c, s) in enumerate(zip(crops, sizes))], DEV)
    S.check(S.lib.sis3d_conv3d(S.ptr(sd), C.c_int64(X * Y * Z), S.ptr(packed), None, None, 0, 0, S.ptr(out), 64, 0,
                               S.ptr(regions), 2, tiles, 2, 64, 3, 1, 1, 1, S.stream()))
    for j, (c, s) in enumerate(zip(crops, sizes)):
        ref = F.relu(F.conv3d(torch.from_numpy(scene[:, :, c[0]:c[3], c[1]:c[4], c[2]:c[5]]), torch.from_numpy(w), padding=1))[0]
        got = out[int(offs[j]) * 64:int(offs[j + 1]) * 64].view(*s, 64).permute(3, 0, 1, 2).cpu()
        torch.testing.assert_close(got, ref, atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("C,dims", [(64, (9, 5, 7)), (64, (48, 24, 48)), (128, (24, 12, 24)), (16, (17, 8, 3)), (8, (6, 9, 11)),
                                    (64, (1, 1, 1))])
def test_maxpool3_exact(S, C, dims):
    """MaxPool3d(3,1,1): tiled kernel (C % 16 == 0) and the generic one, written into a channel slice of a wider tensor."""
    x = torch.randn(1, C, *dims)
    ref = F.max_pool3d(x, 3, 1, 1)[0]
    xd = x[0].to(DEV).permute(1, 2, 3, 0).contiguous()
    out = torch.zeros(*dims, 2 * C, device=DEV)
    S.check(S.lib.sis3d_maxpool3(S.ptr(xd), S.ptr(out), 2 * C, C, *dims, C, S.stream()))
    assert torch.equal(out[..., C:].permute(3, 0, 1, 2).cpu(), ref)
    assert not out[..., :C].any()


# ---------------------------------------------------------------- projection
def _views(dims, n_img, seed):
    data, boxes = synth.make_scene(seed, dims)
    return synth.make_views(seed, dims, n_img, boxes)


@pytest.mark.parametrize("tag,dims,n_img,seed", [("odd_45x27x41", (45, 27, 41), 3, 202), ("cfg2_96x48x96", (96, 48, 96), 5, 303)])
def test_compute_projection_index_lists_exact(oracle, tag, dims, n_img, seed):
    from lib.layer_utils.projection import ProjectionHelper
    g = load_golden(f"forward_{tag}.npz")
    cfg = oracle.make_cfg("scannet")
    v = _views(dims, n_img, seed)
    helper = ProjectionHelper(cfg.INTRINSIC, cfg.PROJ_DEPTH_MIN, cfg.PROJ_DEPTH_MAX, cfg.DEPTH_SHAPE, dims, cfg.VOXEL_SIZE)
    for i in range(n_img):
        m = helper.compute_projection(torch.from_numpy(v["depths"][i]).to(DEV), torch.from_numpy(v["poses"][i]),
                                      torch.from_numpy(v["world2grid"]))
        assert m is not None
        k = int(m[0][0].item())
        assert k == len(g[f"proj3d_{i}"]), f"view {i}: {k} vs {len(g[f'proj3d_{i}'])}"
        assert np.array_equal(m[0][1:1 + k].cpu().numpy(), g[f"proj3d_{i}"])
        assert np.array_equal(m[1][1:1 + k].cpu().numpy(), g[f"proj2d_{i}"])


def test_compute_projection_none_when_nothing_valid(oracle):
    from lib.layer_utils.projection import ProjectionHelper
    cfg = oracle.make_cfg("scannet")
    dims = (16, 16, 16)
    helper = ProjectionHelper(cfg.INTRINSIC, cfg.PROJ_DEPTH_MIN, cfg.PROJ_DEPTH_MAX, cfg.DEPTH_SHAPE, dims, cfg.VOXEL_SIZE)
    v = _views(dims, 1, 1)
    depth = torch.full((32, 41), 9.0)  # beyond depth_max everywhere
    assert helper.compute_projection(depth.to(DEV), torch.from_numpy(v["poses"][0]), torch.from_numpy(v["world2grid"])) is None
    assert oracle.compute_projection(cfg, depth, v["poses"][0], v["world2grid"], dims) is None


def test_projection_apply_and_running_max(oracle):
    from lib.layer_utils.projection import Projection, ProjectionHelper
    cfg = oracle.make_cfg("scannet")
    dims, n_img = (45, 27, 41), 3
    v = _views(dims, n_img, 202)
    helper = ProjectionHelper(cfg.INTRINSIC, cfg.PROJ_DEPTH_MIN, cfg.PROJ_DEPTH_MAX, cfg.DEPTH_SHAPE, dims, cfg.VOXEL_SIZE)
    for i in range(n_img):
        m = helper.compute_projection(torch.from_numpy(v["depths"][i]).to(DEV), torch.from_numpy(v["poses"][i]),
                                      torch.from_numpy(v["world2grid"]))
        got = Projection.apply(torch.from_numpy(v["feats"][i]).to(DEV), m[0], m[1], dims)
        l3, l2 = oracle.compute_projection(cfg, v["depths"][i], v["poses"][i], v["world2grid"], dims)
        want = oracle.projection_scatter(v["feats"][i], l3, l2, dims)
        assert torch.equal(got.cpu(), want)


# ---------------------------------------------------------------- proposals
@pytest.mark.parametrize("dims,seed", [((24, 12, 24), 1), ((11, 7, 10), 2), ((8, 8, 8), 3)])
def test_rpn_proposals_vs_oracle(oracle, dims, seed):
    """Same logits/deltas in -> same top-N order, same NMS keep, boxes within float tolerance."""
    from lib.layer_utils.proposal_layer import rpn_proposals
    from lib.utils.config import cfg, cfg_from_file, cfg_reset
    cfg_reset()
    cfg_from_file(os.path.join(ROOT, "3d-sis_b200", "experiments", "cfgs", "ScanNet", "rpn_class_mask_5.yml"))
    ocfg = oracle.make_cfg("scannet")
    rng = np.random.default_rng(seed)
    scene = tuple(4 * d for d in dims)
    levels, olevels = [], []
    for A, tab in ((3, "scannet14_3.txt"), (11, "scannet14_11.txt")):
        n = dims[0] * dims[1] * dims[2]
        cls = (rng.standard_normal((n, 2 * A)) * 2).astype(np.float32)
        dl = (rng.standard_normal((n, 6 * A)) * 0.2).astype(np.float32)
        sizes = oracle.read_anchor_table(tab)
        levels.append(dict(cls=torch.from_numpy(cls).to(DEV), deltas=torch.from_numpy(dl).to(DEV),
                           sizes=torch.tensor(sizes, dtype=torch.float32, device=DEV), grid=dims, A=A, cls_mode=0))
        logits = torch.from_numpy(cls).view(n, 2, A)
        prob = F.softmax(logits, dim=1)[:, 1, :].reshape(-1)
        olevels.append((prob, torch.from_numpy(dl).view(-1, 6), oracle.generate_anchors(dims, sizes, 4)))
    want = oracle.proposal_layer(ocfg, olevels, scene, fma_mode=1)
    rois, scores, lvl, num, order = rpn_proposals(levels, scene, "TEST", want_order=True)
    n = int(num.item())
    # flat index (level, voxel, a) of the oracle's order: oracle indices are into the inside-compacted list
    inside = np.concatenate([oracle.inside_mask(l[2], scene) for l in olevels])
    flat_of_compact = np.nonzero(inside)[0]
    want_flat = flat_of_compact[want["order"]]
    got_flat = order.cpu().numpy()[:len(want_flat)]
    sc = want["all_scores"]
    if not np.array_equal(got_flat, want_flat):
        # only allowed difference: scores that differ by < 1 ulp-ish between expf implementations
        diff = np.nonzero(got_flat != want_flat)[0]
        s_sorted = sc[want["order"]]
        assert np.all(np.abs(s_sorted[diff] - s_sorted[np.clip(diff + 1, 0, len(s_sorted) - 1)]) < 1e-6) or \
            np.all(np.abs(s_sorted[diff] - s_sorted[np.clip(diff - 1, 0, len(s_sorted) - 1)]) < 1e-6)
        pytest.skip("top-N order differs only among near-tied scores")
    assert n == len(want["rois"])
    np.testing.assert_allclose(rois[:n].cpu().numpy(), want["rois"].numpy(), atol=1e-4, rtol=1e-5)
    np.testing.assert_allclose(scores[:n].cpu().numpy(), want["scores"].numpy(), atol=1e-6)
    assert np.array_equal(lvl[:n].cpu().numpy(), want["level_inds"].numpy().astype(np.int32))
    assert not rois[n:].any()


def test_rpn_proposals_few_candidates(oracle):
    """Fewer inside anchors than pre_top_n (empty-ish edge case, SURVEY appendix A: SUNCG 32^3 level 2)."""
    from lib.layer_utils.proposal_layer import rpn_proposals
    from lib.utils.config import cfg, cfg_from_file, cfg_reset
    cfg_reset()
    cfg_from_file(os.path.join(ROOT, "3d-sis_b200", "experiments", "cfgs", "SUNCG", "rpn_class_mask_5.yml"))
    ocfg = oracle.make_cfg("suncg")
    dims, scene = (8, 8, 8), (32, 32, 32)
    rng = np.random.default_rng(9)
    levels, olevels = [], []
    for A, tab in ((3, "suncg9_3.txt"), (6, "suncg9_6.txt")):
        n = 512
        cls = rng.standard_normal((n, 2 * A)).astype(np.float32)
        dl = (rng.standard_normal((n, 6 * A)) * 0.1).astype(np.float32)
        sizes = oracle.read_anchor_table(tab)
        levels.append(dict(cls=torch.from_numpy(cls).to(DEV), deltas=torch.from_numpy(dl).to(DEV),
                           sizes=torch.tensor(sizes, dtype=torch.float32, device=DEV), grid=dims, A=A, cls_mode=0))
        prob = F.softmax(torch.from_numpy(cls).view(n, 2, A), dim=1)[:, 1, :].reshape(-1)
        olevels.append((prob, torch.from_numpy(dl).view(-1, 6), oracle.generate_anchors(dims, sizes, 4)))
    assert oracle.inside_mask(olevels[1][2], scene).sum() == 0  # level 2 contributes nothing
    want = oracle.proposal_layer(ocfg, olevels, scene, fma_mode=1)
    rois, scores, lvl, num = rpn_proposals(levels, scene, "TEST")
    n = int(num.item())
    assert n == len(want["rois"])
    np.testing.assert_allclose(rois[:n].cpu().numpy(), want["rois"].numpy(), atol=1e-4)


# ---------------------------------------------------------------- tensor-core 3x3x3 conv (tcgen05, TF32)
TC_CASES = [  # cin, cout, dims, bias, res, act, ks
    (32, 32, (8, 4, 4), True, False, 1, 3), (32, 32, (17, 9, 11), True, False, 1, 3), (64, 64, (24, 12, 24), True, False, 1, 3),
    (128, 128, (11, 6, 10), False, False, 1, 3), (128, 256, (24, 12, 24), True, False, 1, 3),
    (64, 64, (9, 5, 3), False, True, 0, 3), (32, 32, (48, 24, 48), True, False, 1, 1), (64, 32, (11, 6, 9), True, False, 1, 1),
    (32, 64, (24, 12, 24), True, True, 1, 1), (128, 64, (24, 12, 24), True, False, 1, 1), (64, 128, (7, 5, 6), True, True, 1, 1)]


@pytest.mark.parametrize("cin,cout,dims,bias,res,act,ks", TC_CASES)
def test_conv3d_tc_tf32_vs_fp32(S, cin, cout, dims, bias, res, act, ks):
    """tcgen05 kind::tf32 implicit GEMM vs torch fp32: TF32 operand rounding (10-bit mantissa) bounds the
    error at ~1e-3 relative; accumulation is fp32 in TMEM."""
    rng = np.random.default_rng(cin + cout + dims[0])
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w = (rng.standard_normal((cout, cin, ks, ks, ks)) / np.sqrt(cin * ks ** 3)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32) if bias else None
    ref = F.conv3d(torch.from_numpy(x), torch.from_numpy(w), None if b is None else torch.from_numpy(b), padding=ks // 2)
    r = rng.standard_normal(tuple(ref.shape)).astype(np.float32) if res else None
    if res:
        ref = ref + torch.from_numpy(r)
    if act == 1:
        ref = F.relu(ref)
    xd = torch.from_numpy(x[0]).to(DEV).permute(1, 2, 3, 0).contiguous()
    wtc = torch.empty(cout, ks ** 3 * cin, device=DEV)
    wdev = torch.from_numpy(w).to(DEV)
    bdev = torch.from_numpy(b).to(DEV) if bias else None
    S.check(S.lib.sis3d_pack_conv_weight_tc(S.ptr(wdev), cout, cin, ks, S.ptr(wtc), S.stream()))
    out = torch.full(dims + (cout + 4,), 7.0, device=DEV)
    rd = torch.from_numpy(r[0]).to(DEV).permute(1, 2, 3, 0).contiguous() if res else None
    S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(xd), S.ptr(wtc), S.ptr(bdev), S.ptr(rd),
                                     cout if res else 0, 0, S.ptr(out), cout + 4, 4, *dims, cin, cout, ks, None, 0, act, S.stream()))
    torch.cuda.synchronize()
    got = out[..., 4:].permute(3, 0, 1, 2).cpu()
    assert torch.all(out[..., :4] == 7.0)
    err = (got - ref[0]).abs().max().item()
    rel = ((got - ref[0]).norm() / ref[0].norm()).item()
    assert rel < 2e-3 and err < 2e-2, f"rel {rel:.2e} max {err:.2e}"


@pytest.mark.parametrize("cin,cout,dims", [(32, 64, (48, 24, 48)), (64, 64, (48, 24, 48)), (64, 64, (45, 27, 41)), (32, 32, (9, 5, 7)),
                                           (64, 128, (16, 6, 18)), (32, 64, (2, 2, 2))])
def test_conv3d_tc_k2s2(S, cin, cout, dims):
    """2x2x2 / stride-2 conv on the tcgen05 kernel (element-strided TMA boxes), incl. odd extents (floor semantics)."""
    rng = np.random.default_rng(cin + cout + dims[0])
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w = (rng.standard_normal((cout, cin, 2, 2, 2)) / np.sqrt(cin * 8)).astype(np.float32)
    ref = F.relu(F.conv3d(torch.from_numpy(x), torch.from_numpy(w), stride=2))
    xd = torch.from_numpy(x[0]).to(DEV).permute(1, 2, 3, 0).contiguous()
    wd = torch.from_numpy(w).to(DEV)
    wtc = torch.empty(cout, 8 * cin, device=DEV)
    S.check(S.lib.sis3d_pack_conv_weight_tc(S.ptr(wd), cout, cin, 2, S.ptr(wtc), S.stream()))
    od = tuple(d // 2 for d in dims)
    out = torch.full(od + (cout + 4,), 7.0, device=DEV)
    S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(xd), S.ptr(wtc), None, None, 0, 0, S.ptr(out), cout + 4, 4, *dims, cin, cout, 2, None, 0, 1,
                                     S.stream()))
    torch.cuda.synchronize()
    assert torch.all(out[..., :4] == 7.0)
    got = out[..., 4:].permute(3, 0, 1, 2).cpu()
    rel = ((got - ref[0]).norm() / ref[0].norm()).item()
    assert rel < 2e-3 and (got - ref[0]).abs().max().item() < 2e-2, f"rel {rel:.2e}"


@pytest.mark.parametrize("cin,cmid,cout,dims,res", [(32, 32, 32, (17, 9, 11), True), (32, 32, 64, (48, 24, 48), True),
                                                     (32, 32, 64, (9, 3, 5), False), (64, 64, 128, (24, 12, 24), True),
                                                     (64, 64, 128, (7, 5, 6), True)])
def test_conv3d_tc_fused_bottleneck_tail(S, cin, cmid, cout, dims, res):
    """conv2 (3x3x3) -> ReLU -> conv3 (1x1) -> +x -> ReLU in one tcgen05 kernel: bit-identical to the two-kernel TF32 path
    (same operand values and accumulation order), and within TF32 rounding of torch fp32."""
    rng = np.random.default_rng(cin + cout + dims[0])
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w2 = (rng.standard_normal((cmid, cin, 3, 3, 3)) / np.sqrt(cin * 27)).astype(np.float32)
    w3 = (rng.standard_normal((cout, cmid, 1, 1, 1)) / np.sqrt(cmid)).astype(np.float32)
    r = rng.standard_normal((1, cout) + dims).astype(np.float32)
    b2, b3 = rng.standard_normal(cmid).astype(np.float32), rng.standard_normal(cout).astype(np.float32)
    ref = F.conv3d(F.relu(F.conv3d(torch.from_numpy(x), torch.from_numpy(w2), torch.from_numpy(b2), padding=1)), torch.from_numpy(w3),
                   torch.from_numpy(b3))
    if res:
        ref = ref + torch.from_numpy(r)
    ref = F.relu(ref)
    xd = torch.from_numpy(x[0]).to(DEV).permute(1, 2, 3, 0).contiguous()
    rd = torch.from_numpy(r[0]).to(DEV).permute(1, 2, 3, 0).contiguous() if res else None
    w2d, w3d = torch.from_numpy(w2).to(DEV), torch.from_numpy(w3).to(DEV)
    w2t, w3t = torch.empty(cmid, 27 * cin, device=DEV), torch.empty(cout, cmid, device=DEV)
    S.check(S.lib.sis3d_pack_conv_weight_tc(S.ptr(w2d), cmid, cin, 3, S.ptr(w2t), S.stream()))
    S.check(S.lib.sis3d_pack_conv_weight_tc(S.ptr(w3d), cout, cmid, 1, S.ptr(w3t), S.stream()))
    assert S.lib.sis3d_conv3d_k3_tc_fused_supported(cin, cmid, cout) == 1
    out = torch.full(dims + (cout + 4,), 7.0, device=DEV)
    b2d, b3d = torch.from_numpy(b2).to(DEV), torch.from_numpy(b3).to(DEV)
    S.check(S.lib.sis3d_conv3d_k3_tc_fused(S.ptr(xd), S.ptr(w2t), S.ptr(b2d), S.ptr(w3t), S.ptr(b3d), S.ptr(rd), cout if res else 0, 0,
                                           S.ptr(out), cout + 4, 4, *dims, cin, cmid, cout, 1, S.stream()))
    mid = torch.empty(dims + (cmid,), device=DEV)
    two = torch.empty(dims + (cout,), device=DEV)
    S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(xd), S.ptr(w2t), S.ptr(b2d), None, 0, 0, S.ptr(mid), cmid, 0, *dims, cin, cmid, 3, None, 0, 1,
                                     S.stream()))
    S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(mid), S.ptr(w3t), S.ptr(b3d), S.ptr(rd), cout if res else 0, 0, S.ptr(two), cout, 0, *dims, cmid,
                                     cout, 1, None, 0, 1, S.stream()))
    torch.cuda.synchronize()
    assert torch.all(out[..., :4] == 7.0)
    assert torch.equal(out[..., 4:], two), "fused kernel differs from the two-kernel path"
    got = out[..., 4:].permute(3, 0, 1, 2).cpu()
    rel = ((got - ref[0]).norm() / ref[0].norm()).item()
    assert rel < 3e-3, f"rel {rel:.2e}"


def test_conv3d_tc_tile_list(S):
    """Explicit tile list: two crops packed on a zero-separated canvas == per-crop zero-padded conv."""
    rng = np.random.default_rng(3)
    cin = cout = 64
    sizes = [(10, 7, 5), (6, 9, 12)]
    Xc, Yc, Zc = sum(s[0] + 1 for s in sizes), 9, 12
    canvas = torch.zeros(Xc, Yc, Zc, cin)
    crops, x = [], 0
    for s in sizes:
        c = torch.from_numpy(rng.standard_normal(s + (cin,)).astype(np.float32))
        canvas[x:x + s[0], :s[1], :s[2]] = c
        crops.append((x, c))
        x += s[0] + 1
    w = (rng.standard_normal((cout, cin, 3, 3, 3)) / np.sqrt(cin * 27)).astype(np.float32)
    tiles = []
    for (x0, c), s in zip(crops, sizes):
        bx_, by_, bz_ = C.c_int32(), C.c_int32(), C.c_int32()
        S.lib.sis3d_conv3d_tc_brick(1, 3, cin, cout, C.byref(bx_), C.byref(by_), C.byref(bz_))
        for bx in range(0, s[0], bx_.value):
            for by in range(0, s[1], by_.value):
                for bz in range(0, s[2], bz_.value):
                    tiles.append([x0 + bx, by, bz, x0 + s[0], s[1], s[2], 0, 0])
    td = torch.tensor(tiles, dtype=torch.int32, device=DEV)
    wtc = torch.empty(cout, 27 * cin, device=DEV)
    wdev = torch.from_numpy(w).to(DEV)
    S.check(S.lib.sis3d_pack_conv_weight_tc(S.ptr(wdev), cout, cin, 3, S.ptr(wtc), S.stream()))
    out = torch.zeros(Xc, Yc, Zc, cout, device=DEV)
    S.check(S.lib.sis3d_conv3d_k3_tc(S.ptr(canvas.to(DEV)), S.ptr(wtc), None, None, 0, 0, S.ptr(out), cout, 0, Xc, Yc, Zc, cin,
                                     cout, 3, S.ptr(td), len(tiles), 1, S.stream()))
    torch.cuda.synchronize()
    for (x0, c), s in zip(crops, sizes):
        ref = F.relu(F.conv3d(c.permute(3, 0, 1, 2).unsqueeze(0), torch.from_numpy(w), padding=1))[0]
        got = out[x0:x0 + s[0], :s[1], :s[2]].permute(3, 0, 1, 2).cpu()
        assert ((got - ref).norm() / ref.norm()).item() < 2e-3
    # nothing outside the crops was written
    mask = torch.ones(Xc, Yc, Zc, dtype=torch.bool)
    for (x0, c), s in zip(crops, sizes):
        mask[x0:x0 + s[0], :s[1], :s[2]] = False
    assert not out.cpu()[mask].any()


@pytest.mark.parametrize("M,K,N,act", [(200, 8192, 256, 1), (200, 256, 128, 1), (200, 128, 19, 0), (200, 128, 114, 0), (7, 64, 5, 0)])
def test_linear_split_k(S, M, K, N, act):
    rng = np.random.default_rng(M + K + N)
    x = rng.standard_normal((M, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    ref = torch.from_numpy(x) @ torch.from_numpy(w).T + torch.from_numpy(b)
    if act:
        ref = F.relu(ref)
    ldw = (N + 3) // 4 * 4
    packed = torch.empty(K, ldw, device=DEV)
    wdev = torch.from_numpy(w).to(DEV).reshape(N, K, 1, 1, 1).contiguous()
    xdev, bdev = torch.from_numpy(x).to(DEV), torch.from_numpy(b).to(DEV)
    S.check(S.lib.sis3d_pack_conv_weight(S.ptr(wdev), N, K, 1,
                                         S.ptr(packed), S.stream()))
    y = torch.empty(M, N, device=DEV)
    nbytes = int(S.lib.sis3d_linear_workspace_bytes(M, N, K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    for _ in range(2):  # twice: deterministic reduction order
        S.check(S.lib.sis3d_linear(S.ptr(xdev), S.ptr(packed), S.ptr(bdev), S.ptr(y),
                                   M, K, N, act, S.ptr(ws), C.c_size_t(nbytes), S.stream()))
        torch.cuda.synchronize()
        torch.testing.assert_close(y.cpu(), ref, atol=3e-5, rtol=1e-4)


@pytest.mark.parametrize("M,K,N,act", [(200, 8192, 256, 1), (61, 1024, 128, 0), (128, 256, 64, 1), (300, 2048, 32, 1)])
def test_linear_tc_tf32(S, M, K, N, act):
    """Fully connected layer on tcgen05 (2-D TMA operands, split-K, deterministic reduce) vs fp32."""
    rng = np.random.default_rng(M + K + N)
    x = rng.standard_normal((M, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    ref = torch.from_numpy(x) @ torch.from_numpy(w).T + torch.from_numpy(b)
    if act:
        ref = F.relu(ref)
    y = torch.full((M, N), 7.0, device=DEV)
    nbytes = int(S.lib.sis3d_linear_tc_workspace_bytes(M, N, K))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    xd, wd, bd = torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV), torch.from_numpy(b).to(DEV)
    outs = []
    for _ in range(2):
        S.check(S.lib.sis3d_linear_tc(S.ptr(xd), S.ptr(wd), S.ptr(bd), S.ptr(y), M, K, N, act, S.ptr(ws), C.c_size_t(nbytes), S.stream()))
        torch.cuda.synchronize()
        outs.append(y.cpu().clone())
    assert torch.equal(outs[0], outs[1])
    rel = ((outs[0] - ref).norm() / ref.norm()).item()
    assert rel < 2e-3, rel


# ---------------------------------------------------------------- fp16-operand tensor-core conv (kind::f16)
F16_CASES = [  # cin, cout, dims, bias, res, act, ks
    (32, 32, (17, 9, 11), True, False, 1, 3), (32, 64, (24, 12, 24), True, True, 1, 1), (32, 32, (48, 24, 48), True, False, 1, 1),
    (64, 64, (24, 12, 24), True, False, 1, 3), (64, 32, (11, 6, 9), True, False, 1, 1), (128, 128, (11, 6, 10), False, False, 1, 3),
    (128, 256, (24, 12, 24), True, False, 1, 3), (64, 128, (7, 5, 6), True, True, 1, 1), (256, 128, (9, 4, 7), True, False, 0, 1),
    (32, 128, (8, 8, 8), True, True, 1, 1)]


@pytest.mark.parametrize("cin,cout,dims,bias,res,act,ks", F16_CASES)
def test_conv3d_tc_f16_vs_fp32(S, cin, cout, dims, bias, res, act, ks):
    """fp16-stored operands, fp32 accumulation: error bounded by the fp16 rounding of inputs/weights (2^-11 relative);
    both the fp32 output and its fp16 twin are produced in one launch."""
    rng = np.random.default_rng(cin * 7 + cout + dims[0])
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w = (rng.standard_normal((cout, cin, ks, ks, ks)) / np.sqrt(cin * ks ** 3)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32) if bias else None
    ref = F.conv3d(torch.from_numpy(x), torch.from_numpy(w), None if b is None else torch.from_numpy(b), padding=ks // 2)
    r = rng.standard_normal(tuple(ref.shape)).astype(np.float32) if res else None
    if res:
        ref = ref + torch.from_numpy(r)
    if act == 1:
        ref = F.relu(ref)
    xd = torch.from_numpy(x[0]).to(DEV).permute(1, 2, 3, 0).contiguous()
    x16 = torch.empty(dims + (cin,), dtype=torch.float16, device=DEV)
    S.check(S.lib.sis3d_cast_f16(S.ptr(xd), cin, 0, C.c_int64(dims[0] * dims[1] * dims[2]), cin, S.ptr(x16), S.stream()))
    assert torch.equal(x16, xd.half())
    wdev = torch.from_numpy(w).to(DEV)
    bdev = torch.from_numpy(b).to(DEV) if bias else None
    w16 = torch.empty(cout, ks ** 3 * cin, dtype=torch.float16, device=DEV)
    S.check(S.lib.sis3d_pack_conv_weight_tc_f16(S.ptr(wdev), cout, cin, ks, S.ptr(w16), S.stream()))
    out = torch.full(dims + (cout + 4,), 7.0, device=DEV)
    out16 = torch.full(dims + (cout + 4,), 7.0, dtype=torch.float16, device=DEV)
    rd = torch.from_numpy(r[0]).to(DEV).permute(1, 2, 3, 0).contiguous() if res else None
    S.check(S.lib.sis3d_conv3d_tc_f16(S.ptr(x16), S.ptr(w16), S.ptr(bdev), S.ptr(rd), cout if res else 0, 0, S.ptr(out), S.ptr(out16),
                                      cout + 4, 4, *dims, cin, cout, ks, None, 0, act, S.stream()))
    torch.cuda.synchronize()
    got = out[..., 4:].permute(3, 0, 1, 2).cpu()
    assert torch.all(out[..., :4] == 7.0) and torch.all(out16[..., :4] == 7.0)
    rel = ((got - ref[0]).norm() / ref[0].norm()).item()
    assert rel < 1.5e-3, f"rel {rel:.2e}"
    assert torch.equal(out16[..., 4:], out[..., 4:].half())
    # fp16-only output (no fp32 store)
    out16b = torch.zeros(dims + (cout,), dtype=torch.float16, device=DEV)
    S.check(S.lib.sis3d_conv3d_tc_f16(S.ptr(x16), S.ptr(w16), S.ptr(bdev), S.ptr(rd), cout if res else 0, 0, None, S.ptr(out16b),
                                      cout, 0, *dims, cin, cout, ks, None, 0, act, S.stream()))
    torch.cuda.synchronize()
    assert torch.equal(out16b, out[..., 4:].half())


def test_simt_conv_and_sparse_fp16_twin(S):
    rng = np.random.default_rng(12)
    cin, cout, dims = 2, 32, (10, 8, 6)
    x = rng.standard_normal((1, cin) + dims).astype(np.float32)
    w = (rng.standard_normal((cout, cin, 2, 2, 2)) / 4).astype(np.float32)
    od = tuple(d // 2 for d in dims)
    xd, wd = torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV)
    packed = torch.empty(8 * cin, cout, device=DEV)
    S.check(S.lib.sis3d_pack_conv_weight(S.ptr(wd), cout, cin, 2, S.ptr(packed), S.stream()))
    out = torch.zeros(od + (cout,), device=DEV)
    out16 = torch.zeros(od + (cout,), dtype=torch.float16, device=DEV)
    X, Y, Z = dims
    regions, tiles = S.make_regions([dict(in_off=0, out_off=0, in_dim=dims, out_dim=od, in_stride=(Y * Z, Z, 1))], DEV)
    S.check(S.lib.sis3d_conv3d_ex(S.ptr(xd), C.c_int64(X * Y * Z), S.ptr(packed), None, None, 0, 0, S.ptr(out), S.ptr(out16), cout, 0,
                                  S.ptr(regions), 1, tiles, cin, cout, 2, 2, 0, 1, S.stream()))
    torch.cuda.synchronize()
    ref = F.relu(F.conv3d(torch.from_numpy(x), torch.from_numpy(w), stride=2))[0].permute(1, 2, 3, 0)
    torch.testing.assert_close(out.cpu(), ref, atol=2e-5, rtol=1e-4)
    assert torch.equal(out16, out.half())
