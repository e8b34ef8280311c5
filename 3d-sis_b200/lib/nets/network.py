"""`Network`: the TEST-mode forward of 3D-SIS on libsis3d kernels.

Public surface kept from the reference (lib/nets/network.py): `init_modules()`, `load_state_dict()`
with the reference's parameter names/shapes, `forward(blobs, 'TEST', killing_inds)`, the
`_predictions` dict (`rois, roi_scores, level_inds, cls_score, cls_pred, cls_prob, bbox_pred,
mask_pred`), `_scene_info`, and `mask_backbone(scene_crop, imageft)`.

Everything between the input blobs and `_predictions` runs as hand-written CUDA (csrc/*.cu) on VC
(channels-last) activations; nn.Module is used only as the parameter container so checkpoints of the
reference load unchanged.  Training mode is out of scope (inference-only hot path).
"""
from __future__ import annotations

import ctypes as C
import gc
import math
import os
import weakref
from typing import NamedTuple, Optional

import numpy as np
import torch
from torch import nn

from lib import _sis3d as S
from lib.layer_utils import projection as proj
from lib.layer_utils.generate_anchors import read_anchor_sizes
from lib.layer_utils.proposal_layer import rpn_proposals
from lib.utils.config import cfg


class Act:
    """A voxel activation: tensor + spatial dims + channels; layout 'vc' ([X,Y,Z,C]) or 'ncdhw'."""
    __slots__ = ("t", "dims", "C", "layout", "ld", "coff", "h")

    def __init__(self, t, dims, Cn, layout="vc", ld=None, coff=0, h=None):
        self.t, self.dims, self.C, self.layout = t, tuple(int(d) for d in dims), int(Cn), layout
        self.ld, self.coff = int(ld if ld is not None else Cn), int(coff)
        self.h = h  # optional dense fp16 twin [X,Y,Z,C] (fp16-operand tensor-core mode); `t` may be None when only `h` exists

    @property
    def nvox(self):
        return self.dims[0] * self.dims[1] * self.dims[2]


def _declare(root, dotted, shape, fan_in):
    """Register parameter `dotted` (e.g. 'geometry1.2.conv1.weight') on nested container modules,
    default-initialised like torch's Conv/Linear (U(-1/sqrt(fan_in), 1/sqrt(fan_in)))."""
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    bound = 1.0 / math.sqrt(fan_in)
    mod.register_parameter(parts[-1], nn.Parameter(torch.empty(shape).uniform_(-bound, bound), requires_grad=False))


def _declare_tensor(root, dotted, tensor, kind):
    """Register `tensor` as parameter / buffer `dotted` on nested container modules (state_dict key == dotted)."""
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    if kind == "param":
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))
    else:
        mod.register_buffer(parts[-1], tensor)


class _MaskList:
    """Sequence of per-RoI mask tensors [1, num_classes, w, h, l] (the reference's `mask_pred[i]` list,
    lib/nets/network.py:303-317) as lazily created views of the packed [total_voxels, num_classes] output."""

    def __init__(self, packed, offs, sizes, ncls):
        self.packed, self.offs, self.sizes, self.ncls = packed, offs, sizes, ncls

    def __len__(self):
        return len(self.sizes)

    def __getitem__(self, j):
        if isinstance(j, slice):
            return [self[i] for i in range(*j.indices(len(self)))]
        if j < 0:
            j += len(self)
        if not 0 <= j < len(self):
            raise IndexError(j)
        w, h, l = (int(v) for v in self.sizes[j])
        m = self.packed[int(self.offs[j]) * self.ncls:int(self.offs[j + 1]) * self.ncls].view(w, h, l, self.ncls)
        return m.permute(3, 0, 1, 2).unsqueeze(0)  # view in the reference layout

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def __eq__(self, other):
        return list(self) == other if isinstance(other, list) else NotImplemented


class Packed(NamedTuple):
    """One layer's weights as the kernels take them."""
    simt: torch.Tensor  # [k^3 C_in][ldw] for the CUDA-core kernels
    bias: Optional[torch.Tensor]
    cout: int
    cin: int
    ks: int
    tc: dict  # tensor-core operand format ('tf32' | 'tf32x3' | 'f16x3' | 'fp16') -> packed weight


# tensor-core operand format -> pack entry point, dtype, packed rows per output channel (tf32x3: hi rows, then lo rows;
# f16x3: [32 hi | 32 lo] halves per 32-channel K slice, i.e. the same bytes as two fp16 rows)
_TC_PACK = {"tf32": ("sis3d_pack_conv_weight_tc", torch.float32, 1),
            "tf32x3": ("sis3d_pack_conv_weight_tc_x3", torch.float32, 2),
            "f16x3": ("sis3d_pack_conv_weight_tc_h3", torch.float16, 2),
            "fp16": ("sis3d_pack_conv_weight_tc_f16", torch.float16, 1)}
# format -> entry point and timing label: convolutions (trailing arguments: the TF32 kernel also takes tile lists), fused
# bottleneck tails, fully connected layers (+ workspace size query; None = the CUDA-core kernel)
_CONV_TC = {"tf32": ("sis3d_conv3d_k3_tc", "conv_tc", (None, 0)),
            "tf32x3": ("sis3d_conv3d_k3_tc_x3", "conv_tc_x3", ()),
            "f16x3": ("sis3d_conv3d_k3_tc_h3", "conv_tc_h3", ())}
_FUSED_TC = {"tf32": ("sis3d_conv3d_k3_tc_fused", "conv_tc_fused"),
             "tf32x3": ("sis3d_conv3d_k3_tc_fused_x3", "conv_tc_fused_x3"),
             "f16x3": ("sis3d_conv3d_k3_tc_fused_h3", "conv_tc_fused_h3")}
_LINEAR = {None: ("sis3d_linear", "sis3d_linear_workspace_bytes", "linear"),
           "tf32": ("sis3d_linear_tc", "sis3d_linear_tc_workspace_bytes", "linear_tc"),
           "tf32x3": ("sis3d_linear_tc_x3", "sis3d_linear_tc_workspace_bytes", "linear_tc_x3"),
           "f16x3": ("sis3d_linear_tc_h3", "sis3d_linear_tc_workspace_bytes", "linear_tc_h3")}


# ---------------------------------------------------------------------------------------------------- conv routing
def fp16_twins(math):
    """Static stage: whether activations that feed tensor-core layers are kept as dense fp16 twins (and an fp32 copy only
    where a consumer needs one), and the sparse back-projection writes one."""
    return math == "fp16"


def tc_format(math, formats, op="conv", tc_ok=True, out32=True, twin=False):
    """Static stage: the tensor-core operand format a layer runs in, or None for the fp32 CUDA-core kernel.

    math: the static-stage conv math; formats: the formats packed for the layer (for op 'fused', the bottleneck's conv2 +
    conv3 in one kernel: those both convs have); tc_ok: geometry, input layout and activation fit the tensor-core kernel;
    out32 / twin: the conv writes an fp32 output / an fp16 twin.  A conv in 'fp16' math without fp16 weights runs the TF32
    kernel when it writes fp32 only; fully connected layers and fused tails have no fp16-operand kernel."""
    if not tc_ok:
        return None
    if math in formats and (op == "conv" or math != "fp16"):
        return math
    if op == "conv" and math == "fp16" and "tf32" in formats and out32 and not twin:
        return "tf32"
    return None


def mask_stage_code(mask_math, formats):
    """The ragged mask stage's `math` (sis3d_mask_stage_launch): 2 = fp16-operand tensor cores on an fp16 canvas, 1 = TF32
    tensor cores, 0 = CUDA-core; formats: those packed for mask_backbone.geometry.2."""
    if mask_math == "fp16" and "tf32" in formats and "fp16" in formats:
        return 2
    return 1 if mask_math in ("tf32", "fp16") and "tf32" in formats else 0


def _pack_tc(w, cout, cin, ks, formats):
    """fp32 weight [cout][cin][ks][ks][ks] -> {format: packed tensor-core weight} for each of `formats`."""
    out = {}
    for f in formats:
        sym, dtype, rows = _TC_PACK[f]
        t = torch.empty(rows * cout, ks ** 3 * cin, dtype=dtype, device=w.device)
        S.check(getattr(S.lib, sym)(S.ptr(w), cout, cin, ks, S.ptr(t), S.stream()), f"pack_{f}")
        out[f] = t
    return out


def _conv_tc_formats(cin, cout, ks):
    """Formats a 3-D convolution is packed in: fp16 storage needs 32 or a multiple of 64 input channels and has no 2x2x2
    kernel."""
    if ks not in (1, 2, 3) or not S.lib.sis3d_conv3d_k3_tc_supported(cin, cout):
        return ()
    return ("tf32", "tf32x3", "f16x3") + (("fp16",) if ks != 2 and (cin % 64 == 0 or cin == 32) else ())


class Network(nn.Module):
    # layer programs of the concrete backbones are provided by subclasses (lib/nets/backbones.py)
    SPEC = None

    def __init__(self):
        super().__init__()
        self._predictions = {}
        self._feat_stride = [4, 4, 4]
        self._packed = {}  # layer name -> Packed
        self._packed_version = None
        self._region_cache = {}
        self._const_cache = {}
        self._keep_debug = False
        # conv math (see set_conv_math).  Default 'exact': error-compensated split products (fp32-class accuracy, tcgen05) in the
        # static stage -- everything that decides an integer output: proposal order, NMS keep list, class argmax, crop
        # bounds -- and fp16-stored operands in the ragged mask stage, whose outputs carry the 1e-3 tolerance.
        self.set_conv_math(os.environ.get("SIS3D_CONV_MATH", str(cfg.get("CONV_MATH", "exact"))).lower())
        self._graphs = {}
        self._slots = []
        self._branches = os.environ.get("SIS3D_BRANCHES", "1") != "0"
        self._replayed_kernels = 0  # libsis3d kernels executed through CUDA-graph replays
        self._sparse_color = os.environ.get("SIS3D_SPARSE_COLOR", "1") != "0"
        self._fuse_bneck = os.environ.get("SIS3D_FUSE_BNECK", "1") != "0"
        self._tc_k2s2 = os.environ.get("SIS3D_TC_K2S2", "1") != "0"
        # host waits yield the core instead of spinning: with one process per GPU on a CPU-quota'd node, eight spinning
        # waiters plus the Python loops would eat the whole quota (cgroup throttling stalls every rank at once)
        # (spinning is ~9 % faster on an otherwise idle host, so it stays the default while cores are plentiful)
        bs = os.environ.get("SIS3D_BLOCKING_SYNC")
        if bs is None:
            try:
                cores = len(os.sched_getaffinity(0))
                with open("/sys/fs/cgroup/cpu.max") as f:
                    quota, period = f.read().split()
                if quota != "max":
                    cores = min(cores, max(1, int(quota) // int(period)))
            except (OSError, ValueError, AttributeError):
                cores = os.cpu_count() or 1
            self._blocking_sync = cores < 3 * int(os.environ.get("LOCAL_WORLD_SIZE", "1"))
        else:
            self._blocking_sync = bs != "0"
        self._pack_dirty = True
        self._arena = {}  # grow-only device/pinned workspaces for the ragged (per-scene sized) stage
        self._use_graph = os.environ.get("SIS3D_CUDA_GRAPH", "1") != "0"
        # a shape is captured the SIS3D_GRAPH_AFTER-th time it is seen (whole-scene inference meets many one-off shapes: those
        # run eagerly), and every stream slot keeps at most SIS3D_GRAPH_CACHE captured shapes (LRU; a graph owns its static
        # buffers and a private memory pool, so an unbounded cache would grow until OOM)
        self._graph_after = max(1, int(os.environ.get("SIS3D_GRAPH_AFTER", "2")))
        self._graph_cache = max(1, int(os.environ.get("SIS3D_GRAPH_CACHE", "4")))
        self._shape_seen = {}
        self._prof = None  # name -> [(start_event, end_event)] when per-kernel timing is on (bench.py)

    # ------------------------------------------------------------------ parameters
    def _declare_conv(self, name, cout, cin, ks, bias):
        _declare(self, name + ".weight", (cout, cin, ks, ks, ks), cin * ks ** 3)
        if bias:
            _declare(self, name + ".bias", (cout,), cin * ks ** 3)

    def _declare_bottleneck(self, name, inpl, planes):
        self._declare_conv(name + ".conv1", planes, inpl, 1, True)
        self._declare_conv(name + ".conv2", planes, planes, 3, True)
        self._declare_conv(name + ".conv3", inpl, planes, 1, True)

    def _declare_linear(self, name, cout, cin):
        _declare(self, name + ".weight", (cout, cin), cin)
        _declare(self, name + ".bias", (cout,), cin)

    def _declare_stack(self, prefix, spec):
        for op in spec:
            if op[0] in ("k2s2", "k3"):
                self._declare_conv(f"{prefix}.{op[1]}", op[3], op[2], 2 if op[0] == "k2s2" else 3, False)
            elif op[0] == "bneck":
                self._declare_bottleneck(f"{prefix}.{op[1]}", op[2], op[3])

    def _init_backbone_classifier(self):
        raise NotImplementedError

    def init_modules(self):
        """Declare every parameter of the 3D model (reference: network.py:35-64)."""
        self._init_backbone_classifier()
        if cfg.USE_RPN:
            for lvl in (1, 2, 3):
                A = cfg["NUM_ANCHORS_LEVEL%d" % lvl]
                if A:
                    self._declare_conv(f"rpn_net_level{lvl}", cfg.RPN_CHANNELS, 128, 3, True)
                    self._declare_conv(f"rpn_cls_score_net_level{lvl}.0", 2 * A, cfg.RPN_CHANNELS, 1, True)
                    self._declare_conv(f"rpn_bbox_pred_net_level{lvl}", 6 * A, cfg.RPN_CHANNELS, 1, True)
        if cfg.USE_CLASS:
            self._declare_linear("classifier_cls_score_net", cfg.NUM_CLASSES, 128)
            self._declare_linear("classifier_bbox_pred_net", cfg.NUM_CLASSES * 6, 128)
        if cfg.USE_MASK:
            from lib.nets import backbones
            self.mask_backbone = getattr(backbones, cfg.MASK_BACKBONE)()
            # weak back-reference: no parent<->child cycle, so a dropped Network (graphs, streams, arenas) is freed by
            # reference counting right away instead of by a later cyclic GC pass in the middle of someone else's capture
            self.mask_backbone._owner = weakref.ref(self)
        if cfg.USE_IMAGES and not cfg.USE_IMAGES_GT:
            self._declare_enet()

    def _declare_enet(self):
        """2-D ENet encoder (SURVEY 8f2; reference: network.py:62-63 -> enet.create_enet_for_3d, enet.py:697-715): parameters and
        BatchNorm buffers under the reference's state_dict names (lib/nets/enet_keys.py), default-initialised, then overwritten
        by cfg.PRETRAINED_ENET_PATH when that file exists (the reference loads it at this point too).  The forward runs on the
        sis3d_enet_* kernels (lib/nets/enet.py); image_enet_classification is kept only for the checkpoint contract."""
        from lib.nets.enet_keys import ENET_KEYS
        n2d = int(cfg.NUM_2D_CLASSES)
        names = {k[0] for k in ENET_KEYS}
        enc = []
        for name, shape, kind, dt in ENET_KEYS:
            if name.startswith("image_enet_classification"):
                shape = (n2d,) + tuple(shape[1:])
            if dt == "int64":
                t = torch.zeros(shape, dtype=torch.int64)
            elif name.endswith("running_var"):
                t = torch.ones(shape)
            elif name.endswith(("running_mean", ".bias")):
                t = torch.zeros(shape)
            elif len(shape) == 4:
                bound = 1.0 / math.sqrt(shape[1] * shape[2] * shape[3])
                t = torch.empty(shape).uniform_(-bound, bound)
            else:  # 1-D weight: BatchNorm scale (has running statistics beside it) or PReLU slope
                t = torch.ones(shape) if name[:-len("weight")] + "running_mean" in names else torch.full(shape, 0.25)
            _declare_tensor(self, name, t, kind)
            if not name.startswith("image_enet_classification") and not name.endswith("num_batches_tracked"):
                enc.append(name)
        self.__dict__["_enet_names"] = enc
        path = str(cfg.get("PRETRAINED_ENET_PATH", "") or "")
        if path and os.path.exists(path):
            src = torch.load(path, map_location="cpu")  # plain create_enet keys ('0.0.weight', ...), same order as ENET_KEYS
            own = dict(self.named_parameters())
            own.update(dict(self.named_buffers()))
            if len(src) != len(ENET_KEYS):
                raise S.Sis3dError(f"{path}: {len(src)} tensors, the ENet of lib/nets/enet.py has {len(ENET_KEYS)}")
            with torch.no_grad():
                for (name, _, _, _), v in zip(ENET_KEYS, src.values()):
                    own[name].copy_(v)

    # ------------------------------------------------------------------ packed weights
    def load_state_dict(self, *a, **k):
        self._pack_dirty = True
        return super().load_state_dict(*a, **k)

    def _apply(self, fn, *a, **k):  # .cuda() / .to() / .float() move parameters -> repack
        self._pack_dirty = True
        return super()._apply(fn, *a, **k)

    def _ws(self, name, numel, dtype, dev, pinned=False):
        """Grow-only workspace: steady-state forwards never hit cudaMalloc for per-scene sized buffers."""
        t = self._arena.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            cap = int(numel * 1.5) + 1024
            t = torch.empty(cap, dtype=dtype, pin_memory=True) if pinned else torch.empty(cap, dtype=dtype, device=dev)
            self._arena[name] = t
        return t[:numel]

    def _version(self):
        v = tuple((n, p._version, p.data_ptr()) for n, p in self.named_parameters())
        if self.__dict__.get("_enet_names"):  # BatchNorm statistics of the 2-D encoder are buffers
            v += tuple((n, b._version, b.data_ptr()) for n, b in self.named_buffers())
        return v

    MATH_MODES = {  # mode -> (static-stage conv math, mask-stage conv math)
        "exact": ("f16x3", "fp16"),    # default: integer outputs equal the fp32 path, masks within 1e-3
        "f16x3": ("f16x3", "tf32"),    # error-compensated fp16 split (3 kind::f16 MMAs per product, fp32-class accuracy)
        "tf32x3": ("tf32x3", "tf32"),  # the same compensation with a TF32 split (3 kind::tf32 MMAs: 2.5x slower tensor pipe)
        "mixed": ("tf32", "fp16"),     # fastest; detections equal the reference only up to near-tied scores
        "tf32": ("tf32", "tf32"),
        "fp16": ("fp16", "fp16"),
        "fp32": ("fp32", "fp32"),      # CUDA-core kernels throughout
    }

    def set_conv_math(self, mode):
        """'exact' (error-compensated fp16-split static stage + fp16-operand mask stage) | 'f16x3' | 'tf32x3' | 'mixed' (TF32 +
        fp16) | 'tf32' | 'fp16' | 'fp32' (CUDA-core path)."""
        if mode not in self.MATH_MODES:
            raise S.Sis3dError(f"unknown conv math {mode!r} ({' | '.join(self.MATH_MODES)})")
        self.__dict__["_math"], self.__dict__["_mask_math"] = self.MATH_MODES[mode]
        self.__dict__["_math_mode"] = mode

    def _ensure_packed(self):
        d = self.__dict__
        if not d["_pack_dirty"] and d["_packed_version"] is not None:  # per-scene fast path: no module traversal
            return
        if not torch.cuda.is_available():
            raise S.Sis3dError("the sm_100a hot path needs a CUDA device (no CPU fallback)")
        if next(self.parameters()).device.type != "cuda":
            self.cuda()
        d["_dev"] = next(self.parameters()).device
        v = self._version()
        self._pack_dirty = False
        if v == self._packed_version:
            return
        self._packed = {}
        params = dict(self.named_parameters())
        self.__dict__["_enet"] = None
        if self.__dict__.get("_enet_names"):
            from lib.nets.enet import EnetEncoder
            sd = dict(params)
            sd.update(dict(self.named_buffers()))
            self.__dict__["_enet"] = EnetEncoder([sd[n].detach() for n in self._enet_names], d["_dev"])
        for name, p in params.items():
            if not name.endswith(".weight") or name.startswith("image_enet_"):
                continue
            base = name[:-7]
            w = p.detach().float().contiguous()
            if w.dim() == 2:
                w = w.reshape(w.shape[0], w.shape[1], 1, 1, 1)
            cout, cin, ks = w.shape[0], w.shape[1], w.shape[2]
            ldw = (cout + 3) // 4 * 4
            packed = torch.empty(ks ** 3 * cin, ldw, dtype=torch.float32, device=w.device)
            S.check(S.lib.sis3d_pack_conv_weight(S.ptr(w), cout, cin, ks, S.ptr(packed), S.stream()), "pack")
            if p.dim() == 5:
                tc = _pack_tc(w, cout, cin, ks, _conv_tc_formats(cin, cout, ks))
            elif cin >= 1024 and S.lib.sis3d_linear_tc_supported(cin, cout):
                # nn.Linear [N][K] is already K-major for the TF32 GEMM; the split formats pack it as a 1x1 conv
                tc = dict(tf32=p.detach(), **_pack_tc(w, cout, cin, 1, ("tf32x3", "f16x3")))
            else:
                tc = {}
            b = params.get(base + ".bias")
            self._packed[base] = Packed(packed, None if b is None else b.detach().float().contiguous(), cout, cin, ks, tc)
        for lvl in (1, 2, 3):  # both RPN heads of a level as ONE 1x1 conv: [2A | 6A] output channels, zero-padded to a
            # tensor-core friendly width (32/64/128k) so the merged head runs on the tcgen05 kernel as well
            c, b = f"rpn_cls_score_net_level{lvl}.0", f"rpn_bbox_pred_net_level{lvl}"
            if c + ".weight" in params and b + ".weight" in params:
                w = torch.cat([params[c + ".weight"], params[b + ".weight"]], 0).detach().float()
                bias = torch.cat([params[c + ".bias"], params[b + ".bias"]], 0).detach().float()
                cout, cin = w.shape[0], w.shape[1]
                cpad = 32 if cout <= 32 else (64 if cout <= 64 else (cout + 127) // 128 * 128)
                wp = torch.zeros(cpad, cin, 1, 1, 1, dtype=torch.float32, device=w.device)
                wp[:cout] = w
                bp = torch.zeros(cpad, dtype=torch.float32, device=w.device)
                bp[:cout] = bias
                packed = torch.empty(cin, cpad, dtype=torch.float32, device=w.device)
                S.check(S.lib.sis3d_pack_conv_weight(S.ptr(wp), cpad, cin, 1, S.ptr(packed), S.stream()), "pack")
                self._packed[f"rpn_heads_level{lvl}"] = Packed(packed, bp, cpad, cin, 1,
                                                               _pack_tc(wp, cpad, cin, 1, _conv_tc_formats(cin, cpad, 1)))
        torch.cuda.current_stream().synchronize()
        self._packed_version = v
        # captured graphs hold the addresses of the previous packed weights: drop them (re-captured on next use)
        self.__dict__["_graphs"] = {}
        for sl in self._slots:
            sl["graphs"].clear()

    # ------------------------------------------------------------------ per-kernel timing hooks
    def _rec(self, name):
        if self._prof is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return name, e

    def _rec_end(self, tok):
        if tok is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._prof.setdefault(tok[0], []).append((tok[1], e))

    # ------------------------------------------------------------------ primitive ops
    def _regions_single(self, x: Act, out_dims, stride):
        key = ("single", x.dims, x.C, x.layout, x.ld, tuple(out_dims), stride)
        hit = self._region_cache.get(key)
        if hit is None:
            X, Y, Z = x.dims
            strides = (Y * Z * x.ld, Z * x.ld, x.ld) if x.layout == "vc" else (Y * Z, Z, 1)
            hit = S.make_regions([dict(in_off=0, out_off=0, res_off=0, in_dim=x.dims, out_dim=out_dims,
                                       in_stride=strides)], x.t.device)
            self._region_cache[key] = hit
        return hit

    def _half(self, x: Act):
        """fp16 twin of an activation (cast once, cached on the Act)."""
        if x.h is None:
            x.h = torch.empty(*x.dims, x.C, dtype=torch.float16, device=x.t.device)
            tok = self._rec("cast_f16")
            S.check(S.lib.sis3d_cast_f16(S.ptr(x.t), x.ld, x.coff, C.c_int64(x.nvox), x.C, S.ptr(x.h), S.stream()), "cast_f16")
            self._rec_end(tok)
        return x.h

    def _conv(self, x: Act, name, stride=1, pad=None, act=0, residual: Act = None, out: Act = None, out_dims=None,
              want32=True, want16=False):
        """One convolution, on the kernel tc_format picks.  want32/want16 choose which of the fp32 output / dense fp16 twin
        are produced where fp16_twins holds (the twin feeds the next tensor-core layer); elsewhere the output is fp32."""
        r = self._packed[name]
        cout, cin, ks = r.cout, r.cin, r.ks
        if cin != x.C:
            raise S.Sis3dError(f"{name}: expected {cin} input channels, got {x.C}")
        if pad is None:
            pad = 1 if ks == 3 else 0
        if out_dims is None:
            out_dims = tuple(d // 2 for d in x.dims) if stride == 2 else x.dims
        dev = (x.t if x.t is not None else x.h).device
        if ks == 2:  # the 2x2x2 / stride-2 downsampling convs run on the tensor cores too (element-strided TMA boxes)
            geom_ok = stride == 2 and pad == 0 and min(x.dims) >= 2 and self._tc_k2s2
        else:
            geom_ok = stride == 1 and pad == (1 if ks == 3 else 0)
        tc_ok = geom_ok and x.layout == "vc" and x.ld == x.C and x.coff == 0 and act in (0, 1)
        if not fp16_twins(self._math):
            want32, want16 = True, False
        if out is None:
            t32 = torch.empty(*out_dims, cout, dtype=torch.float32, device=dev) if want32 else None
            out = Act(t32, out_dims, cout)
        want16 = want16 and out.ld == cout and out.coff == 0  # the twin shares the geometry of the fp32 output
        if want16:
            out.h = torch.empty(*out_dims, cout, dtype=torch.float16, device=dev)
        h_ptr = S.ptr(out.h) if want16 else None
        res_args = (S.ptr(residual.t) if residual is not None else None, residual.ld if residual is not None else 0,
                    residual.coff if residual is not None else 0)
        fmt = tc_format(self._math, r.tc, "conv", tc_ok, out32=out.t is not None or not want16, twin=want16)
        if fmt == "fp16":
            tok = self._rec(f"conv_tc16[{name}]")
            S.check(S.lib.sis3d_conv3d_tc_f16(S.ptr(self._half(x)), S.ptr(r.tc[fmt]), S.ptr(r.bias), *res_args,
                                              S.ptr(out.t) if out.t is not None else None, h_ptr, out.ld, out.coff, *x.dims,
                                              cin, cout, ks, None, 0, act, S.stream()), f"conv3d_tc_f16[{name}]")
            self._rec_end(tok)
            return out
        if x.t is None:
            raise S.Sis3dError(f"{name}: this layer needs the fp32 activation but only the fp16 twin was produced")
        if out.t is None and h_ptr is None:
            out.t = torch.empty(*out_dims, cout, dtype=torch.float32, device=dev)
        if fmt is not None:
            sym, label, tiles = _CONV_TC[fmt]
            tok = self._rec(f"{label}[{name}]")
            S.check(getattr(S.lib, sym)(S.ptr(x.t), S.ptr(r.tc[fmt]), S.ptr(r.bias), *res_args, S.ptr(out.t), out.ld, out.coff,
                                        *x.dims, cin, cout, ks, *tiles, act, S.stream()), f"{sym}[{name}]")
            self._rec_end(tok)
            return out
        regions, n_tiles = self._regions_single(x, out_dims, stride)
        in_sc = 1 if x.layout == "vc" else x.nvox
        xin = x.t if x.coff == 0 else x.t.reshape(-1)[x.coff:]
        tok = self._rec(f"conv[{name}]")
        S.check(S.lib.sis3d_conv3d_ex(S.ptr(xin), C.c_int64(in_sc), S.ptr(r.simt), S.ptr(r.bias), *res_args,
                                      S.ptr(out.t) if out.t is not None else None, h_ptr, out.ld, out.coff, S.ptr(regions),
                                      regions.numel() // S.REGION_BYTES, n_tiles, cin, cout, ks, stride, pad, act, S.stream()),
                f"conv3d[{name}]")
        self._rec_end(tok)
        return out

    def _linear(self, x, name, act):
        """y = act(x W^T + b) through a split-K kernel (classifier MLP + heads)."""
        r = self._packed[name]
        M = x.shape[0]
        y = torch.empty(M, r.cout, dtype=torch.float32, device=x.device)
        fmt = tc_format(self._math, r.tc, "linear")
        sym, ws_sym, label = _LINEAR[fmt]
        nbytes = int(getattr(S.lib, ws_sym)(M, r.cout, r.cin))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        tok = self._rec(f"{label}[{name}]")
        S.check(getattr(S.lib, sym)(S.ptr(x), S.ptr(r.tc[fmt] if fmt else r.simt), S.ptr(r.bias), S.ptr(y), M, r.cin, r.cout, act,
                                    S.ptr(ws), C.c_size_t(nbytes), S.stream()), f"{label}[{name}]")
        self._rec_end(tok)
        return y

    def _bottleneck(self, x: Act, name, out: Act = None):
        """1x1 -> relu -> 3x3x3 -> relu -> 1x1 (+x) -> relu  (reference: backbones.py:28-40).  In 'fp16' math the two inner
        activations exist only as fp16 (they feed tensor-core layers only); the block output is fp32 (+ fp16 twin when it
        is a dense tensor, for the next block's first conv)."""
        y = self._conv(x, name + ".conv1", act=1, want32=False, want16=True)
        n2, n3 = name + ".conv2", name + ".conv3"
        r2, r3 = self._packed[n2], self._packed[n3]
        fused_ok = (self._fuse_bneck and y.t is not None and y.ld == y.C and y.coff == 0
                    and bool(S.lib.sis3d_conv3d_k3_tc_fused_supported(r2.cin, r2.cout, r3.cout)))
        fmt = tc_format(self._math, r2.tc.keys() & r3.tc.keys(), "fused", fused_ok)
        if fmt is not None:
            # conv2 + conv3 (+x, ReLU) in one tcgen05 kernel: the cmid-wide activation never leaves the SM
            if out is None:
                out = Act(torch.empty(*y.dims, r3.cout, dtype=torch.float32, device=y.t.device), y.dims, r3.cout)
            sym, label = _FUSED_TC[fmt]
            tok = self._rec(f"{label}[{name}]")
            S.check(getattr(S.lib, sym)(S.ptr(y.t), S.ptr(r2.tc[fmt]), S.ptr(r2.bias), S.ptr(r3.tc[fmt]), S.ptr(r3.bias),
                                        S.ptr(x.t), x.ld, x.coff, S.ptr(out.t), out.ld, out.coff, *y.dims, r2.cin, r2.cout,
                                        r3.cout, 1, S.stream()), f"{sym}[{name}]")
            self._rec_end(tok)
            return out
        y = self._conv(y, n2, act=1, want32=False, want16=True)
        return self._conv(y, n3, act=1, residual=x, out=out, want32=True, want16=True)

    def _pool(self, x: Act, out: Act = None):
        if out is None:
            out = Act(torch.empty(*x.dims, x.C, dtype=torch.float32, device=x.t.device), x.dims, x.C)
        if x.ld != x.C or x.coff:
            raise S.Sis3dError("maxpool3 expects a dense VC input")
        tok = self._rec("maxpool3")
        S.check(S.lib.sis3d_maxpool3(S.ptr(x.t), S.ptr(out.t), out.ld, out.coff, *x.dims, x.C, S.stream()), "maxpool3")
        self._rec_end(tok)
        return out

    def _run_stack(self, x: Act, prefix, spec, final_out=None):
        """Execute a backbone stage program; the last op writes into `final_out` (a slice of the
        concatenated level-1 tensor) when given."""
        for i, op in enumerate(spec):
            dst = final_out(x, op) if (final_out is not None and i == len(spec) - 1) else None
            if op[0] == "k2s2":
                x = self._conv(x, f"{prefix}.{op[1]}", stride=2, pad=0, act=1, out=dst, want16=True)
            elif op[0] == "k3":
                x = self._conv(x, f"{prefix}.{op[1]}", act=1, out=dst, want16=True)
            elif op[0] == "bneck":
                x = self._bottleneck(x, f"{prefix}.{op[1]}", out=dst)
            elif op[0] == "pool":
                x = self._pool(x, out=dst)
        return x

    # ------------------------------------------------------------------ stages of the forward
    def _const(self, key, builder):
        v = self._const_cache.get(key)
        if v is None:
            v = builder()
            self._const_cache[key] = v
        return v

    def _backproject(self, blobs, killing_inds, dims, dev, fused=None):
        """Views -> VC feature volume (reference: trainval.py:797-820 + network.py:194-239)."""
        w, h = int(cfg.DEPTH_SHAPE[0]), int(cfg.DEPTH_SHAPE[1])
        if fused is not None:
            feats = fused["feats"]
        else:
            feats = blobs["nearest_images"]["images"][0]
            feats = feats.to(dev, torch.float32, non_blocking=True)
        if not cfg.USE_IMAGES_GT:
            # raw images [n,3,H,W] -> ENet features [n,128,H/8,W/8] on the sis3d_enet_* kernels (reference: network.py:204-205)
            if self.__dict__.get("_enet") is None:
                raise S.Sis3dError("USE_IMAGES_GT=False but the 2-D ENet encoder was not declared (init_modules with this cfg)")
            tok = self._rec("enet_encoder")
            feats = self._enet(feats)
            self._rec_end(tok)
        n = feats.shape[0]
        if fused is None:
            # reference calling convention: precomputed, stacked index lists + killing_inds
            l3 = blobs["proj_ind_3d"][0].to(dev).contiguous()
            l2 = blobs["proj_ind_2d"][0].to(dev).contiguous()
            nreal = l3.shape[0]
            pix = torch.empty(nreal, dims[0] * dims[1] * dims[2], dtype=torch.int16, device=dev)
            S.check(S.lib.sis3d_project_scatter_lists(S.ptr(l3), S.ptr(l2), nreal, *dims, S.ptr(pix), S.stream()), "scatter")
            kill = set(int(k) for k in (killing_inds or []))
            pl = [(k, k) for k in range(min(n, nreal)) if k not in kill]  # zip(imageft, proj3d) + skip by position
            if not pl:
                raise S.Sis3dError("every view was skipped: nothing to back-project")
            pairs = torch.tensor([v for p in pl for v in p], dtype=torch.int32).to(dev)
            n_pairs = torch.tensor([len(pl)], dtype=torch.int32, device=dev)
            self._proj_counts = None
        else:
            # fused path: depth/pose/world2grid in, no index lists ever materialised
            vp, depths = fused["vp"], fused["depths"]
            intr = (cfg.INTRINSIC[0][0], cfg.INTRINSIC[1][1], cfg.INTRINSIC[0][2], cfg.INTRINSIC[1][2])
            tok = self._rec("project_map")
            pix, counts = proj.project_maps(vp, depths, intr, (cfg.PROJ_DEPTH_MIN, cfg.PROJ_DEPTH_MAX, cfg.VOXEL_SIZE),
                                            dims, w, h)
            self._rec_end(tok)
            pairs = torch.empty(3 * n, dtype=torch.int32, device=dev)
            n_pairs = torch.empty(1, dtype=torch.int32, device=dev)
            S.check(S.lib.sis3d_backproject_pairs(S.ptr(counts), n, S.ptr(pairs), S.ptr(n_pairs), S.stream()), "pairs")
            self._proj_counts = counts
        first = self.SPEC["color"][0]
        if (self._sparse_color and not self._keep_debug and first[0] == "k2s2" and feats.shape[1] % 16 == 0
                and first[3] in (32, 64)):
            # fused + sparse: never materialise the back-projected volume (csrc/sparse.cu)
            r = self._packed[f"color.{first[1]}"]
            cout = r.cout
            od = tuple(d // 2 for d in dims)
            out = Act(torch.empty(*od, cout, dtype=torch.float32, device=dev), od, cout)
            if fp16_twins(self._math):
                out.h = torch.empty(*od, cout, dtype=torch.float16, device=dev)
            feats = feats.contiguous()
            feats_t = torch.empty(feats.shape[0], w * h, feats.shape[1], dtype=torch.float32, device=dev)
            nbytes = int(S.lib.sis3d_backproject_conv_k2s2_workspace_bytes(*dims, cout))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            tok = self._rec("backproject_conv_k2s2")
            S.check(S.lib.sis3d_backproject_conv_k2s2_ex(S.ptr(feats), S.ptr(feats_t), S.ptr(pix), S.ptr(pairs), S.ptr(n_pairs),
                                                         feats.shape[0], feats.shape[1], w, h, *dims, S.ptr(r.simt), cout,
                                                         S.ptr(out.t), S.ptr(out.h), out.ld, 0, S.ptr(ws), C.c_size_t(nbytes),
                                                         S.stream()),
                    "backproject_conv_k2s2")
            self._rec_end(tok)
            return ("color0", out)
        tok = self._rec("backproject_max")
        vol = proj.backproject(feats, pix, pairs, n_pairs, dims, w, h)
        self._rec_end(tok)
        return Act(vol, dims, feats.shape[1])

    def _parallel(self, fns):
        """Run independent launch sequences as parallel branches: forked side streams that join back, which CUDA-graph
        capture records as concurrent graph branches.  The layers at 24x12x24 launch only 54-108 CTAs on 148 SMs, so
        independent stacks (colour || geometry, RPN level 1 || level 2) overlap instead of queueing."""
        if not self._branches or self._prof is not None or len(fns) < 2:
            return [f() for f in fns]
        cur = torch.cuda.current_stream()
        key = ("branch_streams", cur.device)
        side = self._const(key, lambda: [torch.cuda.Stream() for _ in range(3)])[:len(fns) - 1]
        out = [None] * len(fns)
        for st in side:
            st.wait_stream(cur)
        pin = S.pin_stream(None)  # launches must follow torch's current stream inside the branches
        try:
            for i, st in enumerate(side, 1):
                with torch.cuda.stream(st):
                    out[i] = fns[i]()
            out[0] = fns[0]()
        finally:
            S.pin_stream(pin)
        for st in side:
            cur.wait_stream(st)
        return out

    def _backbone(self, scene: Act, imageft: Act):
        """reference: backbones.py:98-113.  Concatenation is free: both producers write their slice of
        the level-1 tensor directly (colour channels first, then geometry)."""
        spec = self.SPEC
        dev = scene.t.device
        if cfg.USE_IMAGES:
            d4 = tuple((d // 2) // 2 for d in scene.dims)
            level1 = Act(torch.empty(*d4, 128, dtype=torch.float32, device=dev), d4, 128)
            def colour():
                if isinstance(imageft, tuple):  # ("color0", act): color.0 already produced by the fused sparse path
                    return self._run_stack(imageft[1], "color", spec["color"][1:],
                                           final_out=lambda x, op: Act(level1.t, d4, 64, ld=128, coff=0))
                return self._run_stack(imageft, "color", spec["color"],
                                       final_out=lambda x, op: Act(level1.t, d4, 64, ld=128, coff=0))

            def geometry():
                return self._run_stack(scene, "geometry1", spec["geometry1"],
                                       final_out=lambda x, op: Act(level1.t, d4, 64, ld=128, coff=64))

            self._parallel([colour, geometry])
        else:
            level1 = self._run_stack(scene, "geometry1", spec["geometry1"])
        level2 = self._run_stack(level1, "geometry2", spec["geometry2"])
        return level1, level2

    def _region_proposal(self, feats, dims, out=None):
        """reference: network.py:537-587 + 657-683 (softmax/anchors/decode/top-N/NMS fused on device)."""
        def head(lvl, f, A):
            h = self._conv(f, f"rpn_net_level{lvl}", act=1, want32=False, want16=True)  # hidden feeds only the merged head
            heads = self._conv(h, f"rpn_heads_level{lvl}")  # [N, ld]: [2A class logits | 6A box deltas | zero pad]
            heads.t.record_stream(torch.cuda.current_stream())
            return heads

        todo = [(lvl, f, cfg["NUM_ANCHORS_LEVEL%d" % lvl]) for lvl, f in enumerate(feats, 1)
                if f is not None and cfg["NUM_ANCHORS_LEVEL%d" % lvl]]
        if [t[0] for t in todo] != list(range(1, len(todo) + 1)):
            # the proposal kernel numbers the levels it is given 1..n and RoI pooling reads level k's features for id k; a gap
            # (e.g. NUM_ANCHORS_LEVEL1 = 0 with level 2 active; the reference keeps the true pyramid level,
            # proposal_layer.py:150-157) would pool from the wrong map.  No released config has one: refuse instead of guessing.
            raise S.Sis3dError("active RPN levels must be contiguous from level 1 (NUM_ANCHORS_LEVELn = 0 only for trailing levels)")
        main = torch.cuda.current_stream()
        outs = self._parallel([(lambda t=t: head(*t)) for t in todo])
        levels = []
        for (lvl, f, A), heads in zip(todo, outs):
            heads.t.record_stream(main)
            ld = heads.C  # padded head width
            cls = Act(heads.t, f.dims, 2 * A, ld=ld, coff=0)
            bbox = Act(heads.t.reshape(-1)[2 * A:], f.dims, 6 * A, ld=ld, coff=0)
            name = cfg["ANCHORS_TYPE_LEVEL%d" % lvl]
            sizes = self._const(("anchors", name, f.t.device), lambda: torch.tensor(
                read_anchor_sizes(name), dtype=torch.float32, device=f.t.device).contiguous())
            if sizes.shape[0] != A:
                raise S.Sis3dError(f"anchor table {name} has {sizes.shape[0]} rows, cfg says {A}")
            levels.append(dict(cls=cls.t, deltas=bbox.t, sizes=sizes, grid=f.dims, A=A, cls_mode=0, cls_ld=ld, deltas_ld=ld))
            if self._keep_debug:
                self._predictions[f"rpn_heads_level{lvl}"] = heads.t  # [..., :2A] class logits, [..., 2A:] box deltas
        tok = self._rec("rpn_proposals")
        res = rpn_proposals(levels, dims, "TEST", want_order=self._keep_debug, out=out)
        self._rec_end(tok)
        if self._keep_debug:
            self._predictions["rpn_order"] = res[4]
        return res[:4]

    def _classify(self, feats, rois, level_ids, out=None):
        """RoI pooling per pyramid level + MLP + heads (reference: network.py:503-534, backbones.py:92-96,
        network.py:589-604).  Always processes the padded post-NMS row count; rows >= num are zeros."""
        P = int(cfg.CLASS_POOLING_SIZE)
        R = rois.shape[0]
        f1 = feats[0]
        dev = rois.device
        pool5 = torch.empty(R, f1.C * P ** 3, dtype=torch.float32, device=dev)
        f = [x.t if x is not None else None for x in feats] + [None, None]
        tok = self._rec("roi_pool_levels")
        S.check(S.lib.sis3d_roi_pool_levels(S.ptr(f[0]), S.ptr(f[1]), S.ptr(f[2]), S.ptr(level_ids),
                                            S.f32(1.0 / self._feat_stride[0]), R, *f1.dims, f1.C, P, P, P, S.ptr(rois),
                                            S.ptr(pool5), None, S.stream()), "roi_pool_levels")
        self._rec_end(tok)
        x1 = self._linear(pool5, "classifier.0", 1)
        nc = int(cfg.NUM_CLASSES)
        if out is not None:
            cls_t, box_t = out
        else:
            cls_t = torch.empty(R, nc, dtype=torch.float32, device=dev)
            box_t = torch.empty(R, nc * 6, dtype=torch.float32, device=dev)
        p2, p3 = self._packed["classifier.2"], self._packed["classifier.4"]
        pc, pb = self._packed["classifier_cls_score_net"], self._packed["classifier_bbox_pred_net"]
        tok = self._rec("mlp_tail")
        S.check(S.lib.sis3d_mlp_tail(S.ptr(x1), R, p2.cin, S.ptr(p2.simt), S.ptr(p2.bias), p2.cout, S.ptr(p3.simt), S.ptr(p3.bias),
                                     p3.cout, S.ptr(pc.simt), S.ptr(pc.bias), pc.cout, S.ptr(pb.simt), S.ptr(pb.bias), pb.cout,
                                     S.ptr(cls_t), S.ptr(box_t), S.stream()), "mlp_tail")
        self._rec_end(tok)
        cls_score, bbox_pred = Act(cls_t, (R, 1, 1), nc), Act(box_t, (R, 1, 1), nc * 6)
        if self._keep_debug:
            self._predictions["pool5"] = pool5
        return cls_score.t.view(R, -1), bbox_pred.t.view(R, -1)

    def _mask_branch(self, scene_ncdhw, det_host, n, extras=None):
        """Ragged per-RoI mask head (reference: network.py:283-317).  All kept crops are packed along x on
        one zeroed canvas [sum(w_j + 1), max h, max l, 64] (one zero slab between crops = the crop-border
        zero padding), so each of the six layers is ONE launch: layer 1 (C_in = 2, windowed NCDHW scene) and
        the 1x1 head on the fp32 CUDA-core kernel, the four 64->64 3x3x3 layers on the tcgen05 kernel driven
        by an explicit list of 4x4x8 bricks.  The tables come from the native planner (sis3d_mask_plan_build)
        and travel in ONE pinned H2D copy; all buffers come from a grow-only arena."""
        dev = scene_ncdhw.device
        X, Y, Z = (int(v) for v in scene_ncdhw.shape[2:])
        ncls = self._packed["mask_backbone.geometry.10"].cout
        math = mask_stage_code(self._mask_math, self._packed["mask_backbone.geometry.2"].tc)
        det_host = np.ascontiguousarray(det_host[:n], dtype=np.float32)
        plan = S.MaskPlan()
        cap = self._arena["mask_tables_host"].numel() if "mask_tables_host" in self._arena else 1 << 18
        while True:
            stage = self._ws("mask_tables_host", cap, torch.uint8, dev, pinned=True)
            rc = S.lib.sis3d_mask_plan_build(C.c_void_p(det_host.ctypes.data), n, X, Y, Z, ncls, 1 if math else 0,
                                             C.c_void_p(stage.data_ptr()), C.c_size_t(stage.numel()), C.byref(plan))
            if rc == -3:  # SIS3D_EWORKSPACE: grow the pinned staging buffer and retry
                cap = int(plan.bytes) * 2
                continue
            S.check(rc, "mask_plan_build")
            break
        nk = int(plan.n_kept)
        if nk == 0:
            return []
        nbytes, total = int(plan.bytes), int(plan.total_voxels)
        host = stage.numpy()
        offs = host[plan.off_offs:plan.off_offs + 8 * (nk + 1)].view(np.int64).copy()
        sizes = host[plan.off_sizes:plan.off_sizes + 12 * nk].view(np.int32).reshape(nk, 3).copy()
        cvox = int(plan.canvas[0]) * int(plan.canvas[1]) * int(plan.canvas[2])
        a = S.MaskStage()
        a.scene, a.X, a.Y, a.Z, a.ncls, a.math = scene_ncdhw.data_ptr(), X, Y, Z, ncls, math
        a.w_first = self._packed["mask_backbone.geometry.0"].simt.data_ptr()
        a.w_last = self._packed["mask_backbone.geometry.10"].simt.data_ptr()
        for i, idx in enumerate((2, 4, 6, 8)):
            r = self._packed[f"mask_backbone.geometry.{idx}"]
            a.w_mid[i] = (r.tc[("tf32", "fp16")[math - 1]] if math else r.simt).data_ptr()
        a.tables = self._ws("mask_tables", nbytes, torch.uint8, dev).data_ptr()
        a.canvas_bytes = 2 * 64 * (total * 4 if math == 0 else cvox * (2 if math == 2 else 4))
        a.canvas = self._ws("mask_canvas", a.canvas_bytes, torch.uint8, dev).data_ptr()
        if math == 2:
            a.canvas32_bytes = cvox * 64 * 4
            a.canvas32 = self._ws("mask_canvas32", a.canvas32_bytes, torch.uint8, dev).data_ptr()
        # handed to the caller (mask_pred views / packed bits): fresh allocations, not arena memory
        outb = torch.empty(total * ncls, dtype=torch.float32, device=dev)
        bits = torch.empty(total, dtype=torch.uint8, device=dev)
        a.masks, a.bits, a.thresh = outb.data_ptr(), bits.data_ptr(), float(cfg.MASK_THRESH)
        if extras is not None:  # the scene loop reads the thresholded masks back: ONE small D2H, queued by the same call
            pin = self._ws("bits_host", total, torch.uint8, dev, pinned=True)
            a.bits_host = pin.data_ptr()
            extras.update(mask_bits=bits, mask_offsets=offs, mask_sizes=sizes, bits_pin=pin[:total])
        tok = self._rec("mask_stage")
        S.check(S.lib.sis3d_mask_stage_launch(C.byref(plan), C.c_void_p(stage.data_ptr()), C.byref(a), S.stream()), "mask_stage")
        self._rec_end(tok)
        return _MaskList(outb, offs, sizes, ncls)

    # ------------------------------------------------------------------ forward
    _carve_layouts = {}

    @staticmethod
    def _carve(pack, R, nc):
        """Typed views of the packed result buffer of the static stage (one buffer -> one clone / one copy)."""
        lay = Network._carve_layouts.get((R, nc))
        if lay is not None and pack.device.type != "meta":
            return {name: pack[a:b].view(dt).view(shape) for name, a, b, dt, shape in lay[0]}, lay[1]
        o, out, rec = 0, {}, []
        for name, shape, dt in (("rois", (R, 6), torch.float32), ("scores", (R,), torch.float32), ("level_ids", (R,), torch.int32),
                                ("num", (4,), torch.int32), ("cls_score", (R, nc), torch.float32),
                                ("bbox_pred", (R, nc * 6), torch.float32), ("cls_prob", (R, nc), torch.float32),
                                ("det", (R, 16), torch.float32), ("cls_pred", (R,), torch.int64)):
            nb = int(np.prod(shape)) * torch.empty(0, dtype=dt).element_size()
            o = (o + 15) // 16 * 16
            out[name] = pack[o:o + nb].view(dt).view(*shape)
            rec.append((name, o, o + nb, dt, shape))
            o += nb
        Network._carve_layouts[(R, nc)] = (rec, o)
        return out, o

    def _static_stage(self, scene_t, dims, blobs=None, killing_inds=None, fused=None):
        """Every fixed-shape step: back-projection -> backbone -> RPN/NMS -> RoI pool -> classifier ->
        detection decode.  No host synchronisation inside, so the whole stage can be replayed as one CUDA
        graph per (scene shape, #views)."""
        dev = scene_t.device
        P = self._predictions
        scene = Act(scene_t, dims, 2, layout="ncdhw")
        imageft = None
        if cfg.USE_IMAGES:
            imageft = self._backproject(blobs, killing_inds, dims, dev, fused)
            self._imageft_vc = imageft.t if (self._keep_debug and not isinstance(imageft, tuple)) else None
        level1, level2 = self._backbone(scene, imageft)
        if self._keep_debug:
            P["level1_vc"], P["level2_vc"] = level1.t, level2.t
        R, nc = int(cfg.TEST.RPN_POST_NMS_TOP_N), max(int(cfg.NUM_CLASSES), 1)
        probe, total = self._carve(torch.empty(1 << 22, dtype=torch.uint8, device="meta"), R, nc)
        pack = torch.empty(total + 16, dtype=torch.uint8, device=dev)
        out, _ = self._carve(pack, R, nc)
        out["pack"] = pack
        rois, scores, level_ids = out["rois"], out["scores"], out["level_ids"]
        num = out["num"][:1]
        out["num"] = num
        self._region_proposal((level1, level2, None), dims, out=(rois, scores, level_ids, num))
        if cfg.USE_CLASS:
            cls_score, bbox_pred = self._classify((level1, level2, None), rois, level_ids, out=(out["cls_score"], out["bbox_pred"]))
            cls_prob, cls_pred, det = out["cls_prob"], out["cls_pred"], out["det"]
            tok = self._rec("detect_decode")
            S.check(S.lib.sis3d_detect_decode(S.ptr(rois), S.ptr(num), R, S.ptr(cls_score), S.ptr(bbox_pred), nc,
                                              *dims, S.f32(cfg.CLASS_THRESH), S.ptr(cls_prob), S.ptr(cls_pred),
                                              S.ptr(det), S.stream()), "detect_decode")
            self._rec_end(tok)
        return out

    def _graph_state(self, key, dims, n_views, feat_shape, dev):
        """Static input buffers + captured graph of `_static_stage` for one input shape (feat_shape = shape of one view's
        2-D input: [128,32,41] ENet features, or [3,256,328] images when the encoder is part of the graph)."""
        st = self._graphs.get(key)
        if st is not None:
            if next(reversed(self._graphs)) != key:
                self._graphs[key] = self._graphs.pop(key)  # most recently used last
            return st
        while len(self._graphs) >= self._graph_cache:  # LRU eviction: drops the graph, its static buffers and its pool
            self._graphs.pop(next(iter(self._graphs)))
        w, h = int(cfg.DEPTH_SHAPE[0]), int(cfg.DEPTH_SHAPE[1])
        st = dict(scene=torch.zeros(1, 2, *dims, dtype=torch.float32, device=dev))
        if cfg.USE_IMAGES:
            st.update(feats=torch.zeros(n_views, *feat_shape, dtype=torch.float32, device=dev),
                      depths=torch.zeros(n_views, h, w, dtype=torch.float32, device=dev),
                      vp=torch.zeros(n_views, 40, dtype=torch.float32, device=dev))
        st["graph"] = None
        self._graphs[key] = st
        return st

    # -- a forward is four host steps (stage inputs, static stage, ragged stage, finalize); `forward` runs them back to back,
    #    `forward_pipelined` overlaps them across consecutive scenes on stream slots (each slot owns its graphs, static
    #    buffers and arena)
    def _slot(self, i):
        while len(self._slots) <= i:
            self._slots.append(dict(stream=torch.cuda.Stream() if self._slots else None, graphs={}, arena={}))
        return self._slots[i]

    class _UseSlot:
        def __init__(self, net, slot):
            self.net, self.slot = net, slot

        def __enter__(self):
            n, sl = self.net, self.slot
            d = n.__dict__  # plain attribute writes: nn.Module.__setattr__ costs ~5 us each
            self.saved = (d["_graphs"], d["_arena"])
            d["_graphs"], d["_arena"] = sl["graphs"], sl["arena"]
            self.prev = None
            if sl["stream"] is not None:  # set_stream is several times cheaper than the torch.cuda.stream() context manager
                self.prev = d.get("_home_stream")  # the scene loop looks it up once, not three times per scene
                if self.prev is None:
                    self.prev = torch.cuda.current_stream()
                torch.cuda.set_stream(sl["stream"])
                handle = sl.get("handle")
                if handle is None:
                    handle = sl["handle"] = C.c_void_p(sl["stream"].cuda_stream)
            else:
                handle = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            self.old_pin = S.pin_stream(handle)

        def __exit__(self, *exc):
            S.pin_stream(self.old_pin)
            if self.prev is not None:
                torch.cuda.set_stream(self.prev)
            d = self.net.__dict__
            d["_graphs"], d["_arena"] = self.saved

    def _submit(self, blobs, killing_inds, slot):
        """Step 1 (async): input copies, static stage (graph replay), packed results -> pinned host (async D2H)."""
        return self._run_static(self._stage_inputs(blobs, killing_inds, slot))

    def _stage_inputs(self, blobs, killing_inds, slot):
        """Step 1a (async): per-view constants on the host + the scene's input copies into the slot's static buffers.
        The scene loop issues this one scene ahead of the graph replay so the H2D transfer hides behind compute."""
        self._ensure_packed()
        dev = self.__dict__["_dev"]
        data = blobs["data"]
        if data.shape[0] != 1:
            raise S.Sis3dError("batch size 1 only (as the reference's RoI pooling / proposal layer)")
        dims = tuple(int(v) for v in data.shape[2:])
        home = self.__dict__.get("_home_stream")  # set while the pipelined scene loop runs
        h = dict(slot=slot, dims=dims, id=blobs["id"][0] if "id" in blobs else None, scene_info=data.shape[2:], blobs=blobs,
                 killing_inds=killing_inds, dev=dev, fresh=home is None)
        if home is not None and slot["stream"] is not None:
            # tensors yielded by the scene loop live in slot-owned buffers (result ring, arena): whatever the consumer queued
            # on its own stream to read them (a clone, a D2H copy) must finish before this slot's stream overwrites them
            slot["stream"].wait_stream(home)
        with torch.no_grad(), Network._UseSlot(self, slot):
            lists = cfg.USE_IMAGES and "proj_ind_3d" in blobs
            use_graph = self._use_graph and not (self._keep_debug or self._prof is not None or lists)
            fused = None
            if cfg.USE_IMAGES and not lists:
                imgs = blobs["nearest_images"]
                w, hh = int(cfg.DEPTH_SHAPE[0]), int(cfg.DEPTH_SHAPE[1])
                vp = proj.view_params(cfg.INTRINSIC, (w, hh), cfg.PROJ_DEPTH_MIN, cfg.PROJ_DEPTH_MAX, dims, None,
                                      imgs["poses"][0], imgs["world2grid"][0])
                fused = dict(vp=vp, feats=imgs["images"][0], depths=torch.as_tensor(imgs["depths"][0]))
            h.update(use_graph=use_graph, fused=fused)
            if use_graph:
                nv = fused["feats"].shape[0] if fused else 0
                fc = tuple(fused["feats"].shape[1:]) if fused else ()
                key = (dims, nv, fc, self._math)
                seen = self._shape_seen[key] = self._shape_seen.get(key, 0) + 1
                if seen < self._graph_after and key not in self._graphs:
                    use_graph = h["use_graph"] = False  # first sight of this shape: run eagerly, capture when it comes back
            if use_graph:
                st = self._graph_state(key, dims, nv, fc, dev)
                st["scene"].copy_(data, non_blocking=True)
                if fused:
                    st["feats"].copy_(fused["feats"], non_blocking=True)
                    st["depths"].copy_(fused["depths"], non_blocking=True)
                    vph = self._ws("vp_host", fused["vp"].numel(), torch.float32, dev, pinned=True)
                    vph.copy_(fused["vp"].reshape(-1))
                    st["vp"].copy_(vph.view_as(st["vp"]), non_blocking=True)
                    h["fdev"] = dict(vp=st["vp"], feats=st["feats"], depths=st["depths"])
                else:
                    h["fdev"] = None
                h["st"] = st
        return h

    def _run_static(self, h):
        """Step 1b (async): static stage (graph replay) on the staged inputs, packed results -> pinned host (async D2H)."""
        blobs, killing_inds, slot, dims, dev = h.pop("blobs"), h.pop("killing_inds"), h["slot"], h["dims"], h.pop("dev")
        data = blobs["data"]
        fused = h.pop("fused")
        before = set(self._predictions) if self._keep_debug else None
        with torch.no_grad(), Network._UseSlot(self, slot):
            if h.pop("use_graph"):
                st, fdev = h.pop("st"), h.pop("fdev")
                if st["graph"] is None:
                    # eager warm-up (fills the region/constant caches, sets kernel attributes), then capture
                    self._static_stage(st["scene"], dims, blobs, None, fdev)
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    n0 = S.launch_count()
                    pin = S.pin_stream(None)  # capture runs on torch's capture stream
                    gc_was_on = gc.isenabled()
                    gc.disable()  # a cyclic-GC pass in the middle of a capture may free CUDA objects (illegal while capturing)
                    try:
                        with torch.cuda.graph(g):
                            st["outs"] = self._static_stage(st["scene"], dims, blobs, None, fdev)
                    finally:
                        if gc_was_on:
                            gc.enable()
                        S.pin_stream(pin)
                    st["graph"], st["n_kernels"] = g, S.launch_count() - n0
                st["graph"].replay()
                self.__dict__["_replayed_kernels"] += st["n_kernels"]
                # results must not alias the replay buffers: ONE copy of the packed result buffer into one of two
                # slot-owned, pre-carved result buffers (valid until this slot has been reused twice)
                ring = st.get("result_ring")
                if h["fresh"]:
                    # reference-compatible forward(): the caller may keep _predictions across scenes (the reference returns
                    # fresh tensors), so hand out a private copy of the packed results and of the scene
                    pk = torch.empty_like(st["outs"]["pack"])
                    outs, _ = self._carve(pk, int(cfg.TEST.RPN_POST_NMS_TOP_N), max(int(cfg.NUM_CLASSES), 1))
                    outs["num"] = outs["num"][:1]
                    outs["pack"] = pk
                    ring = False
                elif ring is None:
                    ring = st["result_ring"] = []
                    for _ in range(2):
                        pk = torch.empty_like(st["outs"]["pack"])
                        o, _ = self._carve(pk, int(cfg.TEST.RPN_POST_NMS_TOP_N), max(int(cfg.NUM_CLASSES), 1))
                        o["num"] = o["num"][:1]
                        o["pack"] = pk
                        ring.append(o)
                    st["ring_pos"] = 0
                if ring is not False:
                    outs = ring[st["ring_pos"]]
                    st["ring_pos"] ^= 1
                outs["pack"].copy_(st["outs"]["pack"], non_blocking=True)
                scene_t = st["scene"].clone() if h["fresh"] else st["scene"]
            else:
                scene_t = data.to(dev, torch.float32, non_blocking=True).contiguous()
                if fused:
                    fused = dict(vp=fused["vp"].to(dev, non_blocking=True),
                                 feats=fused["feats"].to(dev, torch.float32, non_blocking=True),
                                 depths=fused["depths"].to(dev, torch.float32, non_blocking=True).contiguous())
                outs = self._static_stage(scene_t, dims, blobs, killing_inds, fused)
            h["outs"], h["scene_t"] = outs, scene_t
            # the one host round trip of a scene: decoded detections with the RoI count in row 0 / col 15 (12.8 KB)
            if cfg.USE_CLASS:
                det_pin = self._ws("det_host", outs["det"].numel(), torch.float32, dev, pinned=True).view_as(outs["det"])
                det_pin.copy_(outs["det"], non_blocking=True)
                h["det_pin"] = det_pin
            h["ev_static"] = torch.cuda.Event(blocking=self._blocking_sync)
            h["ev_static"].record()
        if self._keep_debug:  # intermediate tensors the static stage left in _predictions (parity tests)
            h["debug"] = {k: v for k, v in self._predictions.items()
                          if k.startswith(("level", "rpn_", "pool5")) or k not in before}
        return h

    def _launch_ragged(self, h):
        """Step 2: wait for the detections of this scene, plan + launch its ragged mask stage, queue the readback."""
        h["ev_static"].synchronize()
        outs = h["outs"]
        P = {}
        with torch.no_grad(), Network._UseSlot(self, h["slot"]):
            if cfg.USE_CLASS:
                det_all = h["det_pin"].numpy()
                n = int(det_all[0, 15])
            else:
                n = int(outs["num"].item())
            P["rois"], P["roi_scores"] = [outs["rois"][:n]], [outs["scores"][:n].view(-1, 1)]
            P["level_inds"] = [outs["level_ids"][:n].float()]
            if cfg.USE_CLASS:
                P["cls_score"], P["cls_pred"], P["cls_prob"] = outs["cls_score"][:n], outs["cls_pred"][:n], outs["cls_prob"][:n]
                P["bbox_pred"] = outs["bbox_pred"][:n]
                P["detections"] = outs["det"][:n]
                if cfg.USE_MASK:
                    det_host = det_all[:n].copy()
                    extras = {}
                    P["mask_pred"] = [self._mask_branch(h["scene_t"], det_host, n, extras)]
                    P["detections_host"] = det_host
                    if "bits_pin" in extras:  # thresholded predicted-class masks -> pinned host (queued by the mask stage)
                        h["bits_pin"] = extras.pop("bits_pin")
                    P.update(extras)
            h["ev_done"] = torch.cuda.Event(blocking=self._blocking_sync)
            h["ev_done"].record()
        h["P"] = P
        return h

    def _finalize(self, h):
        """Step 3: wait for the scene's last kernel / copy and hand out its predictions."""
        h["ev_done"].synchronize()
        P = h["P"]
        if "bits_pin" in h:
            P["mask_bits_host"] = h["bits_pin"].numpy().copy()
        self.__dict__.update(_scene_info=h["scene_info"], _id=h["id"], _scene=h["scene_t"], batch_size=1, _mode="TEST")
        self._predictions.clear()
        self._predictions.update(h.get("debug", {}))
        self._predictions.update(P)
        return self._predictions

    def _check_mode(self, mode):
        if mode != "TEST":
            raise NotImplementedError("only the inference (TEST) forward is implemented on the B200 path")
        if not (cfg.USE_BACKBONE and cfg.USE_RPN):
            raise NotImplementedError("USE_BACKBONE/USE_RPN=False (ground-truth RoIs) are training/ablation modes")

    def forward(self, blobs, mode="TEST", killing_inds=None):
        """Reference-compatible synchronous forward of one scene (lib/nets/network.py:72,187-317)."""
        self._check_mode(mode)
        return self._finalize(self._launch_ragged(self._submit(blobs, killing_inds, self._slot(0))))

    def forward_pipelined(self, blobs_iter, mode="TEST"):
        """Throughput form of the scene loop (lib/model/trainval.py:787-822): yields (blobs, predictions) in order while
        seven scenes are in flight on seven stream slots -- scene i+1: input H2D (issued one scene ahead so the transfer
        hides behind compute); scenes i .. i-3: static stage (four graph replays overlapping: one alone is a latency
        chain of small grids; measured 3 -> 4: +1 %, 5: no further gain); then the ragged mask stage and the read-back.
        The yielded dict is only valid until the next iteration."""
        self._check_mode(mode)
        self._ensure_packed()
        blobs_iter = self._reject_index_lists(blobs_iter)
        self.__dict__["_home_stream"] = torch.cuda.current_stream()  # restored after every slot switch of this loop
        try:
            yield from self._scene_loop(blobs_iter)
        finally:
            self.__dict__["_home_stream"] = None

    @staticmethod
    def _reject_index_lists(blobs_iter):
        """The scene loop computes the projection on the device from depth / pose / world2grid; blobs that carry precomputed
        proj_ind_3d/2d lists need their killing_inds (lib/model/trainval.py:805-822), which this API has no slot for: they go
        through the synchronous forward(blobs, 'TEST', killing_inds)."""
        for b in blobs_iter:
            if "proj_ind_3d" in b:
                raise S.Sis3dError("forward_pipelined takes depth/pose/world2grid blobs; use forward(blobs, 'TEST', killing_inds) "
                                   "for blobs with precomputed proj_ind_3d/2d lists")
            yield b

    def _scene_loop(self, blobs_iter):
        from collections import deque
        q = deque()      # [blobs, handle, ragged_launched] of scenes whose static stage has been launched
        staged = None    # (blobs, handle) of the scene whose inputs are uploading
        i = 0
        n_static = max(1, int(os.environ.get("SIS3D_PIPE_STATIC", "4")))  # static stages (graph replays) in flight at once
        depth = max(n_static + 2, int(os.environ.get("SIS3D_PIPE_DEPTH", str(n_static + 3))))  # scenes in flight (= stream slots)
        for blobs in blobs_iter:
            if len(q) == depth - 1:  # frees the slot the new scene is about to use
                b, h, _ = q.popleft()
                yield b, self._finalize(h)
            nxt = (blobs, self._stage_inputs(blobs, None, self._slot(1 + i % depth)))
            i += 1
            if staged is not None:
                q.append([staged[0], self._run_static(staged[1]), False])
            staged = nxt
            # the mask stage of a scene needs its detections on the host: wait for the static stage launched n_static
            # iterations ago, so that n_static graph replays overlap on the GPU (one alone is a latency chain of small grids)
            if len(q) > n_static and not q[-n_static - 1][2]:
                self._launch_ragged(q[-n_static - 1][1])
                q[-n_static - 1][2] = True
        if staged is not None:
            q.append([staged[0], self._run_static(staged[1]), False])
        while q:
            b, h, launched = q.popleft()
            if not launched:
                self._launch_ragged(h)
            yield b, self._finalize(h)

    def kernel_launches(self):
        """libsis3d kernels executed so far by this process: direct launches + kernels inside replayed graphs."""
        return S.launch_count() + self._replayed_kernels

    def delete_intermediate_states(self):
        self._predictions.clear()
