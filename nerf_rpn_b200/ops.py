"""Torch-tensor front-ends of the C ABI. PyTorch only provides device memory and the current stream here;
every computation is a kernel of libnerf_rpn_b200.so.  All functions require CUDA tensors and raise otherwise
(no CPU fallback)."""
import ctypes
from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import WgradDesc, ConvDesc, FcosDesc, FcosLossDesc, FcosTargetDesc, GnLevel, RpnDesc, check, lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(t: torch.Tensor, dtype, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"nerf_rpn_b200: {name} must be a CUDA tensor (this package has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"nerf_rpn_b200: {name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"nerf_rpn_b200: {name} must be contiguous")
    return t


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


# ------------------------------------------------------------------------------------------------ boxes
def set_nms_cull_mode(mode: int) -> None:
    """0 (default): only exact-zero culls -- the keep set is provably the reference's.  1 / 3: + geometric ratio culls (+ footprint lens) from
    16 384 boxes up: 4-5x faster at 1 M boxes, may differ from the reference in ~1e-5 of the boxes (include/nerf_rpn_b200.h)."""
    lib().nrpn_set_nms_cull_mode(int(mode))


def iou3d_pairs(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    a = _req(a, torch.float32, "a"); b = _req(b, torch.float32, "b")
    if a.shape != b.shape or a.dim() != 2 or a.shape[1] not in (6, 7):
        raise ValueError("iou3d_pairs expects two (n,6) or two (n,7) tensors")
    out = torch.empty(a.shape[0], dtype=torch.float32, device=a.device)
    check(lib().nrpn_iou3d_pairs(_ptr(a), _ptr(b), a.shape[0], a.shape[1], _ptr(out), _stream()), "iou3d_pairs")
    return out


def iou3d_matrix(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    a = _req(a, torch.float32, "a"); b = _req(b, torch.float32, "b")
    if a.dim() != 2 or b.dim() != 2 or a.shape[1] != b.shape[1] or a.shape[1] not in (6, 7):
        raise ValueError("The second dimension of boxes1 and boxes2 should be the same, both 6 or 7. But get {} and {}."
                         .format(a.shape[-1], b.shape[-1]))
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=a.device)
    check(lib().nrpn_iou3d_matrix(_ptr(a), a.shape[0], _ptr(b), b.shape[0], a.shape[1], _ptr(out), _stream()), "iou3d_matrix")
    return out


def assign_targets(anchors: torch.Tensor, gt: torch.Tensor, valid: Optional[torch.Tensor], high: float, low: float,
                   allow_low_quality_matches: bool = True):
    """anchors (N,6), gt (G,6|7), valid (N) bool or None -> labels (N) f32 in {1,0,-1}, matched_idxs (N) i64 (rpn.py:240-290)."""
    anchors = _req(anchors, torch.float32, "anchors")
    gt = _req(gt, torch.float32, "gt")
    n, g = anchors.shape[0], gt.shape[0]
    v = None
    if valid is not None:
        v = valid.to(torch.uint8).contiguous()
    labels = torch.empty((n,), dtype=torch.float32, device=anchors.device)
    matched = torch.empty((n,), dtype=torch.int64, device=anchors.device)
    ws = _workspace(lib().nrpn_assign_targets_workspace_bytes(n, g), anchors.device)
    check(lib().nrpn_assign_targets(_ptr(anchors), n, _ptr(gt), g, int(gt.shape[1]), _ptr(v), float(high), float(low),
                                    int(bool(allow_low_quality_matches)), _ptr(labels), _ptr(matched), _ptr(ws), ws.numel(), _stream()),
          "assign_targets")
    return labels, matched


def rowmax(m: torch.Tensor):
    """(rows, cols) fp32 -> (max, first argmax) per row, on the device."""
    m = _req(m, torch.float32, "m")
    rows, cols = m.shape
    mv = torch.empty((rows,), dtype=torch.float32, device=m.device)
    am = torch.empty((rows,), dtype=torch.int32, device=m.device)
    check(lib().nrpn_rowmax_f32(_ptr(m), rows, cols, _ptr(mv), _ptr(am), _stream()), "rowmax")
    return mv, am


def recall_match(overlaps: torch.Tensor) -> torch.Tensor:
    """(P, G) fp32 IoU matrix -> the min(P, G) IoUs recorded by the greedy loop of eval.py:33-52 (device resident)."""
    overlaps = _req(overlaps, torch.float32, "overlaps")
    p, g = overlaps.shape
    out = torch.zeros((min(p, g),), dtype=torch.float32, device=overlaps.device)
    check(lib().nrpn_recall_match(_ptr(overlaps), p, g, _ptr(out), _stream()), "recall_match")
    return out


def sort_vertices_forward(vertices: torch.Tensor, mask: torch.Tensor, num_valid: torch.Tensor) -> torch.Tensor:
    """Same contract as the reference's pybind op (cuda_op/sort_vert.cpp:6-34)."""
    if not vertices.is_cuda:
        raise RuntimeError("vertices must be a CUDA tensor")
    if not mask.is_cuda:
        raise RuntimeError("mask must be a CUDA tensor")
    if not num_valid.is_cuda:
        raise RuntimeError("num_valid must be a CUDA tensor")
    if not (vertices.is_contiguous() and mask.is_contiguous() and num_valid.is_contiguous()):
        raise RuntimeError("inputs must be contiguous tensors")
    if vertices.dtype != torch.float32:
        raise RuntimeError("vertices must be a float tensor")
    if mask.dtype != torch.bool:
        raise RuntimeError("mask must be a bool tensor")
    if num_valid.dtype != torch.int32:
        raise RuntimeError("num_valid must be a int tensor")
    b, n, m = vertices.shape[0], vertices.shape[1], vertices.shape[2]
    idx = torch.zeros((b, n, 9), dtype=torch.int32, device=vertices.device)
    with torch.cuda.device(vertices.device):
        check(lib().nrpn_sort_vertices(_ptr(vertices), _ptr(mask), _ptr(num_valid), b, n, m, _ptr(idx), _stream()),
              "sort_vertices")
    return idx


_ws_cache = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = ws
    return ws


def nms_device(boxes: torch.Tensor, scores: torch.Tensor, groups: Optional[torch.Tensor], thr: float):
    """Returns (keep int64 (n,), n_keep int32 (1,)) on the device -- no host synchronisation."""
    boxes = _req(boxes, torch.float32, "boxes"); scores = _req(scores, torch.float32, "scores")
    n = boxes.shape[0]
    if groups is not None:
        groups = _req(groups, torch.int32, "groups")
    keep = torch.empty(max(n, 1), dtype=torch.int64, device=boxes.device)
    n_keep = torch.zeros(1, dtype=torch.int32, device=boxes.device)
    if n == 0:
        return keep[:0], n_keep
    if n > lib().nrpn_nms_max_boxes():
        raise ValueError(f"nms: at most {lib().nrpn_nms_max_boxes()} boxes per call are supported, got {n}")
    wsb = lib().nrpn_nms_workspace_bytes(n)
    ws = _workspace(wsb, boxes.device)
    check(lib().nrpn_nms(_ptr(boxes), boxes.shape[1], _ptr(scores), _ptr(groups), n, float(thr), _ptr(keep), _ptr(n_keep),
                         _ptr(ws), ws.numel(), _stream()), "nms")
    return keep, n_keep


# ------------------------------------------------------------------------------------------------ conv
def conv_block_n(cout: int) -> int:
    return lib().nrpn_conv3d_block_n(int(cout))


class ConvLevelArgs:
    __slots__ = ("x", "y", "res", "n", "in_dims", "out_dims", "res_dims", "ldy", "ldr")

    def __init__(self, x, y, n, in_dims, out_dims, ldy, res=None, res_dims=None, ldr=0):
        self.x, self.y, self.res, self.n = x, y, res, n
        self.in_dims, self.out_dims = tuple(in_dims), tuple(out_dims)
        self.res_dims = tuple(res_dims) if res_dims is not None else tuple(out_dims)
        self.ldy, self.ldr = ldy, ldr


def _conv_desc(levels, w, shift, cin, cout, taps, stride, relu, out_fp32) -> ConvDesc:
    d = ConvDesc()
    d.cin, d.cout, d.n_taps = int(cin), int(cout), len(taps)
    for t, off in enumerate(taps):
        for k in range(3):
            d.tap_off[t][k] = int(off[k])
    d.stride, d.relu, d.out_fp32 = int(stride), int(relu), int(bool(out_fp32))      # relu: 0 none, 1 ReLU, 2 GELU
    d.w, d.shift = w.data_ptr(), shift.data_ptr()
    d.wsplit = 1 if w.dim() == 4 else 0          # (taps, 2, CoutPad, Cin): hi / lo weight planes (packing.split_hi_lo)
    d.n_levels = len(levels)
    for i, L in enumerate(levels):
        lv = d.level[i]
        lv.x, lv.y = L.x.data_ptr(), L.y.data_ptr()
        lv.res = 0 if L.res is None else L.res.data_ptr()
        lv.n = int(L.n)
        lv.xi, lv.yi, lv.zi = (int(v) for v in L.in_dims)
        lv.xo, lv.yo, lv.zo = (int(v) for v in L.out_dims)
        lv.xr, lv.yr, lv.zr = (int(v) for v in L.res_dims)
        lv.ldy, lv.ldr = int(L.ldy), int(L.ldr)
    d.workspace, d.workspace_bytes = 0, 0
    d.act_fp16 = 1 if levels[0].x.dtype == torch.float16 else 0
    if w.dtype != levels[0].x.dtype:
        raise TypeError(f"conv3d: weights are {w.dtype} but activations are {levels[0].x.dtype}")
    return d


def conv3d_workspace_bytes(levels, w, shift, cin, cout, taps, stride=1, relu=False, out_fp32=False) -> int:
    """Bytes of (zero-filled) split-K scratch this layer would like; 0 if it is not split."""
    d = _conv_desc(levels, w, shift, cin, cout, taps, stride, relu, out_fp32)
    return int(lib().nrpn_conv3d_workspace_bytes(ctypes.byref(d)))


def conv3d_variant(levels, w, shift, cin, cout, taps, stride=1, relu=False, out_fp32=False) -> str:
    """Which kernel variant nrpn_conv3d_fprop launches for this layer (host-side query, no launch)."""
    d = _conv_desc(levels, w, shift, cin, cout, taps, stride, relu, out_fp32)
    return lib().nrpn_conv3d_variant(ctypes.byref(d)).decode()


def conv3d_fprop(levels: Sequence[ConvLevelArgs], w: torch.Tensor, shift: torch.Tensor, cin: int, cout: int,
                 taps: Sequence[Sequence[int]], stride: int = 1, relu: bool = False, out_fp32: bool = False,
                 workspace: Optional[torch.Tensor] = None):
    """One persistent tcgen05 implicit-GEMM launch over 1..4 levels sharing (w, shift).  `workspace`: optional uint8
    tensor that was zero-filled once (split-K scratch, left zero-filled by every launch)."""
    d = _conv_desc(levels, w, shift, cin, cout, taps, stride, relu, out_fp32)
    if workspace is not None:
        d.workspace, d.workspace_bytes = workspace.data_ptr(), workspace.numel()
    check(lib().nrpn_conv3d_fprop(ctypes.byref(d), _stream()), "conv3d_fprop")


def _act16(t: torch.Tensor, name: str) -> int:
    """16-bit activation tensors are bf16 (default) or fp16 (higher-parity mode); returns the C ABI's act_fp16 flag."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"nerf_rpn_b200: {name} must be a CUDA tensor (this package has no CPU path)")
    if t.dtype not in (torch.bfloat16, torch.float16):
        raise TypeError(f"nerf_rpn_b200: {name} must be bfloat16 or float16, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"nerf_rpn_b200: {name} must be contiguous")
    return 1 if t.dtype == torch.float16 else 0


def is_channels_last_grid(grid: torch.Tensor) -> bool:
    """True for an (N,4,X,Y,Z) tensor whose memory is (N,X,Y,Z,4): what datasets.py:55-56 produces (np.transpose view)."""
    return grid.dim() == 5 and not grid.is_contiguous() and grid.permute(0, 2, 3, 4, 1).is_contiguous()


def to_planar(x: torch.Tensor, z_shift: int = 0) -> torch.Tensor:
    """(N, X, Y, Z, ld) 16-bit channels-last -> planar (N, ld, X, Y, Z) VIEW of a zero-filled buffer whose z pitch is Z + 1 rounded up
    to a multiple of 8; z_shift = s writes out[z'] = x[z' + s] (zero where the source falls outside): the operand layout of
    conv3d_wgrad (TMA wants 16-byte aligned inner coordinates, so z offsets live in shifted copies)."""
    _act16(x, "x")
    n, X, Y, Z, c = x.shape
    zp = (Z + 1 + 7) // 8 * 8
    buf = torch.zeros((n, c, X, Y, zp), dtype=x.dtype, device=x.device)
    check(lib().nrpn_transpose_to_planar(_ptr(x), n, X, Y, Z, c, c, _ptr(buf), zp, int(z_shift), _stream()), "transpose_to_planar")
    return buf[..., :Z]


def conv3d_wgrad(dys: Sequence[torch.Tensor], xs: Sequence[torch.Tensor], taps: Sequence[Sequence[int]], operands: str = "channels_last") -> torch.Tensor:
    """dW (taps, Cout, Cin) fp32 of a stride-1 'same' conv from channels-last 16-bit dY (N,X,Y,Z,Cout) and X (N,X,Y,Z,Cin), one pair per
    pyramid level that shares the weights.  operands="channels_last": the tensors are read where they live (MN-major tcgen05 operands);
    "planar": through transposed, z-shifted staging copies (tap z offsets in {-1, 0, +1}) -- the earlier path, kept for comparison."""
    if operands == "channels_last":
        return _conv3d_wgrad_cl(dys, xs, taps)
    d = WgradDesc()
    d.cout, d.cin, d.n_taps = int(dys[0].shape[-1]), int(xs[0].shape[-1]), len(taps)
    for t, off in enumerate(taps):
        for k in range(3):
            d.tap_off[t][k] = int(off[k])
    dzs = sorted({int(off[2]) for off in taps})
    if any(abs(z) > 1 for z in dzs):
        raise ValueError("conv3d_wgrad: tap z offsets must be in {-1, 0, +1}")
    d.n_levels = len(dys)
    keep = []
    for i, (dy, x) in enumerate(zip(dys, xs)):
        f16 = _act16(dy, "dy")
        if _act16(x, "x") != f16 or dy.shape[:4] != x.shape[:4]:
            raise ValueError("conv3d_wgrad: dy and x must share dtype, batch and spatial extent (stride-1 'same' convolution)")
        pdy = to_planar(dy)
        keep.append(pdy)
        lv = d.level[i]
        lv.dy_planar = pdy.data_ptr()
        for z in dzs:
            px = to_planar(x, z)
            keep.append(px)
            lv.x_planar[z + 1] = px.data_ptr()
        lv.n, lv.x, lv.y, lv.z = int(dy.shape[0]), int(dy.shape[1]), int(dy.shape[2]), int(dy.shape[3])
        lv.z_pitch = int(pdy.stride(3))
    d.act_fp16 = f16
    dw = torch.empty((len(taps), d.cout, d.cin), dtype=torch.float32, device=dys[0].device)
    need = lib().nrpn_conv3d_wgrad_workspace_bytes(ctypes.byref(d))
    if need == 0:
        raise ValueError("conv3d_wgrad: unsupported shape (cout % 128 == 0, cin % 32 == 0, cin <= 256)")
    ws = _workspace(need, dys[0].device)
    d.dw, d.workspace, d.workspace_bytes = dw.data_ptr(), ws.data_ptr(), ws.numel()
    check(lib().nrpn_conv3d_wgrad(ctypes.byref(d), _stream()), "conv3d_wgrad")
    return dw


def _conv3d_wgrad_cl(dys, xs, taps):
    d = WgradDesc()
    d.cout, d.cin, d.n_taps = int(dys[0].shape[-1]), int(xs[0].shape[-1]), len(taps)
    for t, off in enumerate(taps):
        for k in range(3):
            d.tap_off[t][k] = int(off[k])
    d.n_levels = len(dys)
    for i, (dy, x) in enumerate(zip(dys, xs)):
        f16 = _act16(dy, "dy")
        if _act16(x, "x") != f16 or dy.shape[0] != x.shape[0] or not (dy.is_contiguous() and x.is_contiguous()):
            raise ValueError("conv3d_wgrad: dy and x must be contiguous (N,X,Y,Z,C) tensors of one dtype and batch")
        lv = d.level[i]
        lv.dy_cl, lv.x_cl, lv.ld_dy, lv.ld_x = dy.data_ptr(), x.data_ptr(), int(dy.shape[-1]), int(x.shape[-1])
        lv.n, lv.x, lv.y, lv.z = int(dy.shape[0]), int(dy.shape[1]), int(dy.shape[2]), int(dy.shape[3])
        lv.xx, lv.xy, lv.xz = int(x.shape[1]), int(x.shape[2]), int(x.shape[3])
    d.act_fp16 = f16
    d.operand_layout = 1
    dw = torch.empty((len(taps), d.cout, d.cin), dtype=torch.float32, device=dys[0].device)
    need = lib().nrpn_conv3d_wgrad_workspace_bytes(ctypes.byref(d))
    if need == 0:
        raise ValueError("conv3d_wgrad: unsupported shape (cout % 8 == 0, cin % 32 == 0, cin <= 256 or cin % 256 == 0)")
    ws = _workspace(need, dys[0].device)
    d.dw, d.workspace, d.workspace_bytes = dw.data_ptr(), ws.data_ptr(), ws.numel()
    check(lib().nrpn_conv3d_wgrad(ctypes.byref(d), _stream()), "conv3d_wgrad")
    return dw


def bias_grad(dy: torch.Tensor) -> torch.Tensor:
    """(..., C) 16-bit channels-last dY -> db (C) fp32 = sum over every row (bit-reproducible two-stage reduction)."""
    f16 = _act16(dy, "dy")
    c = int(dy.shape[-1])
    rows = dy.numel() // c
    db = torch.empty((c,), dtype=torch.float32, device=dy.device)
    ws = _workspace(lib().nrpn_bias_grad_workspace_bytes(c), dy.device)
    check(lib().nrpn_bias_grad(_ptr(dy), rows, c, c, f16, _ptr(db), _ptr(ws), ws.numel(), _stream()), "bias_grad")
    return db


def relu_backward_(dy: torch.Tensor, act: torch.Tensor) -> torch.Tensor:
    """dy *= (act > 0) in place (16-bit tensors of equal shape): the ReLU of a conv + bias + ReLU layer, backwards."""
    f16 = _act16(dy, "dy")
    if _act16(act, "act") != f16 or act.shape != dy.shape:
        raise ValueError("relu_backward_: dy and act must have the same dtype and shape")
    check(lib().nrpn_relu_backward(_ptr(dy), _ptr(act), dy.numel(), f16, _stream()), "relu_backward")
    return dy


def pack_stem_input(grid: torch.Tensor, out: Optional[torch.Tensor] = None, dtype=torch.bfloat16, density_to_alpha: bool = False) -> torch.Tensor:
    """(N,4,X,Y,Z) fp32 -> (N, ceil(X/2), ceil(Y/2), ceil(Z/2)+1, 64) bf16 (or fp16: dtype of `out`).
    `grid` may be contiguous NCDHW or the channels-last view the reference's dataset yields (memory (N,X,Y,Z,4))."""
    if isinstance(grid, torch.Tensor) and grid.is_cuda and grid.dtype == torch.uint8 and grid.dim() == 5:
        # raw uint8 grid in its on-disk order: normalised (/ 255) on the device
        if not grid.permute(0, 2, 3, 4, 1).is_contiguous():
            raise ValueError("nerf_rpn_b200: uint8 grids must be the (N,4,X,Y,Z) view of a contiguous (N,X,Y,Z,4) array")
        n, c, x, y, z = grid.shape
        shape = (n, (x + 1) // 2, (y + 1) // 2, (z + 1) // 2 + 1, 64)
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=grid.device)
        check(lib().nrpn_pack_stem_input_u8(_ptr(grid), n, x, y, z, _ptr(out), _act16(out, "out"), _stream()), "pack_stem_input_u8")
        return out
    if not isinstance(grid, torch.Tensor) or not grid.is_cuda or grid.dtype != torch.float32 or grid.dim() != 5:
        raise RuntimeError("nerf_rpn_b200: grid must be a 5-D fp32 (or channels-last uint8) CUDA tensor")
    cl = is_channels_last_grid(grid)
    if not cl and not grid.is_contiguous():
        raise ValueError("nerf_rpn_b200: grid must be contiguous (N,4,X,Y,Z) or a permuted view of a contiguous (N,X,Y,Z,4) array")
    n, c, x, y, z = grid.shape
    if c != 4:
        raise ValueError("stem packing expects 4 input channels (RGB + density)")
    shape = (n, (x + 1) // 2, (y + 1) // 2, (z + 1) // 2 + 1, 64)
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=grid.device)
    check(lib().nrpn_pack_stem_input_ex(_ptr(grid), n, x, y, z, _ptr(out), _act16(out, "out"), int(cl), int(bool(density_to_alpha)), _stream()),
          "pack_stem_input")
    return out


def maxpool3d_k3s2(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(N,X,Y,Z,C) bf16 / fp16 channels-last -> k3 s2 p1 max pool."""
    f16 = _act16(x, "x")
    n, X, Y, Z, C = x.shape
    shape = (n, (X - 1) // 2 + 1, (Y - 1) // 2 + 1, (Z - 1) // 2 + 1, C)
    if out is None:
        out = torch.empty(shape, dtype=x.dtype, device=x.device)
    if out.dtype != x.dtype:
        raise TypeError("maxpool3d_k3s2: out must have the dtype of x")
    check(lib().nrpn_maxpool3d_k3s2(_ptr(x), n, X, Y, Z, C, _ptr(out), f16, _stream()), "maxpool3d_k3s2")
    return out


def maxpool3d_k2s2_ceil(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(N,X,Y,Z,C) bf16 / fp16 channels-last -> MaxPool3d(2, 2, ceil_mode=True)."""
    f16 = _act16(x, "x")
    n, X, Y, Z, C = x.shape
    if out is None:
        out = torch.empty((n, (X + 1) // 2, (Y + 1) // 2, (Z + 1) // 2, C), dtype=x.dtype, device=x.device)
    check(lib().nrpn_maxpool3d_k2s2_ceil(_ptr(x), n, X, Y, Z, C, _ptr(out), f16, _stream()), "maxpool3d_k2s2_ceil")
    return out


def pack_stem_input_s1(grid: torch.Tensor, out: Optional[torch.Tensor] = None, dtype=torch.bfloat16) -> torch.Tensor:
    """(N,4,X,Y,Z) fp32 -> (N, X, Y+1, Z, 64) bf16 / fp16 (stride-1 7^3 stem)."""
    grid = _req(grid, torch.float32, "grid")
    n, c, x, y, z = grid.shape
    if c != 4:
        raise ValueError("stem packing expects 4 input channels (RGB + density)")
    if out is None:
        out = torch.empty((n, x, y + 1, z, 64), dtype=dtype, device=grid.device)
    check(lib().nrpn_pack_stem_input_s1(_ptr(grid), n, x, y, z, _ptr(out), _act16(out, "out"), _stream()), "pack_stem_input_s1")
    return out


# ------------------------------------------------------------------------------------------------ rpn post
def make_rpn_desc(preds: List[torch.Tensor], grids, strides, cells, num_anchors: int, rotated: bool, pre_nms_top_n: int,
                  post_nms_top_n: int, nms_thresh: float, score_thresh: float, min_size: float, mesh, valid=None) -> RpnDesc:
    d = RpnDesc()
    d.n_levels = len(preds)
    for l, p in enumerate(preds):
        p = _req(p, torch.float32, f"pred[{l}]")
        lv = d.level[l]
        lv.pred = p.data_ptr(); lv.ld = int(p.shape[-1])
        lv.gx, lv.gy, lv.gz = (int(v) for v in grids[l])
        lv.sx, lv.sy, lv.sz = (int(v) for v in strides[l])
        for a in range(num_anchors):
            for k in range(6):
                d.cell_anchors[l][a][k] = float(cells[l][a][k])
    d.num_anchors = int(num_anchors); d.rotated = int(bool(rotated))
    d.pre_nms_top_n, d.post_nms_top_n = int(pre_nms_top_n), int(post_nms_top_n)
    d.nms_thresh, d.score_thresh, d.min_size = float(nms_thresh), float(score_thresh), float(min_size)
    for k in range(3):
        d.mesh[k] = int(mesh[k]); d.valid[k] = int((valid or mesh)[k])
    return d


def rpn_proposals(desc: RpnDesc, device, out=None, workspace: Optional[torch.Tensor] = None):
    """Runs the device-side post-processing; returns (boxes, scores, levels, count) device tensors (count int32 (1,))."""
    box_dim = 7 if desc.rotated else 6
    k = desc.post_nms_top_n
    if out is None:
        boxes = torch.empty((k, box_dim), dtype=torch.float32, device=device)
        scores = torch.empty((k,), dtype=torch.float32, device=device)
        levels = torch.empty((k,), dtype=torch.float32, device=device)
        count = torch.zeros((1,), dtype=torch.int32, device=device)
    else:
        boxes, scores, levels, count = out
    wsb = lib().nrpn_rpn_workspace_bytes(ctypes.byref(desc))
    if wsb == 0:
        raise ValueError("nerf_rpn_b200: invalid RPN descriptor")
    ws = workspace if workspace is not None else _workspace(wsb, device)
    check(lib().nrpn_rpn_proposals(ctypes.byref(desc), _ptr(boxes), _ptr(scores), _ptr(levels), _ptr(count), _ptr(ws),
                                   ws.numel(), _stream()), "rpn_proposals")
    return boxes, scores, levels, count


# ------------------------------------------------------------------------------------------------ FCOS
def groupnorm_relu_(levels: Sequence[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, relu: bool = True,
                    groups: int = 32, workspace: Optional[torch.Tensor] = None):
    """In-place GroupNorm(groups, C) (+ReLU) on channels-last bf16 tensors (N, X, Y, Z, C) that share gamma / beta."""
    n, c = levels[0].shape[0], levels[0].shape[-1]
    arr = (GnLevel * len(levels))()
    for i, t in enumerate(levels):
        f16 = _act16(t, f"levels[{i}]")
        arr[i].x = t.data_ptr(); arr[i].voxels = int(t.shape[1] * t.shape[2] * t.shape[3])
    need = lib().nrpn_groupnorm_workspace_bytes(len(levels), n)
    ws = workspace if workspace is not None else _workspace(need, levels[0].device)
    check(lib().nrpn_groupnorm_relu(arr, len(levels), n, c, groups, _ptr(gamma), _ptr(beta), float(eps), int(relu), f16, _ptr(ws),
                                    ws.numel(), _stream()), "groupnorm_relu")


def make_fcos_desc(cls_preds, reg_preds, grids, strides, scales, use_obb, pre_nms_thresh, pre_nms_top_n, nms_thresh,
                   post_nms_top_n, min_size, grid_size, padded=False) -> FcosDesc:
    d = FcosDesc()
    d.n_levels = len(cls_preds)
    for l, (c, r) in enumerate(zip(cls_preds, reg_preds)):
        c = _req(c, torch.float32, f"cls[{l}]"); r = _req(r, torch.float32, f"reg[{l}]")
        lv = d.level[l]
        lv.cls, lv.reg = c.data_ptr(), r.data_ptr()
        lv.ld_cls, lv.ld_reg = int(c.shape[-1]), int(r.shape[-1])
        lv.gx, lv.gy, lv.gz = (int(v) for v in grids[l])
        lv.stride, lv.scale = int(strides[l]), float(scales[l])
    d.use_obb = int(bool(use_obb))
    d.pre_nms_top_n, d.post_nms_top_n = int(pre_nms_top_n), int(post_nms_top_n)
    d.pre_nms_thresh, d.nms_thresh, d.min_size = float(pre_nms_thresh), float(nms_thresh), float(min_size)
    for k in range(3):
        d.grid_size[k] = int(grid_size[k])
    d.padded = int(bool(padded))
    return d


def fcos_proposals(desc: FcosDesc, device, out=None, workspace: Optional[torch.Tensor] = None):
    """Returns (boxes (cap, 1+6|7) with the level id in column 0, scores (cap,), count int32 (1,)) device tensors."""
    cap = lib().nrpn_fcos_max_proposals(ctypes.byref(desc))
    if cap <= 0:
        raise ValueError("nerf_rpn_b200: invalid FCOS descriptor")
    dim = 7 if desc.use_obb else 6
    if out is None:
        boxes = torch.empty((cap, 1 + dim), dtype=torch.float32, device=device)
        scores = torch.empty((cap,), dtype=torch.float32, device=device)
        count = torch.zeros((1,), dtype=torch.int32, device=device)
    else:
        boxes, scores, count = out
    wsb = lib().nrpn_fcos_workspace_bytes(ctypes.byref(desc))
    ws = workspace if workspace is not None else _workspace(wsb, device)
    check(lib().nrpn_fcos_proposals(ctypes.byref(desc), _ptr(boxes), _ptr(scores), _ptr(count), _ptr(ws), ws.numel(), _stream()),
          "fcos_proposals")
    return boxes, scores, count


# ------------------------------------------------------------------------------------------------ FCOS training loss (fcos/loss.py)
FCOS_SIZES_OF_INTEREST = ((-1.0, 16.0), (16.0, 32.0), (32.0, 64.0), (64.0, 100000000.0))          # loss.py:263-268
FCOS_LOSS_TYPES = {"smooth_l1": 0, "iou": 1, "linear_iou": 2, "giou": 3}


def fcos_targets(locations: torch.Tensor, n_points: Sequence[int], strides: Sequence[int], gt: torch.Tensor, center_sampling_radius: float,
                 norm_reg_targets: bool = True):
    """One scene: locations (P,3) f32 (levels concatenated), gt (G, 6|7) -> labels (P) f32 in {0,1}, reg_targets (P, 6|8) f32
    (prepare_targets / compute_targets_for_locations[_obb], loss.py:262-441)."""
    locations = _req(locations, torch.float32, "locations")
    gt = _req(gt, torch.float32, "gt")
    if len(n_points) != len(strides) or not 1 <= len(n_points) <= _lib.MAX_LEVELS:
        raise ValueError(f"nerf_rpn_b200: FCOS targets take 1..{_lib.MAX_LEVELS} levels (object_sizes_of_interest has four rows, fcos/loss.py:263-268)")
    if gt.dim() != 2 or gt.shape[1] not in (6, 7) or locations.shape != (sum(n_points), 3):
        raise ValueError("nerf_rpn_b200: gt must be (G, 6|7) and locations (sum(n_points), 3)")
    d = FcosTargetDesc()
    d.n_levels = len(n_points)
    for l, (n, s) in enumerate(zip(n_points, strides)):
        d.n_points[l], d.stride[l] = int(n), int(s)
        d.size_lo[l], d.size_hi[l] = FCOS_SIZES_OF_INTEREST[l]
    d.center_sampling_radius = float(center_sampling_radius)
    d.norm_reg_targets = int(bool(norm_reg_targets))
    p, dim = locations.shape[0], 8 if gt.shape[1] == 7 else 6
    labels = torch.empty((p,), dtype=torch.float32, device=locations.device)
    reg = torch.empty((p, dim), dtype=torch.float32, device=locations.device)
    check(lib().nrpn_fcos_targets(ctypes.byref(d), _ptr(locations), _ptr(gt) if gt.shape[0] else ctypes.c_void_p(0), int(gt.shape[0]), int(gt.shape[1]),
                                  _ptr(labels), _ptr(reg), _stream()), "fcos_targets")
    return labels, reg


def fcos_loss_sums(box_cls, box_regression, centerness, labels: torch.Tensor, reg_targets: torch.Tensor, mask: Optional[torch.Tensor],
                   loss_type: str, use_obb: bool, additional_l1: bool, want_grad: bool = True):
    """The head's per-level NCDHW outputs + targets (N,P) / (N,P,D) [+ mask (N,P) u8] -> (sums (8,) f64 on the device, centerness targets (N,P),
    raw gradients (dcls, dreg, dctr lists shaped like the inputs) or None); see nrpn_fcos_loss in include/nerf_rpn_b200.h."""
    n_lvl = len(box_cls)
    if not (n_lvl == len(box_regression) == len(centerness)) or not 1 <= n_lvl <= _lib.MAX_LEVELS:
        raise ValueError("nerf_rpn_b200: FCOS loss takes the same 1..4 levels for box_cls, box_regression and centerness")
    dim = 8 if use_obb else 6
    n = box_cls[0].shape[0]
    d = FcosLossDesc()
    d.n_levels, d.n_images, d.use_obb, d.additional_l1 = n_lvl, n, int(bool(use_obb)), int(bool(additional_l1))
    d.loss_type = FCOS_LOSS_TYPES[loss_type]
    grads = ([], [], []) if want_grad else None
    total = 0
    for l in range(n_lvl):
        c, r, t = _req(box_cls[l], torch.float32, "box_cls"), _req(box_regression[l], torch.float32, "box_regression"), _req(centerness[l], torch.float32, "centerness")
        pl = c[0, 0].numel()
        if c.shape[:2] != (n, 1) or r.shape[:2] != (n, dim) or t.shape[:2] != (n, 1) or r[0, 0].numel() != pl or t[0, 0].numel() != pl:
            raise ValueError("nerf_rpn_b200: FCOS head outputs must be (N,1,w,l,h), (N,6|8,w,l,h), (N,1,w,l,h) per level")
        L = d.level[l]
        L.cls, L.reg, L.ctr, L.n_points = c.data_ptr(), r.data_ptr(), t.data_ptr(), pl
        if want_grad:
            for lst, src in zip(grads, (c, r, t)):
                lst.append(torch.empty_like(src))
            L.dcls, L.dreg, L.dctr = grads[0][l].data_ptr(), grads[1][l].data_ptr(), grads[2][l].data_ptr()
        total += pl
    labels = _req(labels, torch.float32, "labels"); reg_targets = _req(reg_targets, torch.float32, "reg_targets")
    if labels.shape != (n, total) or reg_targets.shape != (n, total, dim):
        raise ValueError("nerf_rpn_b200: labels must be (N, P) and reg_targets (N, P, 6|8) with P = all levels' locations")
    if mask is not None:
        mask = _req(mask, torch.uint8, "mask")
        if mask.shape != (n, total):
            raise ValueError("nerf_rpn_b200: mask must be (N, P)")
    dev = labels.device
    sums = torch.empty((8,), dtype=torch.float64, device=dev)
    ct = torch.empty((n, total), dtype=torch.float32, device=dev)
    ws = _workspace(lib().nrpn_fcos_loss_workspace_bytes(), dev)
    check(lib().nrpn_fcos_loss(ctypes.byref(d), _ptr(labels), _ptr(reg_targets), _ptr(mask), _ptr(ct), _ptr(sums), _ptr(ws), ws.numel(), _stream()),
          "fcos_loss")
    return sums, ct, grads


# ------------------------------------------------------------------------------------------------ Swin
def patch_embed_pack(grid: torch.Tensor, out: torch.Tensor):
    grid = _req(grid, torch.float32, "grid")
    n, c, x, y, z = grid.shape
    check(lib().nrpn_patch_embed_pack(_ptr(grid), n, x, y, z, _ptr(out), _act16(out, "out"), _stream()), "patch_embed_pack")
    return out


def layernorm(x: torch.Tensor, out: torch.Tensor, c: int, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5):
    """x, out: (..., ld) bf16 channels-last; normalises the first c channels of every row."""
    tokens = x.numel() // x.shape[-1]
    check(lib().nrpn_layernorm(_ptr(x), int(x.shape[-1]), _ptr(out), int(out.shape[-1]), tokens, int(c), _ptr(gamma), _ptr(beta),
                               float(eps), _act16(x, "x"), _stream()), "layernorm")
    return out


def patch_merge_ln(x: torch.Tensor, out: torch.Tensor, c: int, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5):
    n, h, w, d, ld = x.shape
    check(lib().nrpn_patch_merge_ln(_ptr(x), int(ld), n, h, w, d, int(c), _ptr(out), _ptr(gamma), _ptr(beta), float(eps),
                                    _act16(x, "x"), _stream()), "patch_merge_ln")
    return out


def window_attention(qkv: torch.Tensor, out: torch.Tensor, qkv_bias: torch.Tensor, table: torch.Tensor, c: int, heads: int, shift: int):
    n, h, w, d, ld = qkv.shape
    check(lib().nrpn_window_attention(_ptr(qkv), int(ld), _ptr(out), int(out.shape[-1]), _ptr(qkv_bias), _ptr(table), n, h, w, d, int(c),
                                      int(heads), int(shift), _act16(qkv, "qkv"), _stream()), "window_attention")
    return out
