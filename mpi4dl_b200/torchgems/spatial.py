"""torchgems.spatial -- drop-in surface of the reference's spatially-partitioned layers, backed by
libspconv.so (hand-written sm_100a CUDA; include/spconv.h).

Mirrors reference src/torchgems/spatial.py:
    conv_spatial          spatial.py:25-1029   (nn.Conv2d subclass; .weight/.bias state_dict keys)
    halo_exchange_layer   spatial.py:1032-1413
    Pool                  spatial.py:1416-1509
Same constructor signatures, attribute names (halo_len_height/width, neighbours,
rank_neighbours, spatial_local_rank ...), assertions and error texts.  What is different is
everything underneath: no ZeroPad2d copy, no per-direction clone / isend / irecv fenced by
torch.cuda.synchronize(), no 8 slice-assign unpack copies, no cuDNN.  One pack kernel writes
all outgoing strips (into the neighbours' mailboxes over NVLink when the peer transport is
active), and the conv / pool kernels read tile + strips in place.

There is NO CPU or PyTorch fallback: forward() raises unless the tensor is on a CUDA device and
libspconv.so loads.
"""
import ctypes as C
import math
import os

import torch
import torch.distributed as dist
import torch.nn as nn

from .. import _lib
from . import halo_transport

# 3x3 neighbour stencil (reference spatial.py:961-964):  0 1 2 / 3 4 5 / 6 7 8
_DIRS = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 0), (0, 1), (1, -1), (1, 0), (1, 1)]


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# Math of fp32 convolutions: "ieee" (default) runs them in exact fp32 on the direct kernels, "tf32" lets the tensor
# cores read their operands as TF32 (10-bit mantissa, fp32 accumulate and output).  The initial value comes from the
# SPCONV_FP32_MATH environment variable.  bf16 convolutions and modules with an explicit `algo` are not affected.
_FP32_MATH_MODES = ("ieee", "tf32")


def _parse_fp32_math(mode, source):
    if mode not in _FP32_MATH_MODES:
        raise ValueError("%s: fp32 math must be one of %s, got %r" % (source, ", ".join(_FP32_MATH_MODES), mode))
    return mode


_fp32_math = _parse_fp32_math(os.environ.get("SPCONV_FP32_MATH", "ieee"), "SPCONV_FP32_MATH")


def set_fp32_math(mode):
    """Select the math of fp32 conv_spatial / local_conv2d layers: "ieee" (exact fp32, the default) or "tf32"
    (tensor cores with TF32 operands)."""
    global _fp32_math
    _fp32_math = _parse_fp32_math(mode, "set_fp32_math")


def get_fp32_math():
    return _fp32_math


def _algo_for(algo, dtype):
    """Descriptor algo of a module whose `algo` attribute is `algo`: AUTO becomes TF32 for fp32 tensors when the
    fp32 math is "tf32"; an explicitly chosen algo is passed through."""
    if algo == _lib.SPC_ALGO_AUTO and dtype == torch.float32 and _fp32_math == "tf32":
        return _lib.SPC_ALGO_TF32
    return algo


def _require_cuda(t, who):
    if not t.is_cuda:
        raise RuntimeError(
            "%s: input must be a CUDA tensor -- the spatial conv path runs only on libspconv "
            "(sm_100a); there is no CPU fallback" % who)


def _workspace(nbytes, device):
    if nbytes == 0:
        return None, C.c_void_p(None)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return ws, C.c_void_p(ws.data_ptr())


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


class _SpatialTopology:
    """Rank-grid arithmetic shared by the three layers (reference spatial.py:868-1017,
    1276-1392).  Kept as a mixin so attribute names match the reference's."""

    def _init_topology(self, local_rank, spatial_size, num_spatial_parts, slice_method):
        self.local_rank = local_rank
        if isinstance(num_spatial_parts, list):  # spatial.py:51-60 / :157-168
            self.spatial_local_rank, self.num_spatial_parts = self.get_local_spatial_rank(
                num_spatial_parts, local_rank)
        else:
            self.spatial_local_rank = local_rank
            self.num_spatial_parts = num_spatial_parts
        self.spatial_size = spatial_size
        self.slice_method = slice_method

    def get_local_spatial_rank(self, num_spatial_parts_list, local_rank):
        temp_sum = 0
        for parts in num_spatial_parts_list:
            if local_rank < temp_sum + parts:
                return local_rank - temp_sum, parts
            temp_sum += parts
        raise ValueError("local_rank %d is not a spatial rank of %s" % (local_rank, num_spatial_parts_list))

    def _grid(self):
        P = self.num_spatial_parts
        if self.slice_method == "square":
            q = int(math.sqrt(P))
            return q, q
        if self.slice_method == "vertical":
            return 1, P
        if self.slice_method == "horizontal":
            return P, 1
        raise ValueError("slice_method must be square|vertical|horizontal, got %r" % (self.slice_method,))

    def get_neighbours(self):
        """0/1 mask over the 3x3 stencil (spatial.py:941-1017)."""
        if self.spatial_local_rank < self.num_spatial_parts:
            self.ENABLE_SPATIAL = True
        else:
            self.ENABLE_SPATIAL = False
            self.neighbours = None
            return
        self.spatial_rank = self.spatial_local_rank
        rows, cols = self._grid()
        # the reference indexes the grid by local_rank (spatial.py:972-973), which only works for
        # the first spatial stage; the rank inside the stage is what is meant.
        r, c = self.spatial_local_rank // cols, self.spatial_local_rank % cols
        self.neighbours = []
        for dr, dc in _DIRS:
            rr, cc = r + dr, c + dc
            ok = (dr, dc) != (0, 0) and 0 <= rr < rows and 0 <= cc < cols
            self.neighbours.append(1 if ok else 0)

    def set_neighbours_based_on_kernel_size(self):
        """1-D kernels exchange along one axis only (spatial.py:921-939)."""
        if self.kernel_size[0] == 1:
            for i in (0, 1, 2, 6, 7, 8):
                self.neighbours[i] = 0
        if self.kernel_size[1] == 1:
            for i in (0, 3, 6, 2, 5, 8):
                self.neighbours[i] = 0

    def get_neighbours_rank(self):
        """World ranks of the neighbours (spatial.py:868-919), incl. the GEMS-inverse mirror."""
        rows, cols = self._grid()
        self.rank_neighbours = []
        for i, (dr, dc) in enumerate(_DIRS):
            if self.neighbours[i] == 1:
                self.rank_neighbours.append(self.local_rank + dr * cols + dc)
            else:
                self.rank_neighbours.append(-1)
        # Which world ranks hold the neighbour tiles.  The reference knows two cases (spatial.py:912-919): the
        # layer's local_rank IS this process's world rank, or -- GEMS inverse replica -- the replica lives on
        # the mirrored rank line (world_size-1-r).  A third case exists once pipelines are data-parallel
        # (world = k * mp_size, mp_pipeline's replica base): the tile line starts at this replica's first rank.
        if dist.is_available() and dist.is_initialized() and self.local_rank != dist.get_rank():
            world_size, rank = dist.get_world_size(), dist.get_rank()
            base = rank - self.local_rank
            if world_size - 1 - rank == self.local_rank or base <= 0:
                # (base <= 0: the scripts also BUILD the spatial cells on ranks that never run them, with
                # local_rank = position % tiles -- keep the reference's formula there, the layers stay idle)
                for i in range(9):
                    if self.neighbours[i] == 1:
                        self.rank_neighbours[i] = world_size - 1 - self.rank_neighbours[i]
            else:
                for i in range(9):
                    if self.neighbours[i] == 1:
                        self.rank_neighbours[i] += base

    def set_tags(self):
        # kept for API compatibility (spatial.py:170-172); stream/flag ordering replaces MPI tags
        self.send_tag = [100, 200, 300, 400, 500, 600, 700, 800, 900]
        self.recv_tag = [900, 800, 700, 600, 500, 400, 300, 200, 100]

    # ---- halo exchange ---------------------------------------------------------------------
    def _exchange(self, x, hh, hw):
        """Send the edge strips of `x` to the neighbours and return the 9 received strips
        (None where there is no neighbour).  Replaces start_halo_exchange / end_halo_exchange
        (spatial.py:336-403)."""
        if self.neighbours is None or not any(self.neighbours):
            return [None] * 9
        tr = halo_transport.get_transport(x.device)
        return tr.exchange(self, x, hh, hw, self.neighbours, self.rank_neighbours)


def _strip_shape(i, N, Cc, H, W, hh, hw):
    dr, dc = _DIRS[i]
    return (N, Cc, H if dr == 0 else hh, W if dc == 0 else hw)


_comm_streams = {}


def _comm_stream(device):
    """High-priority side stream for the halo exchange (one per device)."""
    key = (device.type, device.index)
    if key not in _comm_streams:
        _comm_streams[key] = torch.cuda.Stream(device=device, priority=-1)
    return _comm_streams[key]


class _ConvSpatialFn(torch.autograd.Function):
    """fprop / dgrad / wgrad through the C ABI.  Halo strips enter as constants: the reference
    unpacks them with in-place slice assignment of detached tensors, so no gradient ever flows
    back to a neighbour (SURVEY 8a N2)."""

    @staticmethod
    def forward(ctx, x, weight, bias, desc_args, *strips):
        """strips[0:9] are the received halo strips; an optional 10th element is a CUDA event that
        fires when they have arrived (exchange running on the comm stream): then the interior pass
        is launched first and only the boundary strips wait for the event."""
        L = _lib.lib()
        d = _lib.ConvDesc(*desc_args)
        ctx.n_tail = len(strips)
        ready = strips[9] if len(strips) > 9 else None
        strips = strips[:9]
        Ho, Wo = C.c_int(), C.c_int()
        L.spc_conv_out_shape(C.byref(d), C.byref(Ho), C.byref(Wo))
        y = torch.empty((d.N, d.K, Ho.value, Wo.value), dtype=x.dtype, device=x.device)
        halo = _lib.make_halo(strips)
        ws, wsp = _workspace(L.spc_conv_workspace_bytes(C.byref(d), 0), x.device)
        if ready is None:
            _lib.check(L.spc_conv2d_fwd(C.byref(d), _ptr(x), C.byref(halo), _ptr(weight), _ptr(bias), _ptr(y), wsp,
                                        0 if ws is None else ws.numel(), _stream()), "spc_conv2d_fwd")
        else:
            _lib.check(L.spc_conv2d_fwd_interior(C.byref(d), _ptr(x), _ptr(weight), _ptr(bias), _ptr(y), wsp,
                                                 0 if ws is None else ws.numel(), _stream()), "spc_conv2d_fwd_interior")
            torch.cuda.current_stream().wait_event(ready)
            _lib.check(L.spc_conv2d_fwd_boundary(C.byref(d), _ptr(x), C.byref(halo), _ptr(weight), _ptr(bias), _ptr(y),
                                                 _stream()), "spc_conv2d_fwd_boundary")
        ctx.desc_args = desc_args
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, weight, *[s for s in strips if s is not None])
        ctx.strip_mask = [s is not None for s in strips]
        return y

    @staticmethod
    def backward(ctx, gy):
        L = _lib.lib()
        saved = ctx.saved_tensors
        x, weight = saved[0], saved[1]
        it = iter(saved[2:])
        strips = [next(it) if m else None for m in ctx.strip_mask]
        d = _lib.ConvDesc(*ctx.desc_args)
        gy = gy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            ws, wsp = _workspace(L.spc_conv_workspace_bytes(C.byref(d), 1), x.device)
            _lib.check(L.spc_conv2d_dgrad(C.byref(d), _ptr(gy), _ptr(weight), _ptr(dx), wsp,
                                          0 if ws is None else ws.numel(), _stream()), "spc_conv2d_dgrad")
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dw32 = torch.empty(weight.shape, dtype=torch.float32, device=x.device)
            db32 = torch.empty(d.K, dtype=torch.float32, device=x.device) if ctx.has_bias else None
            halo = _lib.make_halo(strips)
            ws, wsp = _workspace(L.spc_conv_workspace_bytes(C.byref(d), 2), x.device)
            _lib.check(L.spc_conv2d_wgrad(C.byref(d), _ptr(x), C.byref(halo), _ptr(gy), _ptr(dw32), _ptr(db32), 0,
                                          wsp, 0 if ws is None else ws.numel(), _stream()), "spc_conv2d_wgrad")
            dw = dw32.to(weight.dtype)
            db = db32.to(weight.dtype) if db32 is not None else None
        return (dx, dw, db, None) + (None,) * ctx.n_tail


class conv_spatial(nn.Conv2d, _SpatialTopology):
    """Spatially-partitioned Conv2d (reference spatial.py:25-1029)."""

    def __init__(self, local_rank, spatial_size, num_spatial_parts, in_channels, out_channels, kernel_size,
                 stride=1, padding=0, dilation=1, groups=1, bias=True, halo_len=None, padding_mode="zeros",
                 slice_method="square"):
        if isinstance(kernel_size, int):
            kernel_size = (kernel_size, kernel_size)
        if isinstance(padding, int):
            padding = (padding, padding)
        self._init_topology(local_rank, spatial_size, num_spatial_parts, slice_method)

        self.fused_halo = halo_len is not None
        if halo_len is not None:
            # D2 "fused halo" variant (spatial.py:67-111): the tile already carries its halo (one wide
            # halo_exchange_layer per block), so there is NO exchange here; only the sides that are
            # true image borders get `padding` zeros, the sides facing a neighbour get none and the
            # output shrinks there.  The reference hard-codes the 2x2 grid (ranks 0-3); here the
            # border sides follow from the rank grid, which is the same table for square-4.
            assert halo_len == 0, "Error: Custom Halo Len is not supported (only halo_len=0 is supported)"
            # padding = (k-1)//2: zero padding on the image-border sides only (amoebanet_d2.py);
            # padding = 0: no padding on any side -- a valid convolution (resnet_spatial_d2.py:135-139 passes 0, and the
            # reference's table puts `padding` on the border sides, spatial.py:75-104)
            self._fused_valid = tuple(padding) == (0, 0)
            assert self._fused_valid or ((kernel_size[0] - 1) // 2 == padding[0] and (kernel_size[1] - 1) // 2 == padding[1]), \
                "conv_spatial(halo_len=0): padding must be (k-1)//2 or 0"
            padding = ((kernel_size[0] - 1) // 2, (kernel_size[1] - 1) // 2)
        # spatial.py:115-121
        self.halo_len_height = int((kernel_size[0] - 1) / 2)
        self.halo_len_width = int((kernel_size[1] - 1) / 2)
        assert (self.halo_len_height == padding[0] or self.halo_len_width == padding[1]), \
            "Spatial not supported yet for this configuration"
        # the base Conv2d carries padding=0, dilation=1, groups=1 exactly like the reference
        # (spatial.py:130-140), so state_dict keys / shapes are identical.
        nn.Conv2d.__init__(self, in_channels, out_channels, kernel_size, stride=stride, padding=0, dilation=1,
                           groups=1, bias=bias, padding_mode="zeros")
        self.neighbours = None
        self.rank_neighbours = [-1] * 9
        if self.halo_len_height > 0 or self.halo_len_width > 0:
            self.get_neighbours()
            if self.neighbours is not None:
                self.set_neighbours_based_on_kernel_size()
                self.get_neighbours_rank()
        if self.fused_halo:
            nb = self.neighbours or [0] * 9
            # sides with a neighbour: (top, bottom, left, right)
            self._inner_sides = (True,) * 4 if self._fused_valid else (bool(nb[1]), bool(nb[7]), bool(nb[3]), bool(nb[5]))
            self.halo_len_height_d2, self.halo_len_width_d2 = 0, 0
            self.neighbours = None          # never exchanges
        self.set_tags()
        self.algo = _lib.SPC_ALGO_AUTO

    def _fused_pre(self, x):
        """D2 variant, strided: a side that faces a neighbour carries NO padding, so the sampling phase of a strided
        convolution starts at the tile's first row / column, while the "same"-padded kernel starts `pad` before it.
        When pad % stride != 0 the two grids never coincide; prepending (stride - pad % stride) dummy rows / columns
        (zeros; no valid output window ever reads them) re-aligns them.  Returns (x', extra_top, extra_left)."""
        sh, sw = self.stride
        ph, pw = self.halo_len_height, self.halo_len_width
        top, _, left, _ = self._inner_sides
        et = (sh - ph % sh) % sh if (top and ph % sh) else 0
        el = (sw - pw % sw) % sw if (left and pw % sw) else 0
        if et or el:
            x = torch.nn.functional.pad(x, (el, 0, et, 0))
        return x, et, el

    def _crop_fused(self, y, H, W, et=0, el=0):
        """Drop the output rows / columns whose window would reach past a neighbour-facing edge
        (those sides carry no padding in the D2 variant).  H, W: the ORIGINAL tile extent; et / el: dummy rows /
        columns prepended by _fused_pre."""
        R, S = self.kernel_size
        sh, sw = self.stride
        ph, pw = self.halo_len_height, self.halo_len_width
        Ho, Wo = y.shape[2], y.shape[3]
        top, bottom, left, right = self._inner_sides
        # output index p of the padded run has its window start at s*p - pad - extra (in original coordinates)
        y0 = (ph + et) // sh if top else 0                                  # first window starting at row 0
        y1 = min(Ho, (H - R + ph + et) // sh + 1) if bottom else Ho         # last window ending inside the tile
        x0 = (pw + el) // sw if left else 0
        x1 = min(Wo, (W - S + pw + el) // sw + 1) if right else Wo
        return y[:, :, y0:y1, x0:x1]

    def forward(self, tensor):
        _require_cuda(tensor, "conv_spatial")
        x = tensor.contiguous()
        if x.dtype != self.weight.dtype:
            raise RuntimeError("conv_spatial: input dtype %s != weight dtype %s" % (x.dtype, self.weight.dtype))
        hh, hw = self.halo_len_height, self.halo_len_width
        H0, W0 = x.shape[2], x.shape[3]
        et = el = 0
        if self.fused_halo:
            x, et, el = self._fused_pre(x)
        N, Cc, H, W = x.shape
        desc_args = (N, Cc, H, W, self.out_channels, self.kernel_size[0], self.kernel_size[1], self.stride[0],
                     self.stride[1], hh, hw, _lib.dtype_code(x.dtype), _algo_for(self.algo, x.dtype))
        exchange = (hh > 0 or hw > 0) and not self.fused_halo and self.neighbours is not None and any(self.neighbours)
        extra = ()
        with torch.no_grad():
            if exchange and halo_transport.overlap_enabled():
                # exchange on the comm stream, overlapped with the interior pass on this stream
                main = torch.cuda.current_stream()
                comm = _comm_stream(x.device)
                comm.wait_stream(main)                     # x is complete
                with torch.cuda.stream(comm):
                    strips = self._exchange(x, hh, hw)
                    ready = torch.cuda.Event()
                    ready.record(comm)
                x.record_stream(comm)
                for t in strips:
                    if t is not None:
                        t.record_stream(main)
                extra = (ready,)
            else:
                strips = self._exchange(x, hh, hw) if exchange else [None] * 9
        y = _ConvSpatialFn.apply(x, self.weight, self.bias, desc_args, *strips, *extra)
        if self.fused_halo:
            y = self._crop_fused(y, H0, W0, et, el)
        return y


class _HaloPadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, halo_len, *strips):
        L = _lib.lib()
        N, Cc, H, W = x.shape
        y = torch.empty((N, Cc, H + 2 * halo_len, W + 2 * halo_len), dtype=x.dtype, device=x.device)
        halo = _lib.make_halo(strips)
        _lib.check(L.spc_halo_pad(N, Cc, H, W, halo_len, halo_len, _lib.dtype_code(x.dtype), _ptr(x),
                                  C.byref(halo), _ptr(y), _stream()), "spc_halo_pad")
        ctx.halo_len = halo_len
        ctx.shape = (N, Cc, H, W)
        return y

    @staticmethod
    def backward(ctx, gy):
        L = _lib.lib()
        N, Cc, H, W = ctx.shape
        gy = gy.contiguous()
        dx = torch.empty(ctx.shape, dtype=gy.dtype, device=gy.device)
        _lib.check(L.spc_halo_crop(N, Cc, H, W, ctx.halo_len, ctx.halo_len, _lib.dtype_code(gy.dtype), _ptr(gy),
                                   _ptr(dx), _stream()), "spc_halo_crop")
        return (dx, None) + (None,) * 9


class halo_exchange_layer(nn.Module, _SpatialTopology):
    """Pad by `halo_len` and fill the pad from all 8 neighbours (reference spatial.py:1032-1413)."""

    def __init__(self, local_rank, spatial_size, num_spatial_parts, halo_len, padding_mode="zeros",
                 slice_method="square"):
        super(halo_exchange_layer, self).__init__()
        self._init_topology(local_rank, spatial_size, num_spatial_parts, slice_method)
        self.halo_len = halo_len
        self.get_neighbours()          # no kernel-shape pruning here (spatial.py:1329-1392)
        self.rank_neighbours = [-1] * 9
        if self.neighbours is not None:
            self.get_neighbours_rank()
        self.set_tags()

    def forward(self, tensor):
        _require_cuda(tensor, "halo_exchange_layer")
        x = tensor.contiguous()
        with torch.no_grad():
            strips = self._exchange(x, self.halo_len, self.halo_len) if self.halo_len > 0 else [None] * 9
        return _HaloPadFn.apply(x, self.halo_len, *strips)


class _PoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, desc_args, *strips):
        L = _lib.lib()
        d = _lib.PoolDesc(*desc_args)
        Ho = (d.H + 2 * d.pad - d.k) // d.stride + 1
        Wo = (d.W + 2 * d.pad - d.k) // d.stride + 1
        y = torch.empty((d.N, d.C, Ho, Wo), dtype=x.dtype, device=x.device)
        halo = _lib.make_halo(strips)
        _lib.check(L.spc_pool2d_fwd(C.byref(d), _ptr(x), C.byref(halo), _ptr(y), _stream()), "spc_pool2d_fwd")
        ctx.desc_args = desc_args
        ctx.save_for_backward(x, *[s for s in strips if s is not None])
        ctx.strip_mask = [s is not None for s in strips]
        return y

    @staticmethod
    def backward(ctx, gy):
        L = _lib.lib()
        saved = ctx.saved_tensors
        x = saved[0]
        it = iter(saved[1:])
        strips = [next(it) if m else None for m in ctx.strip_mask]
        d = _lib.PoolDesc(*ctx.desc_args)
        gy = gy.contiguous()
        dx = torch.empty_like(x)
        halo = _lib.make_halo(strips)
        _lib.check(L.spc_pool2d_bwd(C.byref(d), _ptr(x), C.byref(halo), _ptr(gy), _ptr(dx), _stream()),
                   "spc_pool2d_bwd")
        return (dx, None) + (None,) * 9


class Pool(nn.Module, _SpatialTopology):
    """Spatially-partitioned Max/Avg pooling (reference spatial.py:1416-1509)."""

    def __init__(self, local_rank, spatial_size, num_spatial_parts, kernel_size, stride, padding,
                 slice_method="square", dilation=1, return_indices=False, count_include_pad=True,
                 divisor_override=None, ceil_mode=False, operation=None):
        super(Pool, self).__init__()
        assert dilation == 1, "dilation > 1, Not Supported"
        assert return_indices == False, "return_indices == True, not supported"  # noqa: E712
        assert ceil_mode == False, "ceil model == True, not supported"  # noqa: E712
        assert operation != None, "operation is none"  # noqa: E711
        if isinstance(kernel_size, int):
            kernel_size = (kernel_size, kernel_size)
        if isinstance(stride, int):
            stride = (stride, stride)
        if isinstance(padding, int):
            padding = (padding, padding)
        halo_len = math.floor((kernel_size[0] - 1) / 2)
        assert kernel_size[0] == kernel_size[1], "Kernel Size should be same in pooling"
        assert stride[0] == stride[1], "Stride should be same in pooling"
        assert padding[0] == padding[1], "Padding should be same in pooling"
        assert halo_len == padding[0], "halo_len should be equal to padding in pool layers "
        assert divisor_override is None, "divisor_override is not supported"
        assert operation in ("MaxPool2d", "AvgPool2d"), "Only MaxPool2d and AvgPool2d are supported"
        self._init_topology(local_rank, spatial_size, num_spatial_parts, slice_method)
        self.halo_len = halo_len
        self.padding = padding
        self.kernel_size = kernel_size
        self.stride = stride
        self.operation = operation
        self.neighbours = None
        self.rank_neighbours = [-1] * 9
        if halo_len != 0:
            self.get_neighbours()
            if self.neighbours is not None:
                self.get_neighbours_rank()
        self.set_tags()

    def forward(self, tensor):
        _require_cuda(tensor, "Pool")
        x = tensor.contiguous()
        with torch.no_grad():
            strips = self._exchange(x, self.halo_len, self.halo_len) if self.halo_len > 0 else [None] * 9
        N, Cc, H, W = x.shape
        mode = _lib.SPC_POOL_MAX if self.operation == "MaxPool2d" else _lib.SPC_POOL_AVG
        desc_args = (N, Cc, H, W, self.kernel_size[0], self.stride[0], self.halo_len, mode,
                     _lib.dtype_code(x.dtype))
        return _PoolFn.apply(x, desc_args, *strips)


class local_conv2d(nn.Conv2d):
    """Conv2d on ONE tile with no exchange, on the libspconv kernels.  The D2 ("fused halo") cells of
    the reference feed plain nn.Conv2d(padding=0) -- cuDNN -- with tensors that already carry a wide
    halo (amoebanet_d2.py:159-191, 297-311); this is their replacement.  The kernel computes the
    "same"-padded convolution of the tile and the result is cropped to the padding actually asked
    for: padding=0 gives the valid convolution (interior windows never see the zero padding, so
    values are identical), padding=(k-1)//2 keeps everything.  Stride 1 only when cropping."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, bias=True):
        super().__init__(in_channels, out_channels, kernel_size, stride=stride, padding=padding, bias=bias)
        self._same = ((self.kernel_size[0] - 1) // 2, (self.kernel_size[1] - 1) // 2)
        for p_, s_ in zip(self.padding, self._same):
            assert p_ in (0, s_), "local_conv2d: padding must be 0 or (k-1)//2"
        assert tuple(self.padding) == self._same or tuple(self.stride) == (1, 1), \
            "local_conv2d: a valid (padding=0) convolution is supported for stride 1 only"
        self.algo = _lib.SPC_ALGO_AUTO

    def forward(self, tensor):
        _require_cuda(tensor, "local_conv2d")
        x = tensor.contiguous()
        if x.dtype != self.weight.dtype:
            raise RuntimeError("local_conv2d: input dtype %s != weight dtype %s" % (x.dtype, self.weight.dtype))
        N, Cc, H, W = x.shape
        ph, pw = self._same
        desc_args = (N, Cc, H, W, self.out_channels, self.kernel_size[0], self.kernel_size[1], self.stride[0],
                     self.stride[1], ph, pw, _lib.dtype_code(x.dtype), _algo_for(self.algo, x.dtype))
        y = _ConvSpatialFn.apply(x, self.weight, self.bias, desc_args, *([None] * 9))
        ch, cw = ph - self.padding[0], pw - self.padding[1]
        if ch or cw:
            y = y[:, :, ch:y.shape[2] - ch, cw:y.shape[3] - cw]
        return y


class local_pool2d(nn.Module):
    """Max/Avg pooling of one tile with no exchange (D2 cells: nn.AvgPool2d(3, padding=0),
    amoebanet_d2.py:88-117): the zero-padded pool of the tile, cropped when padding=0."""

    def __init__(self, operation, kernel_size, stride=1, padding=0):
        super().__init__()
        assert operation in ("MaxPool2d", "AvgPool2d")
        self.operation, self.kernel_size, self.stride, self.padding = operation, kernel_size, stride, padding
        self._same = (kernel_size - 1) // 2
        assert padding in (0, self._same) and (padding == self._same or stride == 1)

    def forward(self, tensor):
        _require_cuda(tensor, "local_pool2d")
        x = tensor.contiguous()
        N, Cc, H, W = x.shape
        mode = _lib.SPC_POOL_MAX if self.operation == "MaxPool2d" else _lib.SPC_POOL_AVG
        y = _PoolFn.apply(x, (N, Cc, H, W, self.kernel_size, self.stride, self._same, mode, _lib.dtype_code(x.dtype)),
                          *([None] * 9))
        c = self._same - self.padding
        return y[:, :, c:y.shape[2] - c, c:y.shape[3] - c] if c else y


# north_star aliases (BASELINE.json names that do not exist in the reference, SURVEY.md section 0)
pool_spatial = Pool
halo_exchange = halo_exchange_layer
