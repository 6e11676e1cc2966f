"""Sparse 3-D convolution layers and the reference's sparse U-Nets on libsstb200 (SURVEY 8f next-1).

Mirrors, by name / constructor kwargs / forward signature / state-dict keys:
  spconv layer surface used by the reference   mmdet3d/ops/spconv/{structure.py:22-69, modules.py:51-137, conv.py:26-206,259-446}
  make_sparse_convmodule, SparseBasicBlock      mmdet3d/ops/sparse_block.py:81-143, 216-289
  SparseUNet, SimpleSparseUNet, VirtualVoxelMixer   mmdet3d/models/middle_encoders/sparse_unet.py:15-505
The reference delegates the arithmetic to spconv (2.2.3 pinned in docs/overall_instructions.md:28, v1 vendored under
mmdet3d/ops/spconv); here a convolution is ONE launch of sstb200_spconv_forward over an output-stationary neighbour table built by
sstb200_spconv_table from the bitmap-rank index.  In eval mode `conv -> BatchNorm1d -> ReLU` chains (make_sparse_convmodule) and the
residual tail of SparseBasicBlock are folded into that launch's epilogue.

Weights keep the reference's checkpoint layout (kD, kH, kW, in, out) (write_spconv2.py:44-60 converts spconv2's to it on save).
There is no CPU / PyTorch fallback.  Gradients: a convolution whose input or weight requires grad runs epilogue-free through
_IndiceConvFunction (dX = the same kernel on the transposed table with W^T, dW = sstb200_spconv_backward_weight) and the containers
compose BatchNorm / activation / residual with torch modules, as the reference does.

Sub-manifold convolutions are always centred: spconv forces stride 1 / padding k//2 in the SubM index generation whatever the layer
was built with (vendored v1: include/spconv/spconv_ops.h:74-78; spconv 2.x: generate_subm_conv_inds takes no padding), so e.g.
VirtualVoxelMixer.conv_out (kernel 3, padding 0) is a centred 3x3x3 convolution."""
import ctypes as C
import math

import numpy as np
import torch
from torch import nn

from . import _lib as L
from .ops import build_norm_layer
from .registry import BACKBONES, MIDDLE_ENCODERS

L.SIGNATURES["sstb200_spconv_out_coors"] = (C.c_int, [L.vp, L.vp, C.c_int, C.c_int, L.P_i32, L.P_i32, L.P_i32, L.P_i32, L.P_i32, L.vp,
                                                     C.c_int, L.vp, L.P_i32])
L.SIGNATURES["sstb200_spconv_table"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, C.c_int, C.c_int, L.P_i32, L.P_i32, L.P_i32, L.P_i32,
                                                 L.P_i32, L.vp, L.vp, L.P_i32])
L.SIGNATURES["sstb200_spconv_backward_weight"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, C.c_int, C.c_int, L.vp, C.c_int, L.vp])
L.SIGNATURES["sstb200_spconv_forward"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, C.c_int, C.c_int, L.vp, L.vp, C.c_int, L.vp, L.vp, L.vp,
                                                   C.c_int, C.c_int, L.vp])
# device-count variants (sync-free engines, sst_b200/fsd_engine.py)
L.SIGNATURES["sstb200_spconv_out_coors_dev"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, C.c_int, L.P_i32, L.P_i32, L.P_i32, L.P_i32, L.P_i32,
                                                         L.vp, C.c_int, L.vp])
L.SIGNATURES["sstb200_spconv_table_dev"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, L.vp, C.c_int, L.vp, C.c_int, L.P_i32, L.P_i32, L.P_i32,
                                                     L.P_i32, L.P_i32, L.vp, L.vp])
L.SIGNATURES["sstb200_spconv_forward_dev"] = (C.c_int, [L.vp, L.vp, C.c_int, C.c_int, L.vp, C.c_int, L.vp, C.c_int, L.vp, L.vp, C.c_int,
                                                       L.vp, L.vp, L.vp, C.c_int, C.c_int, C.c_int, L.vp, C.c_int])
L.SIGNATURES["sstb200_spconv_decoder_merge"] = (C.c_int, [L.vp, L.vp, L.vp, C.c_int, C.c_int, C.c_int, L.vp, L.vp])

PREC = {"fp32": 0, "bf16": 1, "fp32_tc": 2}   # fp32_tc: fp32 tolerance on the tensor core (split-fp16 operands, 3 products per stage)


def split_h16(weight):
    """[KV, Cin, Cout] fp32 -> the 16-bit operand copy of the tensor-core paths, laid out [KV, Cout, Cin]; with residue=True the fp16
    residue  w - float(half(w))  follows the hi copy ([2 KV, Cout, Cin]) as SSTB200_PREC_FP32_TC expects."""
    w = weight.detach().permute(0, 2, 1).contiguous().float()
    hi = w.half()
    return hi, (w - hi.float()).half()
FUSE_EPILOGUE = True   # eval mode: fold BatchNorm1d / residual / ReLU into the convolution launch (False = conv launch + torch modules)


def _triple(v, ndim):
    v = list(v) if isinstance(v, (list, tuple)) else [v] * ndim
    assert len(v) == ndim
    return [1] * (3 - ndim) + [int(x) for x in v] if ndim < 3 else [int(x) for x in v]


def _i3(v):
    return L.arr(C.c_int32, [int(x) for x in v])


def get_conv_output_size(input_size, kernel_size, stride, padding, dilation):
    """mmdet3d/ops/spconv/ops.py:20-31"""
    return [(i + 2 * p - d * (k - 1) - 1) // s + 1 for i, k, s, p, d in zip(input_size, kernel_size, stride, padding, dilation)]


# ------------------------------------------------------------------------------------------------------------------------
# functional layer over the C ABI
# ------------------------------------------------------------------------------------------------------------------------
def _coors4(indices):
    """(b, [z,] y, x) int32 rows -> contiguous (b, z, y, x)."""
    assert indices.dim() == 2 and indices.shape[1] in (3, 4), "indices must be [N, 1 + ndim], ndim 2 or 3"
    ind = indices.int()
    if ind.shape[1] == 3:
        ind = torch.cat([ind[:, :1], torch.zeros_like(ind[:, :1]), ind[:, 1:]], 1)
    return ind.contiguous()


def conv_out_coors(indices, batch_size, in_shape, out_shape, ksize, stride, padding):
    """Active output coordinates of a strided sparse convolution, lexicographically sorted (b,z,y,x).  One host sync (row count)."""
    ind = _coors4(indices)
    if not ind.is_cuda:
        raise L.SSTB200Error("sst_b200 spconv needs CUDA tensors (no CPU fallback)")
    n = ind.shape[0]
    per_in = 1
    cells = int(batch_size)
    for k, s, o in zip(ksize, stride, out_shape):
        per_in *= (k + s - 1) // s
        cells *= o
    cap = max(1, min(n * per_in, cells))
    out = torch.empty((cap, 4), dtype=torch.int32, device=ind.device)
    num_dev = torch.empty((1,), dtype=torch.int32, device=ind.device)
    num_host = C.c_int32(0)
    c = L.ctx(ind.device)
    L.check(c, L.lib().sstb200_spconv_out_coors(c, ind.data_ptr(), n, int(batch_size), _i3(in_shape), _i3(out_shape), _i3(ksize),
                                                _i3(stride), _i3(padding), out.data_ptr(), cap, num_dev.data_ptr(), C.byref(num_host)))
    return out[:num_host.value]


def conv_table(in_indices, out_indices, batch_size, in_shape, out_shape, ksize, stride, padding, want_nbr=True, want_inv=False, check=True):
    """(nbr [n_out, KV], nbr_inv [n_in, KV]) int32 neighbour tables (None when not asked for).  check: read the status word back (one
    host sync) and raise on coordinates outside the grid; callers pass False for coordinate sets this package produced itself."""
    ci, co = _coors4(in_indices), _coors4(out_indices)
    if not ci.is_cuda:
        raise L.SSTB200Error("sst_b200 spconv needs CUDA tensors (no CPU fallback)")
    kv = int(np.prod(ksize))
    nbr = torch.empty((co.shape[0], kv), dtype=torch.int32, device=ci.device) if want_nbr else None
    inv = torch.empty((ci.shape[0], kv), dtype=torch.int32, device=ci.device) if want_inv else None
    status = C.c_int32(0)
    c = L.ctx(ci.device)
    L.check(c, L.lib().sstb200_spconv_table(c, ci.data_ptr(), ci.shape[0], co.data_ptr(), co.shape[0], int(batch_size), _i3(in_shape),
                                            _i3(out_shape), _i3(ksize), _i3(stride), _i3(padding), L.ptr(nbr), L.ptr(inv),
                                            C.byref(status) if check else None))
    return nbr, inv


def _indice_conv_launch(features, nbr, weight, weight_h16, scale, shift, residual, relu, precision):
    feats = features.float().contiguous()
    kv, cin, cout = weight.shape
    assert feats.shape[1] == cin and nbr.shape[1] == kv and nbr.dtype == torch.int32 and nbr.is_contiguous()
    weight = weight.detach().contiguous()
    n_out = nbr.shape[0]
    out = torch.empty((n_out, cout), dtype=torch.float32, device=feats.device)
    if residual is not None:
        residual = residual.float().contiguous()
        assert residual.shape == out.shape
    prec = PREC[precision]
    if prec != 0 and weight_h16 is None:
        hi, lo = split_h16(weight)
        weight_h16 = hi if prec == 1 else torch.cat([hi, lo], 0)
    c = L.ctx(feats.device)
    L.check(c, L.lib().sstb200_spconv_forward(c, feats.data_ptr(), cin, nbr.data_ptr(), n_out, kv, weight.data_ptr(), L.ptr(weight_h16), cout,
                                              L.ptr(scale), L.ptr(shift), L.ptr(residual), int(bool(relu)), prec, out.data_ptr()))
    return out


def indice_conv_backward_weight(features, nbr, grad_out, kv, cin, cout):
    """dW [KV, Cin, Cout] = sum over pairs of features[nbr[o,k]]^T grad_out[o]"""
    feats, g = features.float().contiguous(), grad_out.float().contiguous()
    dw = torch.empty((kv, cin, cout), dtype=torch.float32, device=feats.device)
    c = L.ctx(feats.device)
    L.check(c, L.lib().sstb200_spconv_backward_weight(c, feats.data_ptr(), cin, nbr.data_ptr(), nbr.shape[0], kv, g.data_ptr(), cout,
                                                      dw.data_ptr()))
    return dw


class _IndiceConvFunction(torch.autograd.Function):
    """autograd bridge of a convolution without epilogue (the reference: spconv's SparseConvFunction / SubMConvFunction /
    SparseInverseConvFunction, mmdet3d/ops/spconv/functional.py:20-98).  dX is the same kernel on the transposed table with W^T."""

    @staticmethod
    def forward(ctx, features, weight, nbr, transposed_table, precision):
        ctx.save_for_backward(features, weight, nbr)
        ctx.transposed_table, ctx.precision = transposed_table, precision
        return _indice_conv_launch(features, nbr, weight, None, None, None, None, False, precision)

    @staticmethod
    def backward(ctx, grad_out):
        features, weight, nbr = ctx.saved_tensors
        grad_out = grad_out.contiguous()
        dx = dw = None
        if ctx.needs_input_grad[0]:
            nbr_t = ctx.transposed_table()
            assert nbr_t.shape[0] == features.shape[0]
            dx = _indice_conv_launch(grad_out, nbr_t, weight.detach().transpose(1, 2).contiguous(), None, None, None, None, False, ctx.precision)
        if ctx.needs_input_grad[1]:
            dw = indice_conv_backward_weight(features, nbr, grad_out, *weight.shape)
        return dx, dw, None, None, None


def indice_conv(features, nbr, weight, weight_h16=None, scale=None, shift=None, residual=None, relu=False, precision="fp32",
                transposed_table=None):
    """out[o] = act((sum_k features[nbr[o,k]] @ weight[k]) * scale + shift + residual[o]); weight [KV, Cin, Cout] fp32.
    With gradients enabled the call must be epilogue-free and name its transposed table (a callable returning nbr_T [n_in, KV])."""
    if not features.is_cuda:
        raise L.SSTB200Error("sst_b200 spconv needs CUDA tensors (no CPU fallback)")
    if torch.is_grad_enabled() and (features.requires_grad or weight.requires_grad):
        if scale is not None or shift is not None or residual is not None or relu or transposed_table is None:
            raise NotImplementedError("gradients flow through epilogue-free sparse convolutions only (the modules compose BatchNorm / "
                                      "activation / residual with torch ops when a gradient is needed)")
        return _IndiceConvFunction.apply(features, weight, nbr, transposed_table, precision)
    return _indice_conv_launch(features, nbr, weight, weight_h16, scale, shift, residual, relu, precision)


def fold_bn(bn, conv_bias=None):
    """eval-mode BatchNorm1d (+ the bias of the convolution in front of it) -> (scale, shift) fp32 [C]; cached on the module until a
    parameter / buffer changes (34 convolutions x 6 tiny torch kernels per U-Net forward otherwise)"""
    ts = (bn.running_mean, bn.running_var, bn.weight, bn.bias, conv_bias)
    key = tuple((t._version, t.data_ptr()) for t in ts if t is not None)
    hit = getattr(bn, "_sstb200_fold", None)
    if hit is not None and hit[0] == key:
        return hit[1], hit[2]
    scale, shift = _fold_bn(bn)
    if conv_bias is not None:
        shift = (shift + conv_bias.detach().float() * scale).contiguous()
    bn._sstb200_fold = (key, scale, shift)
    return scale, shift


def _fold_bn(bn):
    var = bn.running_var.float()
    inv = torch.rsqrt(var + bn.eps)
    w = bn.weight.detach().float() if bn.weight is not None else torch.ones_like(var)
    b = bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(var)
    scale = w * inv
    shift = b - bn.running_mean.float() * scale
    return scale.contiguous(), shift.contiguous()


# ------------------------------------------------------------------------------------------------------------------------
# tensor + containers
# ------------------------------------------------------------------------------------------------------------------------
class SparseConvTensor:
    """features [N, C], indices [N, 1 + ndim] int32 (batch first), spatial_shape, batch_size (structure.py:22-69; replace_feature as
    in spconv 2.x, which sparse_unet.py:181-186 relies on)."""

    def __init__(self, features, indices, spatial_shape, batch_size, grid=None):
        self.features = features
        self.indices = indices.int() if indices.dtype != torch.int32 else indices
        self.spatial_shape = list(int(s) for s in spatial_shape)
        self.batch_size = int(batch_size)
        self.indice_dict = {}
        self.grid = grid

    @property
    def spatial_size(self):
        return int(np.prod(self.spatial_shape))

    def find_indice_pair(self, key):
        return None if key is None else self.indice_dict.get(key)

    def replace_feature(self, feature):
        t = SparseConvTensor(feature, self.indices, self.spatial_shape, self.batch_size, self.grid)
        t.indice_dict = self.indice_dict
        return t

    def dense(self, channels_first=True):
        shape = [self.batch_size] + list(self.spatial_shape) + [self.features.shape[1]]
        res = torch.zeros(shape, dtype=self.features.dtype, device=self.features.device)
        idx = self.indices.long()
        res[tuple(idx[:, i] for i in range(idx.shape[1]))] = self.features
        if not channels_first:
            return res
        nd = len(self.spatial_shape)
        return res.permute(0, nd + 1, *range(1, nd + 1)).contiguous()

    @property
    def sparity(self):
        return self.indices.shape[0] / self.spatial_size / self.batch_size


class IndiceData:
    """What spconv keeps per indice_key (conv.py:169-172: outids, indices, indice_pairs, indice_pair_num, spatial_shape) in the
    output-stationary form: nbr [n_out, KV]; the transposed table for the inverse conv is built on first use."""

    def __init__(self, out_indices, in_indices, nbr, batch_size, in_shape, out_shape, ksize, stride, padding):
        self.out_indices, self.in_indices, self.nbr = out_indices, in_indices, nbr
        self.batch_size, self.in_shape, self.out_shape = batch_size, in_shape, out_shape
        self.ksize, self.stride, self.padding = ksize, stride, padding
        self._inv = None

    def inverse_table(self):
        if self._inv is None:
            _, self._inv = conv_table(self.in_indices, self.out_indices, self.batch_size, self.in_shape, self.out_shape, self.ksize,
                                      self.stride, self.padding, want_nbr=False, want_inv=True, check=False)
        return self._inv


class SparseModule(nn.Module):
    """marker base class: SparseSequential hands these the SparseConvTensor itself (modules.py:45-48)"""


def _wants_grad(x, conv):
    return torch.is_grad_enabled() and (x.features.requires_grad or conv.weight.requires_grad)


def _is_relu(m):
    return isinstance(m, nn.ReLU)


class SparseSequential(SparseModule):
    """modules.py:51-137.  In eval mode a `SparseConvolution, BatchNorm1d[, ReLU]` run becomes one launch."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        if len(args) == 1 and isinstance(args[0], dict):
            for k, m in args[0].items():
                self.add_module(k, m)
        else:
            for i, m in enumerate(args):
                self.add_module(str(i), m)
        for k, m in kwargs.items():
            if k in self._modules:
                raise ValueError("name exists.")
            self.add_module(k, m)

    def __getitem__(self, idx):
        if not -len(self) <= idx < len(self):
            raise IndexError(f"index {idx} is out of range")
        return list(self._modules.values())[idx % len(self)]

    def __len__(self):
        return len(self._modules)

    def add(self, module, name=None):
        self.add_module(str(len(self._modules)) if name is None else name, module)

    def forward(self, input):
        mods = list(self._modules.values())
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, SparseConvolution):
                fuse = FUSE_EPILOGUE and not _wants_grad(input, m)
                bn = mods[i + 1] if (fuse and i + 1 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm1d)
                                     and not mods[i + 1].training) else None
                relu = bn is not None and i + 2 < len(mods) and _is_relu(mods[i + 2])
                if fuse and bn is None and i + 1 < len(mods) and _is_relu(mods[i + 1]):
                    input = m(input, relu=True)
                    i += 2
                    continue
                input = m(input, bn=bn, relu=relu)
                i += 1 + (bn is not None) + relu
            elif isinstance(m, SparseModule):
                input = m(input)
                i += 1
            else:
                if isinstance(input, SparseConvTensor):
                    if input.indices.shape[0] != 0:
                        input = input.replace_feature(m(input.features))
                else:
                    input = m(input)
                i += 1
        return input


class ToDense(SparseModule):
    def forward(self, x):
        return x.dense()


# ------------------------------------------------------------------------------------------------------------------------
# convolution layers
# ------------------------------------------------------------------------------------------------------------------------
class SparseConvolution(SparseModule):
    """conv.py:45-206.  precision: 'fp32' (FFMA, exact path), 'bf16' (tcgen05, 16-bit operands) or 'fp32_tc' (tcgen05 with split-fp16
    operands: fp32 tolerance at tensor-core speed; channels % 64) - module attribute, also settable for a whole model with
    set_spconv_precision()."""

    def __init__(self, ndim, in_channels, out_channels, kernel_size=3, stride=1, padding=0, dilation=1, groups=1, bias=True, subm=False,
                 output_padding=0, transposed=False, inverse=False, indice_key=None, fused_bn=False):
        super().__init__()
        assert groups == 1 and ndim in (2, 3)
        if transposed:
            raise NotImplementedError("SparseConvTranspose is not used by the reference's configs and is not built")
        as_list = lambda v: list(v) if isinstance(v, (list, tuple)) else [v] * ndim
        self.ndim = ndim
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding = as_list(kernel_size), as_list(stride), as_list(padding)
        self.dilation, self.output_padding = as_list(dilation), as_list(output_padding)
        assert all(d == 1 for d in self.dilation), "dilation > 1 is not used by the reference's configs and is not built"
        self.conv1x1 = int(np.prod(self.kernel_size)) == 1
        self.transposed, self.inverse, self.groups, self.subm = transposed, inverse, groups, subm
        self.indice_key = indice_key
        self.fused_bn = fused_bn
        self.precision = "fp32"
        self.weight = nn.Parameter(torch.empty(*self.kernel_size, in_channels, out_channels))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self._h16 = None
        self.reset_parameters()

    def reset_parameters(self):
        # conv.py:103-108: kaiming_uniform(a=sqrt(5)) with fan_in of the (D,H,W,in,out) layout
        fan_in = self.in_channels * int(np.prod(self.kernel_size))
        bound = math.sqrt(6.0 / ((1 + 5.0) * fan_in))
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)
            if self.bias is not None:
                b = 1 / math.sqrt(fan_in)
                self.bias.uniform_(-b, b)

    def _weight_h16(self):
        key = (self.weight._version, self.weight.data_ptr(), self.precision)
        if self._h16 is None or self._h16[0] != key:
            kv = int(np.prod(self.kernel_size))
            hi, lo = split_h16(self.weight.reshape(kv, self.in_channels, self.out_channels))
            self._h16 = (key, hi if self.precision == "bf16" else torch.cat([hi, lo], 0))
        return self._h16[1]

    def _geometry(self, spatial_shape):
        nd = self.ndim
        ks, st, pd = _triple(self.kernel_size, nd), _triple(self.stride, nd), _triple(self.padding, nd)
        in_shape = _triple(spatial_shape, nd)
        if self.subm:   # spconv_ops.h:74-78: stride 1, padding k//2, whatever the layer says
            return in_shape, in_shape, ks, [1, 1, 1], [k // 2 for k in ks]
        out_shape = get_conv_output_size(in_shape, ks, st, pd, [1, 1, 1])
        return in_shape, out_shape, ks, st, pd

    def forward(self, input, bn=None, relu=False, residual=None):
        assert isinstance(input, SparseConvTensor)
        feats = input.features
        indices = input.indices
        kv = int(np.prod(self.kernel_size))
        w = self.weight.reshape(kv, self.in_channels, self.out_channels)
        grad = _wants_grad(input, self)
        if grad:
            assert bn is None and not relu and residual is None, "fused epilogues carry no gradient (SparseSequential composes them)"
            scale = shift = None
        elif bn is not None:
            scale, shift = fold_bn(bn, self.bias)
        else:
            scale, shift = None, (self.bias.detach().float().contiguous() if self.bias is not None else None)
        h16 = self._weight_h16() if self.precision != "fp32" and not grad else None
        if self.conv1x1:
            nbr = torch.arange(feats.shape[0], dtype=torch.int32, device=feats.device).view(-1, 1)
            out = indice_conv(feats, nbr, w, h16, scale, shift, residual, relu, self.precision, transposed_table=lambda: nbr)
            if grad and self.bias is not None:
                out = out + self.bias
            t = SparseConvTensor(out, indices, input.spatial_shape, input.batch_size, input.grid)
            t.indice_dict = input.indice_dict
            return t
        datas = input.find_indice_pair(self.indice_key)
        if self.inverse:
            assert datas is not None and self.indice_key is not None, "inverse conv needs the indice pairs of its couple conv"
            assert datas.nbr.shape[1] == kv, "inverse conv must have same kernel size as its couple conv"
            nbr, out_indices = datas.inverse_table(), datas.in_indices
            out_shape = datas.in_shape[3 - self.ndim:]
            transposed = lambda d=datas: d.nbr
        else:
            if self.indice_key is not None and datas is not None:
                assert datas.nbr.shape[1] == kv
            else:
                in_shape, oshape, ks, st, pd = self._geometry(input.spatial_shape)
                # conv_out_coors validates the input coordinates; rows this package produced (output of an earlier conv: the tensor
                # already carries tables) need no second status round trip
                derived = bool(input.indice_dict)
                out_ids = indices if self.subm else conv_out_coors(indices, input.batch_size, in_shape, oshape, ks, st, pd)
                nbr_, _ = conv_table(indices, out_ids, input.batch_size, in_shape, oshape, ks, st, pd, check=self.subm and not derived)
                if not self.subm and self.ndim == 2:
                    out_ids = out_ids[:, [0, 2, 3]].contiguous()
                datas = IndiceData(out_ids, indices, nbr_, input.batch_size, in_shape, oshape, ks, st, pd)
                if self.indice_key is not None:
                    input.indice_dict[self.indice_key] = datas
            nbr, out_indices = datas.nbr, datas.out_indices
            out_shape = datas.out_shape[3 - self.ndim:]
            transposed = datas.inverse_table
        out = indice_conv(feats, nbr, w, h16, scale, shift, residual, relu, self.precision, transposed_table=transposed)
        if grad and self.bias is not None:
            out = out + self.bias
        t = SparseConvTensor(out, out_indices, out_shape, input.batch_size, input.grid)
        t.indice_dict = input.indice_dict
        return t


def _conv_class(name, ndim, **fixed):
    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True, indice_key=None):
        kw = dict(stride=stride, padding=padding, dilation=dilation, groups=groups, bias=bias, indice_key=indice_key)
        if fixed.get("inverse"):   # SparseInverseConv*: (in, out, kernel_size, indice_key, bias=True)  conv.py:386-446
            kw = dict(bias=bias, indice_key=indice_key)
        SparseConvolution.__init__(self, ndim, in_channels, out_channels, kernel_size, **kw, **fixed)
    return type(name, (SparseConvolution,), {"__init__": __init__, "__doc__": f"mmdet3d/ops/spconv/conv.py {name}"})


SparseConv2d = _conv_class("SparseConv2d", 2)
SparseConv3d = _conv_class("SparseConv3d", 3)
SubMConv2d = _conv_class("SubMConv2d", 2, subm=True)
SubMConv3d = _conv_class("SubMConv3d", 3, subm=True)
SparseInverseConv2d = _conv_class("SparseInverseConv2d", 2, inverse=True)
SparseInverseConv3d = _conv_class("SparseInverseConv3d", 3, inverse=True)
CONV_LAYERS = {c.__name__: c for c in (SparseConv2d, SparseConv3d, SubMConv2d, SubMConv3d, SparseInverseConv2d, SparseInverseConv3d)}


def build_conv_layer(cfg, *args, **kwargs):
    """mmcv.cnn.build_conv_layer for the sparse layer types"""
    cfg = dict(cfg)
    t = cfg.pop("type")
    if t not in CONV_LAYERS:
        raise KeyError(f"conv type {t} is not a sparse convolution of this package")
    return CONV_LAYERS[t](*args, **kwargs, **cfg)


def set_spconv_precision(module, precision):
    assert precision in PREC
    for m in module.modules():
        if isinstance(m, SparseConvolution):
            m.precision = precision
    return module


_ACTS = {"relu": lambda: nn.ReLU(inplace=True), "gelu": nn.GELU, "silu": lambda: nn.SiLU(inplace=True)}


def make_sparse_convmodule(in_channels, out_channels, kernel_size, indice_key, stride=1, padding=0, conv_type="SubMConv3d",
                           act_type="relu", norm_cfg=None, order=("conv", "norm", "act")):
    """mmdet3d/ops/sparse_block.py:216-289"""
    assert isinstance(order, tuple) and len(order) <= 3 and set(order) <= {"conv", "norm", "act"}
    conv_cfg = dict(type=conv_type, indice_key=indice_key)
    layers = []
    for layer in order:
        if layer == "conv":
            if conv_type.startswith("SparseInverseConv"):
                layers.append(build_conv_layer(conv_cfg, in_channels, out_channels, kernel_size, bias=False))
            else:
                layers.append(build_conv_layer(conv_cfg, in_channels, out_channels, kernel_size, stride=stride, padding=padding, bias=False))
        elif layer == "norm":
            layers.append(build_norm_layer(norm_cfg, out_channels)[1])
        else:
            if act_type.lower() not in _ACTS:
                raise NotImplementedError
            layers.append(_ACTS[act_type.lower()]())
    return SparseSequential(*layers)


class SparseBasicBlock(SparseModule):
    """sparse_block.py:81-143 over mmdet's BasicBlock (conv1, bn1, conv2, bn2, relu; state-dict keys conv1.weight, bn1.*, ...).
    Eval mode with ReLU: two launches (conv1+bn1+relu, conv2+bn2+identity+relu)."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None, conv_cfg=None, norm_cfg=None, act_type="relu"):
        super().__init__()
        assert stride == 1 and downsample is None, "the reference only builds stride-1 blocks without a downsample branch"
        self.bn1 = build_norm_layer(norm_cfg, planes)[1]
        self.bn2 = build_norm_layer(norm_cfg, planes)[1]
        self.conv1 = build_conv_layer(conv_cfg, inplanes, planes, 3, stride=stride, padding=1, dilation=1, bias=False)
        self.conv2 = build_conv_layer(conv_cfg, planes, planes, 3, padding=1, bias=False)
        self.relu = _ACTS[act_type.lower()]()
        self.downsample = downsample

    @property
    def norm1(self):
        return self.bn1

    @property
    def norm2(self):
        return self.bn2

    def forward(self, x):
        identity = x.features
        assert x.features.dim() == 2, f"x.features.dim()={x.features.dim()}"
        fused = (FUSE_EPILOGUE and _is_relu(self.relu) and not self.bn1.training and not self.bn2.training
                 and not _wants_grad(x, self.conv1) and not _wants_grad(x, self.conv2))
        if fused:
            out = self.conv1(x, bn=self.bn1, relu=True)
            return self.conv2(out, bn=self.bn2, relu=True, residual=identity)
        out = self.conv1(x)
        out = out.replace_feature(self.relu(self.bn1(out.features)))
        out = self.conv2(out)
        out = out.replace_feature(self.bn2(out.features))
        return out.replace_feature(self.relu(out.features + identity))


# ------------------------------------------------------------------------------------------------------------------------
# the U-Nets
# ------------------------------------------------------------------------------------------------------------------------
@MIDDLE_ENCODERS.register_module()
class SparseUNet(nn.Module):
    """mmdet3d/models/middle_encoders/sparse_unet.py:15-321 (PartA2's U-Net; base class of the two FSD backbones)."""

    def __init__(self, in_channels, sparse_shape, order=("conv", "norm", "act"), norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01),
                 base_channels=16, output_channels=128, encoder_channels=((16,), (32, 32, 32), (64, 64, 64), (64, 64, 64)),
                 encoder_paddings=((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1)),
                 decoder_channels=((64, 64, 64), (64, 64, 32), (32, 32, 16), (16, 16, 16)),
                 decoder_paddings=((1, 0), (1, 0), (0, 0), (0, 1)), ndim=3, act_type="relu", init_cfg=None):
        super().__init__()
        self.sparse_shape, self.in_channels, self.order = sparse_shape, in_channels, tuple(order)
        self.base_channels, self.output_channels = base_channels, output_channels
        self.encoder_channels, self.encoder_paddings = encoder_channels, encoder_paddings
        self.decoder_channels, self.decoder_paddings = decoder_channels, decoder_paddings
        self.stage_num = len(encoder_channels)
        self.ndim, self.is_3d, self.act_type = ndim, ndim == 3, act_type
        self.fp16_enabled = False
        assert len(self.order) == 3 and set(self.order) == {"conv", "norm", "act"}
        nd = ndim
        pre_act = self.order[0] != "conv"
        self.conv_input = make_sparse_convmodule(in_channels, base_channels, 3, norm_cfg=norm_cfg, padding=1, indice_key="subm1",
                                                 conv_type=f"SubMConv{nd}d", act_type=act_type,
                                                 **(dict(order=("conv",)) if pre_act else {}))
        enc_out = self.make_encoder_layers(make_sparse_convmodule, norm_cfg, base_channels)
        self.make_decoder_layers(make_sparse_convmodule, norm_cfg, enc_out)
        self.conv_out = make_sparse_convmodule(enc_out, output_channels, kernel_size=(3, 1, 1) if self.is_3d else (1,) * nd,
                                               stride=(2, 1, 1) if self.is_3d else (1,) * nd, norm_cfg=norm_cfg, padding=0,
                                               indice_key="spconv_down2", conv_type=f"SparseConv{nd}d", act_type=act_type)

    def make_encoder_layers(self, make_block, norm_cfg, in_channels):
        self.encoder_layers = SparseSequential()
        out_channels = in_channels
        for i, blocks in enumerate(self.encoder_channels):
            stage = []
            for j, out_channels in enumerate(tuple(blocks)):
                padding = tuple(self.encoder_paddings[i])[j]
                down = i != 0 and j == 0   # every stage but the first opens with a stride-2 SparseConv
                stage.append(make_block(in_channels, out_channels, 3, norm_cfg=norm_cfg, padding=padding, act_type=self.act_type,
                                        **(dict(stride=2, indice_key=f"spconv{i + 1}", conv_type=f"SparseConv{self.ndim}d") if down else
                                           dict(indice_key=f"subm{i + 1}", conv_type=f"SubMConv{self.ndim}d"))))
                in_channels = out_channels
            self.encoder_layers.add_module(f"encoder_layer{i + 1}", SparseSequential(*stage))
        return out_channels

    def make_decoder_layers(self, make_block, norm_cfg, in_channels):
        n = len(self.decoder_channels)
        for i, ch in enumerate(self.decoder_channels):
            lvl = n - i
            pads = self.decoder_paddings[i]
            setattr(self, f"lateral_layer{lvl}", SparseBasicBlock(in_channels, ch[0], norm_cfg=norm_cfg, act_type=self.act_type,
                                                                   conv_cfg=dict(type=f"SubMConv{self.ndim}d", indice_key=f"subm{lvl}")))
            setattr(self, f"merge_layer{lvl}", make_block(in_channels * 2, ch[1], 3, norm_cfg=norm_cfg, padding=pads[0],
                                                           indice_key=f"subm{lvl}", conv_type=f"SubMConv{self.ndim}d",
                                                           act_type=self.act_type))
            if lvl != 1:
                up = make_block(in_channels, ch[2], 3, norm_cfg=norm_cfg, indice_key=f"spconv{lvl}",
                                conv_type=f"SparseInverseConv{self.ndim}d", act_type=self.act_type)
            else:   # the last block upsamples with a submanifold conv
                up = make_block(in_channels, ch[2], 3, norm_cfg=norm_cfg, padding=pads[1], indice_key="subm1",
                                conv_type=f"SubMConv{self.ndim}d", act_type=self.act_type)
            setattr(self, f"upsample_layer{lvl}", up)
            in_channels = ch[2]

    @staticmethod
    def reduce_channel(x, out_channels):
        feats = x.features
        n, cin = feats.shape
        assert cin % out_channels == 0 and cin >= out_channels
        return x.replace_feature(feats.view(n, out_channels, -1).sum(dim=2))

    def decoder_layer_forward(self, x_lateral, x_bottom, lateral_layer, merge_layer, upsample_layer):
        x = lateral_layer(x_lateral)
        x = x.replace_feature(torch.cat((x_bottom.features, x.features), dim=1))
        x_merge = merge_layer(x)
        x = self.reduce_channel(x, x_merge.features.shape[1])
        x = x.replace_feature(x_merge.features + x.features)
        return upsample_layer(x)

    def _encode(self, voxel_features, coors, batch_size):
        x = self.conv_input(SparseConvTensor(voxel_features, coors.int(), self.sparse_shape, batch_size))
        feats = []
        for layer in self.encoder_layers:
            x = layer(x)
            feats.append(x)
        return feats

    def _decode(self, enc, collect=None):
        x = enc[-1]
        for i in range(self.stage_num, 0, -1):
            x = self.decoder_layer_forward(enc[i - 1], x, getattr(self, f"lateral_layer{i}"), getattr(self, f"merge_layer{i}"),
                                           getattr(self, f"upsample_layer{i}"))
            if collect is not None:
                collect.append(x)
        return x

    def forward(self, voxel_features, coors, batch_size):
        assert self.is_3d, "This forward function only supports 3D spconv"
        enc = self._encode(voxel_features, coors, batch_size)
        spatial = self.conv_out(enc[-1]).dense()
        N, Cc, D, H, W = spatial.shape
        x = self._decode(enc)
        return dict(spatial_features=spatial.view(N, Cc * D, H, W), seg_features=x.features)


def _select_coors(self, coors):
    if self.ndim == 2:
        assert (coors[:, 1] == 0).all()
        coors = coors[:, [0, 2, 3]]
    if self.keep_coors_dims is not None:
        coors = coors[:, self.keep_coors_dims]
    return coors.int()


@BACKBONES.register_module()
class SimpleSparseUNet(SparseUNet):
    """sparse_unet.py:323-413: the U-Net without the dense head branch; consumes / returns the voxel_info dict like SSTv2."""

    def __init__(self, in_channels, sparse_shape, order=("conv", "norm", "act"), norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01),
                 base_channels=16, output_channels=128, ndim=3, encoder_channels=((16,), (32, 32, 32), (64, 64, 64), (64, 64, 64)),
                 encoder_paddings=((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1)),
                 decoder_channels=((64, 64, 64), (64, 64, 32), (32, 32, 16), (16, 16, 16)),
                 decoder_paddings=((1, 0), (1, 0), (0, 0), (0, 1)), keep_coors_dims=None, act_type="relu",
                 return_multiscale_features=False, init_cfg=None):
        super().__init__(in_channels=in_channels, sparse_shape=sparse_shape, order=order, norm_cfg=norm_cfg, base_channels=base_channels,
                         output_channels=output_channels, encoder_channels=encoder_channels, encoder_paddings=encoder_paddings,
                         decoder_channels=decoder_channels, decoder_paddings=decoder_paddings, ndim=ndim, act_type=act_type,
                         init_cfg=init_cfg)
        self.conv_out = None
        self.keep_coors_dims = keep_coors_dims
        self.return_multiscale_features = return_multiscale_features

    def forward(self, voxel_info):
        coors = _select_coors(self, voxel_info["voxel_coors"])
        batch_size = int(coors[:, 0].max().item()) + 1
        enc = self._encode(voxel_info["voxel_feats"], coors, batch_size)
        decode_features = [] if self.return_multiscale_features else None
        x = self._decode(enc, decode_features)
        return [dict(voxel_feats=x.features, voxel_coors=x.indices, sparse_shape=x.spatial_shape, batch_size=x.batch_size,
                     decoder_features=decode_features or [])]


@BACKBONES.register_module()
class VirtualVoxelMixer(SparseUNet):
    """sparse_unet.py:416-505 (FSDv2's mixer over real + virtual voxels)."""

    def __init__(self, in_channels, sparse_shape, order=("conv", "norm", "act"), norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01),
                 base_channels=16, output_channels=128, ndim=3, encoder_channels=((16,), (32, 32, 32), (64, 64, 64), (64, 64, 64)),
                 encoder_paddings=((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1)),
                 decoder_channels=((64, 64, 64), (64, 64, 32), (32, 32, 16), (16, 16, 16)),
                 decoder_paddings=((1, 0), (1, 0), (0, 0), (0, 1)), keep_coors_dims=None, act_type="relu", init_cfg=None):
        super().__init__(in_channels=in_channels, sparse_shape=sparse_shape, order=order, norm_cfg=norm_cfg, base_channels=base_channels,
                         output_channels=output_channels, encoder_channels=encoder_channels, encoder_paddings=encoder_paddings,
                         decoder_channels=decoder_channels, decoder_paddings=decoder_paddings, ndim=ndim, act_type=act_type,
                         init_cfg=init_cfg)
        self.keep_coors_dims = keep_coors_dims
        self.conv_out = make_sparse_convmodule(decoder_channels[-1][-1], self.output_channels, kernel_size=3, stride=1, norm_cfg=norm_cfg,
                                               padding=0, indice_key="out_conv", conv_type=f"SubMConv{self.ndim}d", act_type=act_type)

    def forward(self, voxel_features, coors, batch_size):
        enc = self._encode(voxel_features, _select_coors(self, coors), batch_size)
        x = self.conv_out(self._decode(enc))
        return x.features, x.indices, x.spatial_shape
