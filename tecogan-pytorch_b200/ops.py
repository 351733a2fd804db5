"""Torch-tensor front end of the C ABI (include/tecogan_b200.h).

PyTorch is plumbing here: it owns device memory and the CUDA stream; every operation below is
one call into libtecogan_b200.so on ``torch.cuda.current_stream()``.  No op has a torch/CPU
fallback -- a tensor that is not on a CUDA device is an error.
"""
import ctypes
import os

import torch

from . import lib as L


LAUNCH_COUNT = 0   # kernels enqueued through the C ABI by this process (each call = 1 launch)


def _stream():
    global LAUNCH_COUNT
    LAUNCH_COUNT += 1
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _req(t, dtype, name, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise L.TecoganB200Error(f'{name}: expected a CUDA tensor (no CPU fallback exists)')
    if t.dtype != dtype:
        raise L.TecoganB200Error(f'{name}: expected dtype {dtype}, got {t.dtype}')
    if ndim is not None and t.dim() != ndim:
        raise L.TecoganB200Error(f'{name}: expected {ndim} dims, got {tuple(t.shape)}')
    if not t.is_contiguous():
        raise L.TecoganB200Error(f'{name}: tensor must be contiguous')
    return t


def sm_count():
    out = ctypes.c_int(0)
    L.check(L.load().tg_device_sm_count(ctypes.byref(out)), 'tg_device_sm_count')
    return out.value


def pad64(c):
    return (c + 63) // 64 * 64


# ---------------------------------------------------------------------------- conv layers
class PackedConv:
    """One 3x3 conv / stride-2 transposed conv of the path with device-packed fp16 weights.

    weight: nn.Conv2d layout [cout,cin,3,3] or nn.ConvTranspose2d layout [cin,cout,3,3] (fp32).
    Stored channel counts are padded to multiples of 64 (cin) and to 64/128/256 or 16 (cout).
    """

    def __init__(self, weight, bias, kind=L.CONV_3X3, act=L.ACT_NONE, epilogue=L.EPI_NHWC_F16):
        self.kind, self.act, self.epilogue = kind, act, epilogue
        if kind == L.CONV_3X3:
            self.cout_real, self.cin_real = weight.shape[0], weight.shape[1]
        else:
            self.cin_real, self.cout_real = weight.shape[0], weight.shape[1]
        self.cin = pad64(self.cin_real)
        self.tapn = epilogue != L.EPI_NHWC_F16      # thin NCHW heads: tap-major N packing
        self.cout = pad64(self.cout_real) if not self.tapn else 48
        self.packed = None
        self.bias = None
        self._ver = None
        self.refresh(weight, bias)

    def refresh(self, weight, bias, force=False):
        """(Re)pack when the parameters changed (optimizer step / load_state_dict).  Change detection
        is the tensors' version counters + storage pointers; writes through ``param.data`` do not
        bump the counter -- call with force=True (FRNet.refresh_packed_weights(force=True)) after such
        an update."""
        ver = (weight._version, bias._version, weight.data_ptr(), bias.data_ptr())
        if ver == self._ver and not force:
            return
        lib = L.load()
        w = _req(weight.detach(), torch.float32, 'weight', 4)
        nbytes = (lib.tg_packed_weight_bytes_tapn(self.cin) if self.tapn
                  else lib.tg_packed_weight_bytes(self.cin, self.cout))
        if self.packed is None:
            self.packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
            self.bias = torch.zeros(self.cout, dtype=torch.float32, device=w.device)
        if self.tapn:
            rc = lib.tg_pack_conv3x3_weights_tapn(_ptr(w), self.cout_real, self.cin_real, _ptr(self.packed),
                                                  self.cin, _stream())
        elif self.kind == L.CONV_3X3:
            rc = lib.tg_pack_conv3x3_weights(_ptr(w), self.cout_real, self.cin_real, _ptr(self.packed),
                                             self.cout, self.cin, _stream())
        else:
            rc = lib.tg_pack_convT3x3s2_weights(_ptr(w), self.cin_real, self.cout_real,
                                                _ptr(self.packed), self.cout, self.cin, _stream())
        L.check(rc, 'tg_pack_weights')
        self.bias[:self.cout_real].copy_(bias.detach())
        self._ver = ver

    def out_shape(self, n, h, w):
        if self.epilogue == L.EPI_NHWC_F16:
            if self.kind == L.CONVT_3X3_S2:
                return (n, 2 * h, 2 * w, self.cout), torch.float16
            return (n, h, w, self.cout), torch.float16
        return (n, self.cout_real, h, w), torch.float32

    def __call__(self, x, y=None, residual=None, impl=None, a_mode=None, max_ctas=0, pool=False):
        """x NHWC fp16 [n,h,w,cin] -> y (allocated when None).  pool=True: nn.MaxPool2d(2,2) folded into the
        epilogue, y = [n,h//2,w//2,cout] (conv3x3 layers with the NHWC epilogue, tcgen05 only)."""
        _req(x, torch.float16, 'conv input', 4)
        n, h, w, cin = x.shape
        if cin != self.cin:
            raise L.TecoganB200Error(f'conv input has {cin} channels, layer expects {self.cin}')
        shape, dtype = self.out_shape(n, h, w)
        if pool:
            if self.epilogue != L.EPI_NHWC_F16 or self.kind != L.CONV_3X3 or residual is not None:
                raise L.TecoganB200Error('pooled epilogue: conv3x3 with the NHWC epilogue and no residual only')
            shape = (n, h // 2, w // 2, self.cout)
        if y is None:
            y = torch.empty(shape, dtype=dtype, device=x.device)
        else:
            _req(y, dtype, 'conv output')
            if tuple(y.shape) != shape:
                raise L.TecoganB200Error(f'conv output shape {tuple(y.shape)} != {shape}')
        if residual is not None:
            _req(residual, torch.float16, 'residual', 4)
            if tuple(residual.shape) != (n, h, w, self.cout):
                raise L.TecoganB200Error('residual shape mismatch')
        d = L.ConvDesc()
        d.x, d.weights, d.bias = x.data_ptr(), self.packed.data_ptr(), self.bias.data_ptr()
        d.residual = residual.data_ptr() if residual is not None else None
        d.y = y.data_ptr()
        d.n, d.h, d.w, d.cin, d.cout, d.cout_real = n, h, w, self.cin, self.cout, self.cout_real
        d.kind, d.act, d.epilogue = self.kind, self.act, (L.EPI_NHWC_F16_POOL2 if pool else self.epilogue)
        d.a_mode = default_a_mode() if a_mode is None else a_mode
        d.max_ctas = max_ctas
        d.cin_real = self.cin_real
        impl = impl or default_conv_impl()
        lib = L.load()
        if impl == 'tcgen05':
            L.check(lib.tg_conv_tcgen05(ctypes.byref(d), _stream()), 'tg_conv_tcgen05')
        elif impl == 'simt':
            L.check(lib.tg_conv_simt(ctypes.byref(d), _stream()), 'tg_conv_simt')
        else:
            raise L.TecoganB200Error(f'unknown conv impl {impl!r}')
        return y


class ConvChain:
    """A chain of 64->64 3x3 convs in ONE persistent launch (tg_conv_chain_tcgen05).

    specs: list of (PackedConv, src, dst, res) where src/dst/res index into `buffers` (res may be
    None).  buffers[0] is the chain input (never written)."""

    def __init__(self, specs):
        if not 1 <= len(specs) <= L.CHAIN_MAX_LAYERS:
            raise L.TecoganB200Error(f'conv chain: {len(specs)} layers (1..{L.CHAIN_MAX_LAYERS})')
        for pc, src, dst, res in specs:
            if pc.kind != L.CONV_3X3 or pc.epilogue != L.EPI_NHWC_F16 or pc.cin != 64 or pc.cout != 64:
                raise L.TecoganB200Error('conv chain: every layer must be a 64->64 3x3 conv (NHWC fp16)')
            if src == dst or dst == 0:
                raise L.TecoganB200Error('conv chain: a layer may not write its own input or the chain input')
        self.specs = list(specs)
        self._ws = {}

    @staticmethod
    def supported(pcs):
        return all(pc.kind == L.CONV_3X3 and pc.epilogue == L.EPI_NHWC_F16 and pc.cin == 64 and pc.cout == 64
                   for pc in pcs) and 1 <= len(pcs) <= L.CHAIN_MAX_LAYERS

    def workspace(self, n, h, w, device):
        key = (n, h, w, str(device))
        ws = self._ws.get(key)
        if ws is None:
            nbytes = L.load().tg_conv_chain_workspace_bytes(n, h, w)
            ws = self._ws[key] = torch.zeros(nbytes, dtype=torch.uint8, device=device)   # zeroed ONCE
        return ws

    def __call__(self, buffers, max_ctas=0):
        x = buffers[0]
        _req(x, torch.float16, 'chain input', 4)
        n, h, w, c = x.shape
        for t in buffers:
            _req(t, torch.float16, 'chain buffer', 4)
            if tuple(t.shape) != (n, h, w, 64):
                raise L.TecoganB200Error(f'conv chain: buffer shape {tuple(t.shape)} != {(n, h, w, 64)}')
        arr = (L.ChainLayer * len(self.specs))()
        for i, (pc, src, dst, res) in enumerate(self.specs):
            arr[i].x, arr[i].weights, arr[i].bias = buffers[src].data_ptr(), pc.packed.data_ptr(), pc.bias.data_ptr()
            arr[i].residual = buffers[res].data_ptr() if res is not None else None
            arr[i].y, arr[i].act, arr[i].reserved = buffers[dst].data_ptr(), pc.act, 0
        ws = self.workspace(n, h, w, x.device)
        L.check(L.load().tg_conv_chain_tcgen05(arr, len(self.specs), n, h, w, _ptr(ws), max_ctas, _stream()),
                'tg_conv_chain_tcgen05')
        return buffers[self.specs[-1][2]]


def fused_tail(up, outc, x, lr_curr, lr_scale, up_mode, y=None, y_u8=None, max_ctas=0, accumulate=False):
    """SRNet tail in one launch (tg_convT_convout_tcgen05): y = conv_out(relu(convT(x))) + upsample_func(lr_curr)
    [, y_u8 = float32_to_uint8(y) as NHWC].  `up` / `outc` are the PackedConv objects of the last transposed
    conv and of conv_out (their packed weights are used as they are)."""
    _req(x, torch.float16, 'tail input', 4)
    n, h, w, c = x.shape
    if (up.kind != L.CONVT_3X3_S2 or up.cin != 64 or up.cout != 64 or c != 64 or not outc.tapn or outc.cin != 64
            or outc.cout_real > 3):
        raise L.TecoganB200Error('fused tail: needs a 64->64 transposed conv and a 64->(<=3) conv_out')
    co = outc.cout_real
    if y is None:
        y = torch.empty((n, co, 2 * h, 2 * w), dtype=torch.float32, device=x.device)
    _req(y, torch.float32, 'tail output', 4)
    if tuple(y.shape) != (n, co, 2 * h, 2 * w):
        raise L.TecoganB200Error(f'fused tail: output shape {tuple(y.shape)}')
    d = L.TailDesc()
    d.x, d.w_up, d.b_up = x.data_ptr(), up.packed.data_ptr(), up.bias.data_ptr()
    d.w_out, d.b_out, d.y = outc.packed.data_ptr(), outc.bias.data_ptr(), y.data_ptr()
    if lr_curr is not None:
        _req(lr_curr, torch.float32, 'lr_curr', 4)
        if tuple(lr_curr.shape) != (n, co, 2 * h // lr_scale, 2 * w // lr_scale):
            raise L.TecoganB200Error(f'fused tail: lr_curr shape {tuple(lr_curr.shape)}')
        d.lr = lr_curr.data_ptr()
    if y_u8 is not None:
        _req(y_u8, torch.uint8, 'uint8 output', 4)
        if tuple(y_u8.shape) != (n, 2 * h, 2 * w, co):
            raise L.TecoganB200Error(f'fused tail: uint8 output shape {tuple(y_u8.shape)}')
        d.y_u8 = y_u8.data_ptr()
    d.n, d.h, d.w, d.cout_real, d.lr_scale, d.up_mode, d.max_ctas, d.reserved = n, h, w, co, lr_scale, up_mode, max_ctas, 0
    d.accumulate = 1 if accumulate else 0
    L.check(L.load().tg_convT_convout_tcgen05(ctypes.byref(d), _stream()), 'tg_convT_convout_tcgen05')
    return y


def tail_mode():
    """TECOGAN_B200_TAIL: '0' = last transposed conv, conv_out, residual upsample and uint8 as four launches;
    'acc' = tg_convT_convout_tcgen05 accumulating onto a pre-written residual; 'fused' = residual and uint8
    evaluated inside the tail kernel.  Default 'acc': measured 0.786 ms per step against 0.849 ('0') and 0.897
    ('fused': the in-kernel gathers and 2-byte uint8 stores sit on the epilogue's critical path) --
    profiles/bench_r2f_tail_*.json."""
    v = os.environ.get('TECOGAN_B200_TAIL', 'acc')
    return {'0': None, '': None, '1': 'fused', 'fused': 'fused', '2': 'acc', 'acc': 'acc'}[v]


def pool_fused():
    """TECOGAN_B200_POOL=0 runs FNet's three max-pools as their own kernels instead of in the epilogue of the
    conv that feeds them (A/B measurements; bit-identical output)."""
    return os.environ.get('TECOGAN_B200_POOL', '1') != '0'


def chain_enabled():
    """TECOGAN_B200_CHAIN=0 runs SRNet's conv_in + residual blocks as 21 launches of
    tg_conv_tcgen05 instead of one tg_conv_chain_tcgen05 launch (A/B measurements)."""
    return os.environ.get('TECOGAN_B200_CHAIN', '1') != '0'


def default_conv_impl():
    """'tcgen05' (the product path) unless TECOGAN_B200_CONV=simt selects the CUDA-core
    cross-check kernel (bring-up / debugging only)."""
    return os.environ.get('TECOGAN_B200_CONV', 'tcgen05')


def default_a_mode():
    return {'auto': L.AMODE_AUTO, 'halo': L.AMODE_HALO, 'tap': L.AMODE_TAP}[
        os.environ.get('TECOGAN_B200_AMODE', 'auto')]


# ---------------------------------------------------------------------------- fused warp
def warp_s2d_concat_hrflow(hr_prev, hr_flow, lr_curr, scale, out=None, cpad=64):
    _req(hr_prev, torch.float32, 'hr_prev', 4)
    _req(hr_flow, torch.float32, 'hr_flow', 4)
    _req(lr_curr, torch.float32, 'lr_curr', 4)
    n, c, h, w = lr_curr.shape
    if tuple(hr_prev.shape) != (n, c, scale * h, scale * w) or tuple(hr_flow.shape) != (n, 2, scale * h, scale * w):
        raise L.TecoganB200Error('warp_s2d_concat: shape mismatch')
    if out is None:
        out = torch.empty((n, h, w, cpad), dtype=torch.float16, device=lr_curr.device)
    L.check(L.load().tg_warp_s2d_concat_hrflow(_ptr(hr_prev), _ptr(hr_flow), _ptr(lr_curr), _ptr(out),
                                               n, c, h, w, scale, cpad, _stream()),
            'tg_warp_s2d_concat_hrflow')
    return out


def warp_s2d_concat_lrflow(hr_prev, lr_flow, lr_curr, scale, up_mode, out=None, cpad=64):
    _req(hr_prev, torch.float32, 'hr_prev', 4)
    _req(lr_flow, torch.float32, 'lr_flow', 4)
    _req(lr_curr, torch.float32, 'lr_curr', 4)
    n, c, h, w = lr_curr.shape
    h8, w8 = lr_flow.shape[2], lr_flow.shape[3]
    if tuple(hr_prev.shape) != (n, c, scale * h, scale * w) or lr_flow.shape[0] != n or lr_flow.shape[1] != 2:
        raise L.TecoganB200Error('warp_s2d_concat: shape mismatch')
    if out is None:
        out = torch.empty((n, h, w, cpad), dtype=torch.float16, device=lr_curr.device)
    L.check(L.load().tg_warp_s2d_concat_lrflow(_ptr(hr_prev), _ptr(lr_flow), _ptr(lr_curr), _ptr(out),
                                               n, c, h, w, h8, w8, scale, up_mode, cpad, _stream()),
            'tg_warp_s2d_concat_lrflow')
    return out


# ---------------------------------------------------------------------------- NHWC fp16 helpers
def maxpool2x2(x, y=None):
    _req(x, torch.float16, 'maxpool input', 4)
    n, h, w, c = x.shape
    if y is None:
        y = torch.empty((n, h // 2, w // 2, c), dtype=torch.float16, device=x.device)
    L.check(L.load().tg_maxpool2x2_nhwc_f16(_ptr(x), _ptr(y), n, h, w, c, _stream()), 'tg_maxpool2x2')
    return y


def upsample2x(x, y=None):
    _req(x, torch.float16, 'upsample2x input', 4)
    n, h, w, c = x.shape
    if y is None:
        y = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.float16, device=x.device)
    L.check(L.load().tg_upsample2x_bilinear_nhwc_f16(_ptr(x), _ptr(y), n, h, w, c, _stream()),
            'tg_upsample2x')
    return y


def pack_pair(x1, x2, y=None, cpad=64):
    _req(x1, torch.float32, 'x1', 4)
    _req(x2, torch.float32, 'x2', 4)
    n, c, h, w = x1.shape
    if y is None:
        y = torch.empty((n, h, w, cpad), dtype=torch.float16, device=x1.device)
    L.check(L.load().tg_pack_pair_nhwc_f16(_ptr(x1), _ptr(x2), _ptr(y), n, c, h, w, cpad, _stream()),
            'tg_pack_pair')
    return y


def nchw_to_nhwc(x, cpad=None, y=None):
    _req(x, torch.float32, 'x', 4)
    n, c, h, w = x.shape
    cpad = cpad or pad64(c)
    if y is None:
        y = torch.empty((n, h, w, cpad), dtype=torch.float16, device=x.device)
    L.check(L.load().tg_nchw_f32_to_nhwc_f16(_ptr(x), _ptr(y), n, c, h, w, cpad, 0, _stream()),
            'tg_nchw_to_nhwc')
    return y


def nhwc_to_nchw(x, c, y=None):
    _req(x, torch.float16, 'x', 4)
    n, h, w, cpad = x.shape
    if y is None:
        y = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    L.check(L.load().tg_nhwc_f16_to_nchw_f32(_ptr(x), _ptr(y), n, c, h, w, cpad, _stream()),
            'tg_nhwc_to_nchw')
    return y


# ---------------------------------------------------------------------------- NCHW fp32 module ops
def backward_warp(x, flow, y=None):
    _req(x, torch.float32, 'x', 4)
    _req(flow, torch.float32, 'flow', 4)
    n, c, h, w = x.shape
    if tuple(flow.shape) != (n, 2, h, w):
        raise L.TecoganB200Error('backward_warp: flow shape mismatch')
    if y is None:
        y = torch.empty_like(x)
    L.check(L.load().tg_backward_warp_nchw_f32(_ptr(x), _ptr(flow), _ptr(y), n, c, h, w, _stream()),
            'tg_backward_warp')
    return y


def space_to_depth(x, scale, y=None):
    _req(x, torch.float32, 'x', 4)
    n, c, h, w = x.shape
    if y is None:
        y = torch.empty((n, c * scale * scale, h // scale, w // scale), dtype=torch.float32, device=x.device)
    L.check(L.load().tg_space_to_depth_nchw_f32(_ptr(x), _ptr(y), n, c, h, w, scale, _stream()),
            'tg_space_to_depth')
    return y


def upsample(x, scale, up_mode, out_hw=None, mul=1.0, y=None, accumulate=False):
    """[y +] mul * upsample_func(reflect_pad(x -> out_hw)); out_hw defaults to x's own size."""
    _req(x, torch.float32, 'x', 4)
    n, c, hin, win = x.shape
    h, w = out_hw if out_hw is not None else (hin, win)
    if y is None:
        y = torch.empty((n, c, h * scale, w * scale), dtype=torch.float32, device=x.device)
    L.check(L.load().tg_upsample_nchw_f32(_ptr(x), _ptr(y), n, c, hin, win, h, w, scale, up_mode,
                                          ctypes.c_float(mul), int(accumulate), _stream()), 'tg_upsample')
    return y


def downsample_bd(x, k2d, scale, pad_data, y=None):
    """x NCHW fp32, k2d [k,k] fp32 (device) -> blurred + subsampled NCHW fp32 (tg_downsample_bd_nchw_f32)."""
    _req(x, torch.float32, 'data', 4)
    _req(k2d, torch.float32, 'kernel', 2)
    n, c, H, W = x.shape
    k = k2d.shape[0]
    if k2d.shape[1] != k:
        raise L.TecoganB200Error('downsample_bd: kernel must be square')
    Hp, Wp = (H + k - 1, W + k - 1) if pad_data else (H, W)
    oh, ow = (Hp - k) // scale + 1, (Wp - k) // scale + 1
    if y is None:
        y = torch.empty((n, c, oh, ow), dtype=torch.float32, device=x.device)
    L.check(L.load().tg_downsample_bd_nchw_f32(_ptr(x), _ptr(k2d), _ptr(y), n, c, H, W, k, scale,
                                               1 if pad_data else 0, _stream()), 'tg_downsample_bd')
    return y


def float_to_uint8_nhwc(x, y=None):
    _req(x, torch.float32, 'x', 4)
    n, c, h, w = x.shape
    if y is None:
        y = torch.empty((n, h, w, c), dtype=torch.uint8, device=x.device)
    L.check(L.load().tg_float_to_uint8_nhwc(_ptr(x), _ptr(y), n, c, h, w, _stream()),
            'tg_float_to_uint8')
    return y


# ============================================================================ training (backward) ops
class GradScale:
    """Device-resident loss scale {scale, 1/scale} of the fp16 gradient path (tg_grad_scale_from_amax /
    tg_flow_head_bwd choose it on the device -- no host round trip)."""

    # amax of the incoming gradient is scaled to ~2^8: 2^8 of headroom below fp16 max.  The scale is capped at
    # 2^24 (scale_from_amax_kernel), so for a mean-reduced loss over N elements (gradients ~1/N) the stored amax
    # is ~2^24/N rather than 2^8.  That is adequate: in the fp16 CPU model (tests/fake_ops.py, 10 blocks,
    # 19 frames) lifting the cap moves the parameter gradients by <= 2e-4 rel-L2, while fp16 storage as a whole
    # costs up to ~1e-2.  tests/gpu_checks.py pins the cap (check_backward_elementwise_large).
    TARGET = 256.0

    def __init__(self, device):
        self.ws = torch.zeros(4, dtype=torch.float32, device=device)       # 16 bytes, zeroed once

    def from_amax(self, a, b=None, target=None):
        _req(a, torch.float32, 'grad')
        if b is not None:
            _req(b, torch.float32, 'grad')
        L.check(L.load().tg_grad_scale_from_amax(_ptr(a), a.numel(), _ptr(b), b.numel() if b is not None else 0,
                                                 ctypes.c_float(target or self.TARGET), _ptr(self.ws), _stream()),
                'tg_grad_scale_from_amax')
        global LAUNCH_COUNT
        LAUNCH_COUNT += 1            # two kernels per call
        return self

    @property
    def ptr(self):
        return ctypes.c_void_p(self.ws.data_ptr())


def _scale_ptr(scale):
    return scale.ptr if scale is not None else ctypes.c_void_p(0)


class PackedDgrad:
    """Data-gradient operand of a conv layer: the same tcgen05 implicit GEMM with the roles of the
    channel dimensions swapped -- conv3x3: taps flipped (tg_pack_conv3x3_weights_dgrad); convT3x3s2: a
    stride-2 conv over the output gradient (TG_CONV_3X3_S2).  Built from the forward PackedConv."""

    def __init__(self, fwd, weight):
        self.fwd = fwd
        self.kind = L.CONV_3X3 if fwd.kind == L.CONV_3X3 else L.CONV_3X3_S2
        self.cin = pad64(fwd.cout_real)        # channels of dz
        self.cout = fwd.cin                    # channels of the input gradient (stored)
        self.packed = None
        self._ver = None
        self.refresh(weight)

    def refresh(self, weight, force=False):
        ver = (weight._version, weight.data_ptr())
        if ver == self._ver and not force:
            return
        lib = L.load()
        w = _req(weight.detach(), torch.float32, 'weight', 4)
        if self.packed is None:
            self.packed = torch.empty(lib.tg_packed_weight_bytes(self.cin, self.cout), dtype=torch.uint8, device=w.device)
            self.bias = torch.zeros(self.cout, dtype=torch.float32, device=w.device)
        f = self.fwd
        if self.kind == L.CONV_3X3:
            rc = lib.tg_pack_conv3x3_weights_dgrad(_ptr(w), f.cout_real, f.cin_real, _ptr(self.packed), self.cout,
                                                   self.cin, _stream())
        else:   # nn.ConvTranspose2d weight [cin,cout,3,3] read as OIHW with out = cin, in = cout
            rc = lib.tg_pack_conv3x3s2_weights(_ptr(w), f.cin_real, f.cout_real, _ptr(self.packed), self.cout,
                                               self.cin, _stream())
        L.check(rc, 'tg_pack_weights (dgrad)')
        self._ver = ver

    def __call__(self, dz, y=None, residual=None, mask=None, mask_act=L.ACT_NONE, impl=None, max_ctas=0):
        """dz NHWC fp16 [n,oh,ow,cin] -> gradient w.r.t. the layer input [n,h,w,cout];
        y = (conv [+ residual]) * act'(mask).  max_ctas > 0 caps the persistent grid (tcgen05 only)."""
        _req(dz, torch.float16, 'dz', 4)
        n, oh, ow, c = dz.shape
        if c != self.cin:
            raise L.TecoganB200Error(f'dgrad: dz has {c} channels, expected {self.cin}')
        if self.kind == L.CONV_3X3_S2:
            if oh % 2 or ow % 2:
                raise L.TecoganB200Error('dgrad of the transposed conv needs even output sizes')
            h, w = oh // 2, ow // 2
        else:
            h, w = oh, ow
        if y is None:
            y = torch.empty((n, h, w, self.cout), dtype=torch.float16, device=dz.device)
        for t, nm in ((y, 'dx'), (residual, 'residual'), (mask, 'mask')):
            if t is not None:
                _req(t, torch.float16, nm, 4)
                if tuple(t.shape) != (n, h, w, self.cout):
                    raise L.TecoganB200Error(f'dgrad: {nm} shape {tuple(t.shape)} != {(n, h, w, self.cout)}')
        if (mask is not None) != (mask_act in (L.ACT_RELU, L.ACT_LRELU02)):
            raise L.TecoganB200Error('dgrad: mask and mask_act (RELU / LRELU02) go together')
        d = L.ConvDesc()
        d.x, d.weights, d.bias = dz.data_ptr(), self.packed.data_ptr(), self.bias.data_ptr()
        d.residual = residual.data_ptr() if residual is not None else None
        d.mask = mask.data_ptr() if mask is not None else None
        d.y = y.data_ptr()
        d.n, d.h, d.w, d.cin, d.cout, d.cout_real = n, h, w, self.cin, self.cout, self.cout
        d.kind, d.epilogue = self.kind, L.EPI_NHWC_F16
        d.act = {L.ACT_NONE: L.ACT_NONE, L.ACT_RELU: L.ACT_DRELU, L.ACT_LRELU02: L.ACT_DLRELU02}[mask_act]
        d.a_mode = L.AMODE_AUTO
        d.max_ctas = max_ctas
        d.cin_real = self.fwd.cout_real          # dz channels beyond the layer's real outputs are zero
        impl = impl or default_conv_impl()
        lib = L.load()
        if impl == 'tcgen05':
            L.check(lib.tg_conv_tcgen05(ctypes.byref(d), _stream()), 'tg_conv_tcgen05 (dgrad)')
        else:
            L.check(lib.tg_conv_simt(ctypes.byref(d), _stream()), 'tg_conv_simt (dgrad)')
        return y


def wgrad(fwd, x, dz, dw, scale=None, impl=None, max_ctas=0, db=None):
    """dw (fp32, the parameter's layout, pre-zeroed or accumulating) += 1/scale * x (*) dz for the
    forward layer `fwd` (PackedConv): x = its NHWC fp16 input, dz = gradient of its pre-activation
    output (NHWC fp16, pad64(cout_real) channels)."""
    _req(x, torch.float16, 'x', 4)
    _req(dz, torch.float16, 'dz', 4)
    _req(dw, torch.float32, 'dw', 4)
    n, h, w, cin = x.shape
    up = 2 if fwd.kind == L.CONVT_3X3_S2 else 1
    cout = pad64(fwd.cout_real)
    if cin != fwd.cin or tuple(dz.shape) != (n, up * h, up * w, cout):
        raise L.TecoganB200Error(f'wgrad: shapes x {tuple(x.shape)} dz {tuple(dz.shape)} do not fit the layer')
    want = (fwd.cout_real, fwd.cin_real, 3, 3) if fwd.kind == L.CONV_3X3 else (fwd.cin_real, fwd.cout_real, 3, 3)
    if tuple(dw.shape) != want:
        raise L.TecoganB200Error(f'wgrad: dw shape {tuple(dw.shape)} != {want}')
    d = L.WgradDesc()
    d.x, d.dz, d.dw = x.data_ptr(), dz.data_ptr(), dw.data_ptr()
    d.scale = scale.ws.data_ptr() if scale is not None else None
    fuse_db = db is not None and fwd.kind == L.CONV_3X3 and (impl or default_conv_impl()) == 'tcgen05'
    if db is not None:
        _req(db, torch.float32, 'db', 1)
        if db.numel() != fwd.cout_real:
            raise L.TecoganB200Error('wgrad: db must have cout_real elements')
        if fuse_db:
            d.db = db.data_ptr()            # bias gradient from the same MMAs
    d.n, d.h, d.w, d.cin, d.cout = n, h, w, cin, cout
    d.cin_real, d.cout_real, d.kind, d.max_ctas, d.reserved = fwd.cin_real, fwd.cout_real, fwd.kind, max_ctas, 0
    lib = L.load()
    impl = impl or default_conv_impl()
    if impl == 'tcgen05':
        L.check(lib.tg_wgrad_tcgen05(ctypes.byref(d), _stream()), 'tg_wgrad_tcgen05')
    else:
        L.check(lib.tg_wgrad_simt(ctypes.byref(d), _stream()), 'tg_wgrad_simt')
    if db is not None and not fuse_db:
        bias_grad(dz, db, scale)            # transposed conv / cross-check path: separate reduction kernel
    return dw


def bias_grad(dz, db, scale=None):
    """db (fp32 [c_real]) += 1/scale * sum over pixels of dz[..., :c_real]"""
    _req(dz, torch.float16, 'dz', 4)
    _req(db, torch.float32, 'db', 1)
    c = dz.shape[-1]
    L.check(L.load().tg_bias_grad_nhwc_f16(_ptr(dz), dz.numel() // c, c, db.numel(), _scale_ptr(scale), _ptr(db),
                                           _stream()), 'tg_bias_grad')
    return db


def grad_pack(a, b=None, scale=None, cpad=64, y=None):
    """(a [+ b]) * scale : NCHW fp32 -> NHWC fp16 (cpad channels)"""
    _req(a, torch.float32, 'grad', 4)
    if b is not None:
        _req(b, torch.float32, 'grad', 4)
    n, c, h, w = a.shape
    if y is None:
        y = torch.empty((n, h, w, cpad), dtype=torch.float16, device=a.device)
    L.check(L.load().tg_grad_pack_nhwc_f16(_ptr(a), _ptr(b), _scale_ptr(scale), _ptr(y), n, c, h, w, cpad, _stream()),
            'tg_grad_pack')
    return y


def grad_unpack(x, c, scale=None, c_offset=0, y=None, accumulate=False):
    """channels [c_offset, c_offset+c) of NHWC fp16 -> NCHW fp32 / scale"""
    _req(x, torch.float16, 'x', 4)
    n, h, w, cpad = x.shape
    if y is None:
        y = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    L.check(L.load().tg_grad_unpack_nchw_f32(_ptr(x), _scale_ptr(scale), _ptr(y), n, c, h, w, cpad, c_offset,
                                             int(accumulate), _stream()), 'tg_grad_unpack')
    return y


def backward_warp_bwd(x, flow, gy, need_x=True, need_flow=True):
    """-> (gx, gflow) of backward_warp(x, flow) given gy; outputs not needed are None"""
    _req(x, torch.float32, 'x', 4)
    _req(flow, torch.float32, 'flow', 4)
    _req(gy, torch.float32, 'gy', 4)
    n, c, h, w = x.shape
    gx = torch.zeros_like(x) if need_x else None              # scatter-add target
    gf = torch.empty_like(flow) if need_flow else None
    L.check(L.load().tg_backward_warp_bwd_nchw_f32(_ptr(x), _ptr(flow), _ptr(gy), _ptr(gx), _ptr(gf), n, c, h, w,
                                                   _stream()), 'tg_backward_warp_bwd')
    return gx, gf


def warp_s2d_concat_bwd(gx, hr_prev, hr_flow, scale_factor, d_hr_prev=None, d_hr_flow=None, scale=None):
    """gradient of warp_s2d_concat_hrflow: accumulates into d_hr_prev (fp32 NCHW), stores d_hr_flow"""
    _req(gx, torch.float16, 'gx', 4)
    _req(hr_prev, torch.float32, 'hr_prev', 4)
    _req(hr_flow, torch.float32, 'hr_flow', 4)
    n, h, w, cpad = gx.shape
    c = hr_prev.shape[1]
    L.check(L.load().tg_warp_s2d_concat_bwd(_ptr(gx), _ptr(hr_prev), _ptr(hr_flow), _scale_ptr(scale), _ptr(d_hr_prev),
                                            _ptr(d_hr_flow), n, c, h, w, scale_factor, cpad, _stream()),
            'tg_warp_s2d_concat_bwd')


def upsample_bwd(gy, scale_factor, up_mode, mul=1.0, gx=None, accumulate=False):
    _req(gy, torch.float32, 'gy', 4)
    n, c, H, W = gy.shape
    h, w = H // scale_factor, W // scale_factor
    if gx is None:
        gx = torch.empty((n, c, h, w), dtype=torch.float32, device=gy.device)
    L.check(L.load().tg_upsample_bwd_nchw_f32(_ptr(gy), _ptr(gx), n, c, h, w, scale_factor, up_mode, ctypes.c_float(mul),
                                              int(accumulate), _stream()), 'tg_upsample_bwd')
    return gx


def maxpool2x2_bwd(x, gy, act, gx=None):
    _req(x, torch.float16, 'x', 4)
    _req(gy, torch.float16, 'gy', 4)
    n, h, w, c = x.shape
    if gx is None:
        gx = torch.empty_like(x)
    L.check(L.load().tg_maxpool2x2_bwd_nhwc_f16(_ptr(x), _ptr(gy), _ptr(gx), n, h, w, c, act, _stream()),
            'tg_maxpool2x2_bwd')
    return gx


def upsample2x_bwd(gy, m, act, gx=None):
    _req(gy, torch.float16, 'gy', 4)
    _req(m, torch.float16, 'm', 4)
    n, h, w, c = m.shape
    if gx is None:
        gx = torch.empty_like(m)
    L.check(L.load().tg_upsample2x_bilinear_bwd_nhwc_f16(_ptr(gy), _ptr(m), _ptr(gx), n, h, w, c, act, _stream()),
            'tg_upsample2x_bwd')
    return gx


def flow_head_bwd(gflow, flow, scale, gflow2=None, cpad=64, dz=None):
    """dz (NHWC fp16) of the 24*tanh flow head; also chooses `scale` (GradScale) for the FNet backward"""
    _req(gflow, torch.float32, 'gflow', 4)
    _req(flow, torch.float32, 'flow', 4)
    n, _, h, w = flow.shape
    if dz is None:
        dz = torch.empty((n, h, w, cpad), dtype=torch.float16, device=flow.device)
    L.check(L.load().tg_flow_head_bwd(_ptr(gflow), _ptr(gflow2), _ptr(flow), scale.ptr, ctypes.c_float(scale.TARGET),
                                      _ptr(dz), n, h, w, cpad, _stream()), 'tg_flow_head_bwd')
    global LAUNCH_COUNT
    LAUNCH_COUNT += 2
    return dz


def depth_to_space(gy, scale_factor):
    _req(gy, torch.float32, 'gy', 4)
    n, cs, oh, ow = gy.shape
    c = cs // (scale_factor * scale_factor)
    gx = torch.empty((n, c, oh * scale_factor, ow * scale_factor), dtype=torch.float32, device=gy.device)
    L.check(L.load().tg_depth_to_space_nchw_f32(_ptr(gy), _ptr(gx), n, c, oh * scale_factor, ow * scale_factor,
                                                scale_factor, _stream()), 'tg_depth_to_space')
    return gx


def st_disc_input(data, bi, flow, t, pad, csize, out=None):
    """[orig | crop_pad(warp) | cond] input of the spatio-temporal discriminator (tg_st_disc_input_nchw_f32)"""
    _req(data, torch.float32, 'data', 5)
    _req(bi, torch.float32, 'bi_data', 5)
    _req(flow, torch.float32, 'hr_flow_merge', 4)
    n, t_full, c, h, w = data.shape
    if bi.shape[0] != n or bi.shape[1] < t or tuple(bi.shape[2:]) != (c, h, w) or bi.shape[1] != t_full:
        raise L.TecoganB200Error(f'st_disc_input: bi_data shape {tuple(bi.shape)} does not match data {tuple(data.shape)}')
    if tuple(flow.shape) != (n * t, 2, h, w):
        raise L.TecoganB200Error(f'st_disc_input: flow shape {tuple(flow.shape)} != {(n * t, 2, h, w)}')
    if out is None:
        out = torch.empty((n * t // 3, 9 * c, h, w), dtype=torch.float32, device=data.device)
    L.check(L.load().tg_st_disc_input_nchw_f32(_ptr(data), _ptr(bi), _ptr(flow), _ptr(out), n, t_full, t, c, h, w, pad,
                                               csize, _stream()), 'tg_st_disc_input')
    return out


def st_disc_input_bwd(gout, flow, shape, t, pad, csize):
    _req(gout, torch.float32, 'gout', 4)
    n, t_full, c, h, w = shape
    gdata = torch.zeros(shape, dtype=torch.float32, device=gout.device)
    L.check(L.load().tg_st_disc_input_bwd_nchw_f32(_ptr(gout), _ptr(flow), _ptr(gdata), n, t_full, t, c, h, w, pad, csize,
                                                   _stream()), 'tg_st_disc_input_bwd')
    return gdata
