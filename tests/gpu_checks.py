"""GPU parity checks of the CUDA path against the CPU oracle (oracle/) and the committed golden
fixtures (tests/golden).  Each check is a plain function returning a dict of measured errors and
raising AssertionError on a parity failure, so the same code backs

  * tests/test_gpu_parity.py   (pytest -m gpu, what the driver runs), and
  * tests/gpu_diag.py          (each check in its own process with a timeout; bring-up tool).

Nothing here reads /root/reference.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import tecogan_b200 as T                      # noqa: E402
from oracle import ops_oracle as K            # noqa: E402
from oracle import frnet_oracle as O          # noqa: E402

ops = sys.modules['tecogan-pytorch_b200.ops']
L = sys.modules['tecogan-pytorch_b200.lib']
G = os.path.join(ROOT, 'tests', 'golden')
DEV = 'cuda:0'


def rand(seed, *shape, lo=0.0, hi=1.0):
    return torch.from_numpy(np.random.default_rng(seed).uniform(lo, hi, size=shape).astype(np.float32))


def relmax(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-12))


def rell2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-12))


def f16(x):
    """round to fp16 and back (the storage precision of the CUDA path)"""
    return x.half().float()


def nhwc(x_nchw_f32, cpad=64):
    """CPU NCHW fp32 -> CUDA NHWC fp16 padded to cpad channels"""
    n, c, h, w = x_nchw_f32.shape
    y = torch.zeros(n, h, w, cpad, dtype=torch.float16)
    y[..., :c] = x_nchw_f32.permute(0, 2, 3, 1).half()
    return y.to(DEV)


def from_nhwc(y, c):
    return y[..., :c].float().permute(0, 3, 1, 2).contiguous().cpu()


# =============================================================================== elementwise
def check_warp_hrflow(scale=4, h=11, w=37, n=2):
    hr_prev = rand(1, n, 3, scale * h, scale * w)
    flow = rand(2, n, 2, scale * h, scale * w, lo=-6, hi=6)
    flow[0, :, 0, 0] = torch.tensor([-100.0, 100.0])
    flow[0, :, -1, -1] = torch.tensor([100.0, -100.0])
    lr = rand(3, n, 3, h, w)
    got = ops.warp_s2d_concat_hrflow(hr_prev.to(DEV), flow.to(DEV), lr.to(DEV), scale)
    torch.cuda.synchronize()
    ref = K.warp_s2d_concat(hr_prev.numpy(), flow.numpy(), lr.numpy(), scale)
    c_used = (scale * scale + 1) * 3
    got_f = from_nhwc(got, c_used).numpy()
    # index math: every output element must be the fp16 rounding of the oracle value up to the
    # closed-form grid (x+u vs the reference's normalised round trip: <= ~1e-4 px)
    err = np.abs(got_f - ref).max()
    assert err <= 2e-3, f'warp_hrflow max abs err {err}'
    assert np.array_equal(got_f[:, :3], f16(lr).numpy()), 'lr_curr channels must be exact fp16 copies'
    assert float(got[..., c_used:].abs().max()) == 0.0, 'pad channels must be zero'
    # space_to_depth placement exactness: integer flow -> warp is an exact gather
    flow_i = torch.round(flow)
    got_i = ops.warp_s2d_concat_hrflow(hr_prev.to(DEV), flow_i.to(DEV), lr.to(DEV), scale)
    ref_i = K.warp_s2d_concat(hr_prev.numpy(), flow_i.numpy(), lr.numpy(), scale, exact_reference_grid=False)
    assert np.array_equal(from_nhwc(got_i, c_used).numpy(), f16(torch.from_numpy(ref_i)).numpy()), \
        'integer-flow warp + space_to_depth must be bit exact'
    return {'max_abs': float(err)}


def check_warp_lrflow(scale=4, mode='BD', h=18, w=28, n=2):
    h8, w8 = h // 8 * 8, w // 8 * 8
    hr_prev = rand(4, n, 3, scale * h, scale * w)
    lr_flow = rand(5, n, 2, h8, w8, lo=-3, hi=3)
    lr = rand(6, n, 3, h, w)
    up_mode = L.UP_BICUBIC if mode == 'BD' else L.UP_BILINEAR
    got = ops.warp_s2d_concat_lrflow(hr_prev.to(DEV), lr_flow.to(DEV), lr.to(DEV), scale, up_mode)
    pad = K.reflect_pad_flow(lr_flow.numpy(), h - h8, w - w8)
    up = K.bicubic_upsample(pad, scale) if mode == 'BD' else K.bilinear_upsample(pad, scale)
    hr_flow = np.float32(scale) * up
    ref = K.warp_s2d_concat(hr_prev.numpy(), hr_flow, lr.numpy(), scale)
    c_used = (scale * scale + 1) * 3
    err = np.abs(from_nhwc(got, c_used).numpy() - ref).max()
    assert err <= 2e-3, f'warp_lrflow({mode},{scale}) max abs err {err}'
    # the standalone flow upsampler must agree with the oracle to fp32 rounding
    hf = ops.upsample(lr_flow.to(DEV), scale, up_mode, out_hw=(h, w), mul=float(scale)).cpu().numpy()
    e2 = np.abs(hf - hr_flow).max()
    assert e2 <= 2e-5, f'flow upsample err {e2}'
    return {'max_abs': float(err), 'flow_up_abs': float(e2)}


def check_pool_upsample():
    x = rand(7, 2, 64, 13, 22, lo=-2, hi=2)
    xg = nhwc(x)
    p = from_nhwc(ops.maxpool2x2(xg), 64).numpy()
    assert np.array_equal(p, K.maxpool2x2(f16(x).numpy())), 'maxpool must be exact'
    u = from_nhwc(ops.upsample2x(xg), 64).numpy()
    ref = K.bilinear_upsample(f16(x).numpy(), 2)
    err = np.abs(u - ref).max()
    assert err <= 2e-3, f'upsample2x err {err}'
    a, b = rand(8, 2, 3, 9, 14), rand(9, 2, 3, 9, 14)
    pk = ops.pack_pair(a.to(DEV), b.to(DEV))
    assert np.array_equal(from_nhwc(pk, 6).numpy(), f16(torch.cat([a, b], 1)).numpy())
    assert float(pk[..., 6:].abs().max()) == 0.0
    return {'upsample2x_abs': float(err)}


def check_module_ops():
    g = np.load(os.path.join(G, 'ops.npz'))
    x = rand(20, 2, 3, 20, 24)
    flow = rand(21, 2, 2, 20, 24, lo=-4.0, hi=4.0)
    flow[0, :, 0, 0] = torch.tensor([-30.0, 40.0])
    w = T.backward_warp(x.to(DEV), flow.to(DEV)).cpu().numpy()
    e_w = np.abs(w - g['warped']).max()
    assert e_w <= 2e-5, f'backward_warp vs reference golden {e_w}'
    s4 = T.space_to_depth(rand(22, 2, 3, 16, 24).to(DEV), 4).cpu().numpy()
    s2 = T.space_to_depth(rand(22, 2, 3, 16, 24).to(DEV), 2).cpu().numpy()
    assert np.array_equal(s4, g['s2d4']) and np.array_equal(s2, g['s2d2']), 'space_to_depth bit exact'
    xs = rand(23, 1, 3, 9, 11).to(DEV)
    e_b = max(np.abs(T.get_upsampling_func(4, 'BD')(xs).cpu().numpy() - g['bic4']).max(),
              np.abs(T.get_upsampling_func(2, 'BD')(xs).cpu().numpy() - g['bic2']).max(),
              np.abs(T.get_upsampling_func(4, 'BI')(xs).cpu().numpy() - g['bil4']).max(),
              np.abs(T.get_upsampling_func(2, 'BI')(xs).cpu().numpy() - g['bil2']).max())
    assert e_b <= 2e-6, f'upsample_func vs reference golden {e_b}'
    q_in = torch.from_numpy(g['q_in']).reshape(1, 1, 1, -1).to(DEV)
    q = ops.float_to_uint8_nhwc(q_in).cpu().numpy().reshape(-1)
    assert np.array_equal(q, g['q']), 'uint8 quantisation (round-half-even) must be bit exact'
    return {'warp_abs': float(e_w), 'upsample_abs': float(e_b)}


def check_downsample_bd():
    """tg_downsample_bd_nchw_f32 (through the data_utils drop-in) vs the reference-generated fixture
    and the oracle, incl. a frame-sized input."""
    g = np.load(os.path.join(G, 'downsample_bd.npz'))
    kern = T.create_kernel(1.5)
    res = {}
    for name, seed, shape, s, pad in (('s4_pad', 30, (2, 3, 36, 44), 4, True), ('s4_valid', 31, (1, 3, 41, 45), 4, False),
                                      ('s2_pad', 32, (1, 3, 27, 30), 2, True)):
        y = T.downsample_bd(rand(seed, *shape).to(DEV), kern, s, pad).cpu().numpy()
        assert y.shape == g[name].shape, (name, y.shape, g[name].shape)
        res[name] = float(np.abs(y - g[name]).max())
        assert res[name] <= 2e-6, f'downsample_bd {name}: max abs {res[name]}'
    x = rand(33, 1, 3, 536, 1280)
    y = T.downsample_bd(x.to(DEV), kern, 4, True).cpu().numpy()
    ref = K.downsample_bd(x.numpy(), K.create_kernel(1.5), 4, True)
    assert y.shape == (1, 3, 134, 320)
    res['frame'] = float(np.abs(y - ref).max())
    assert res['frame'] <= 2e-6
    return res


# =============================================================================== convolutions
def _conv_ref(x, wt, b, kind, act, residual=None):
    """CPU fp32 reference on fp16-rounded operands."""
    xr, wr = f16(x), f16(wt)
    if kind == L.CONV_3X3:
        y = F.conv2d(xr, wr, b, padding=1)
    else:
        y = torch.from_numpy(K.conv_transpose3x3s2_parity(xr.numpy(), wr.numpy(), b.numpy()))
    if act == L.ACT_RELU:
        y = y.clamp_min(0)
    elif act == L.ACT_LRELU02:
        y = torch.where(y >= 0, y, 0.2 * y)
    if residual is not None:
        y = y + f16(residual)
    return y


def check_conv(impl='tcgen05', a_mode=None, cin=64, cout=64, h=20, w=24, n=2, kind=None,
               act=None, residual=False, seed=30, cin_real=None, cout_real=None):
    kind = L.CONV_3X3 if kind is None else kind
    act = L.ACT_RELU if act is None else act
    cin_real = cin_real or cin
    cout_real = cout_real or cout
    x = rand(seed, n, cin_real, h, w, lo=-1, hi=1)
    bound = 1.5 / np.sqrt(9 * cin_real)
    wshape = (cout_real, cin_real, 3, 3) if kind == L.CONV_3X3 else (cin_real, cout_real, 3, 3)
    wt = rand(seed + 1, *wshape, lo=-bound, hi=bound)
    b = rand(seed + 2, cout_real, lo=-0.5, hi=0.5)
    res = rand(seed + 3, n, cout_real, h, w, lo=-1, hi=1) if residual else None
    pc = ops.PackedConv(wt.to(DEV), b.to(DEV), kind, act)
    assert pc.cin == cin and pc.cout == cout
    y = pc(nhwc(x, cin), residual=nhwc(res, cout) if residual else None, impl=impl, a_mode=a_mode)
    torch.cuda.synchronize()
    ref = _conv_ref(x, wt, b, kind, act, res)
    got = from_nhwc(y, cout_real)
    e = relmax(got.numpy(), ref.numpy())
    assert e <= 3e-3, f'conv {impl} amode={a_mode} cin={cin} cout={cout} kind={kind}: rel max err {e}'
    if cout_real < cout:
        assert float(y[..., cout_real:].abs().max()) == 0.0, 'padded output channels must be zero'
    return {'rel_max': e, 'rel_l2': rell2(got.numpy(), ref.numpy())}


def check_conv_vs_simt(a_mode=None, cin=64, cout=64, h=134, w=320, n=1, kind=None, residual=True,
                       max_ctas=0):
    """tcgen05 vs the CUDA-core kernel on identical packed weights: only the fp32 summation
    order differs, so after fp16 rounding they agree to 1 ulp almost everywhere."""
    kind = L.CONV_3X3 if kind is None else kind
    residual = residual and kind == L.CONV_3X3
    x = nhwc(rand(40, n, cin, h, w, lo=-1, hi=1), cin)
    bound = 1.5 / np.sqrt(9 * cin)
    wshape = (cout, cin, 3, 3) if kind == L.CONV_3X3 else (cin, cout, 3, 3)
    pc = ops.PackedConv(rand(41, *wshape, lo=-bound, hi=bound).to(DEV),
                        rand(42, cout, lo=-0.5, hi=0.5).to(DEV), kind, L.ACT_RELU)
    res = nhwc(rand(43, n, cout, h, w, lo=-1, hi=1), cout) if residual else None
    a = pc(x, residual=res, impl='tcgen05', a_mode=a_mode, max_ctas=max_ctas)
    b = pc(x, residual=res, impl='simt')
    torch.cuda.synchronize()
    d = (a.float() - b.float()).abs()
    e = float(d.max() / b.float().abs().max())
    frac = float((d > 0).float().mean())
    assert e <= 2e-3, f'tcgen05 vs simt: rel max {e} (differing elements {frac:.4f})'
    return {'rel_max': e, 'frac_diff': frac}


def check_conv_issue_variants(kind=None, cin_real=64, cout_real=64, h=61, w=45, n=3, residual=False):
    """The halo convs' issue variants are the same arithmetic in the same order and must agree BIT FOR BIT:
    two MMA issuer warps (default) vs one (TG_DBG_FLAGS=16, read per launch), and the thin-layer k-step skip
    (tg_conv_desc.cin_real) vs all four k-steps (cin_real = 0: the skipped products are x * 0)."""
    kind = L.CONV_3X3 if kind is None else kind
    cin, cout = 64, 64
    x = nhwc(rand(140, n, cin_real, h, w, lo=-1, hi=1), cin)
    bound = 1.5 / np.sqrt(9 * cin_real)
    wshape = (cout_real, cin_real, 3, 3) if kind == L.CONV_3X3 else (cin_real, cout_real, 3, 3)
    pc = ops.PackedConv(rand(141, *wshape, lo=-bound, hi=bound).to(DEV),
                        rand(142, cout_real, lo=-0.5, hi=0.5).to(DEV), kind, L.ACT_RELU)
    res = nhwc(rand(143, n, cout_real, h, w, lo=-1, hi=1), cout) if (residual and kind == L.CONV_3X3) else None
    old = os.environ.get('TG_DBG_FLAGS')
    try:
        os.environ.pop('TG_DBG_FLAGS', None)
        dual = pc(x, residual=res, impl='tcgen05', a_mode=L.AMODE_HALO)
        real = pc.cin_real
        pc.cin_real = 0                                  # descriptor says: every stored input channel may be non-zero
        dual_all_k = pc(x, residual=res, impl='tcgen05', a_mode=L.AMODE_HALO)
        pc.cin_real = real
        os.environ['TG_DBG_FLAGS'] = '16'
        single = pc(x, residual=res, impl='tcgen05', a_mode=L.AMODE_HALO)
    finally:
        if old is None:
            os.environ.pop('TG_DBG_FLAGS', None)
        else:
            os.environ['TG_DBG_FLAGS'] = old
    ref = pc(x, residual=res, impl='simt')
    torch.cuda.synchronize()
    assert torch.equal(dual, single), 'two issuers vs one issuer differ'
    assert torch.equal(dual, dual_all_k), 'k-step skip (cin_real) changed the result'
    e = float((dual.float() - ref.float()).abs().max() / ref.float().abs().max())
    assert e <= 2e-3, f'tcgen05 vs simt: rel max {e}'
    return {'bit_identical': True, 'rel_max_vs_simt': e}


def check_conv_chain(n=2, h=37, w=29, blocks=2, max_ctas=0, repeats=1, seed=50):
    """tg_conv_chain_tcgen05 (conv_in + `blocks` residual blocks in ONE persistent launch, tiles
    gated by progress flags) vs the same layers as 1+2*blocks launches of tg_conv_tcgen05 on
    identical packed weights: same MMAs in the same order, so the outputs are bit-identical (the
    tolerance only guards against a future change of the issue order); `repeats` relaunches on
    the same workspace exercise the epoch stamping of the flags.  The work buffers are poisoned
    with NaN so a tile consumed before it was produced cannot go unnoticed."""
    bound = 1.2 / np.sqrt(9 * 64)
    pcs = []
    for i in range(1 + 2 * blocks):
        act = L.ACT_RELU if (i == 0 or i % 2 == 1) else L.ACT_NONE
        pcs.append(ops.PackedConv(rand(seed + 3 * i, 64, 64, 3, 3, lo=-bound, hi=bound).to(DEV),
                                  rand(seed + 3 * i + 1, 64, lo=-0.2, hi=0.2).to(DEV), L.CONV_3X3, act))
    specs = [(pcs[0], 0, 1, None)]
    for b in range(blocks):
        specs += [(pcs[1 + 2 * b], 1, 2, None), (pcs[2 + 2 * b], 2, 1, 1)]
    chain = ops.ConvChain(specs)
    worst, frac = 0.0, 0.0
    for rep in range(repeats):
        x = nhwc(rand(seed + 100 + rep, n, 64, h, w, lo=-1, hi=1), 64)
        a = pcs[0](x)
        for b in range(blocks):
            t = pcs[1 + 2 * b](a)
            a = pcs[2 + 2 * b](t, residual=a)
        # poison the chain's work buffers: stale data must never be read before it is produced
        b1 = torch.full_like(x, float('nan'))
        b2 = torch.full_like(x, float('nan'))
        y = chain([x, b1, b2], max_ctas=max_ctas)
        torch.cuda.synchronize()
        assert torch.isfinite(y.float()).all(), f'chain output has non-finite values (rep {rep})'
        d = (y.float() - a.float()).abs()
        e = float(d.max() / a.float().abs().max())
        worst = max(worst, e)
        frac = max(frac, float((d > 0).float().mean()))
        assert e <= 4e-3, f'conv chain vs per-layer launches: rel max {e} (rep {rep}, n={n} h={h} w={w} blocks={blocks})'
    return {'rel_max': worst, 'frac_diff': frac}


def check_conv_chain_plain(n=2, h=33, w=50, layers=24, seed=90):
    """The longest chain the ABI takes (24 layers), no residuals, ping-pong over two work buffers,
    LeakyReLU between layers -- vs the same layers launched one by one."""
    bound = 1.4 / np.sqrt(9 * 64)
    pcs = [ops.PackedConv(rand(seed + 2 * i, 64, 64, 3, 3, lo=-bound, hi=bound).to(DEV),
                          rand(seed + 2 * i + 1, 64, lo=-0.1, hi=0.1).to(DEV), L.CONV_3X3, L.ACT_LRELU02)
           for i in range(layers)]
    specs = [(pcs[i], 0 if i == 0 else 1 + (i - 1) % 2, 1 + i % 2, None) for i in range(layers)]
    x = nhwc(rand(seed + 200, n, 64, h, w, lo=-1, hi=1), 64)
    a = x
    for pc in pcs:
        a = pc(a)
    y = ops.ConvChain(specs)([x, torch.full_like(x, float('nan')), torch.full_like(x, float('nan'))])
    torch.cuda.synchronize()
    assert torch.isfinite(y.float()).all()
    d = (y.float() - a.float()).abs()
    e = float(d.max() / a.float().abs().max())
    assert e <= 4e-3, f'24-layer chain vs per-layer launches: rel max {e}'
    return {'rel_max': e, 'frac_diff': float((d > 0).float().mean())}


def check_conv_chain_vs_reference(n=1, h=20, w=24, blocks=1, seed=70):
    """conv chain vs the CPU fp32 reference of the same three layers (fp16-rounded between layers)."""
    bound = 1.2 / np.sqrt(9 * 64)
    ws = [rand(seed + 3 * i, 64, 64, 3, 3, lo=-bound, hi=bound) for i in range(1 + 2 * blocks)]
    bs = [rand(seed + 3 * i + 1, 64, lo=-0.2, hi=0.2) for i in range(1 + 2 * blocks)]
    acts = [L.ACT_RELU if (i == 0 or i % 2 == 1) else L.ACT_NONE for i in range(1 + 2 * blocks)]
    pcs = [ops.PackedConv(ws[i].to(DEV), bs[i].to(DEV), L.CONV_3X3, acts[i]) for i in range(len(ws))]
    specs = [(pcs[0], 0, 1, None)]
    for b in range(blocks):
        specs += [(pcs[1 + 2 * b], 1, 2, None), (pcs[2 + 2 * b], 2, 1, 1)]
    x = rand(seed + 50, n, 64, h, w, lo=-1, hi=1)
    xd = nhwc(x, 64)
    y = ops.ConvChain(specs)([xd, torch.empty_like(xd), torch.empty_like(xd)])
    torch.cuda.synchronize()
    a = f16(_conv_ref(x, ws[0], bs[0], L.CONV_3X3, acts[0]))
    for b in range(blocks):
        t = f16(_conv_ref(a, ws[1 + 2 * b], bs[1 + 2 * b], L.CONV_3X3, acts[1 + 2 * b]))
        a = f16(_conv_ref(t, ws[2 + 2 * b], bs[2 + 2 * b], L.CONV_3X3, acts[2 + 2 * b], a))
    e = relmax(from_nhwc(y, 64).numpy(), a.numpy())
    assert e <= 4e-3, f'conv chain vs CPU reference: rel max {e}'
    return {'rel_max': e}


def check_conv_epilogues(impl='tcgen05'):
    out = {}
    # flow head: 24*tanh(conv) -> NCHW fp32 [n,2,h,w]
    x = rand(50, 2, 64, 16, 24, lo=-1, hi=1)
    wt = rand(51, 2, 64, 3, 3, lo=-0.08, hi=0.08)
    b = rand(52, 2, lo=-0.1, hi=0.1)
    pc = ops.PackedConv(wt.to(DEV), b.to(DEV), L.CONV_3X3, L.ACT_NONE, L.EPI_FLOW_NCHW_F32)
    y = pc(nhwc(x), impl=impl).cpu()
    ref = 24 * torch.tanh(F.conv2d(f16(x), f16(wt), b, padding=1))
    out['flow_rel'] = relmax(y.numpy(), ref.numpy())
    assert out['flow_rel'] <= 1e-3, out
    # output head: conv + bias + upsample_func(lr_curr) -> NCHW fp32
    for mode, s in (('BD', 4), ('BI', 2)):
        hh, ww = 6 * s, 10 * s
        x = rand(53, 1, 64, hh, ww, lo=-1, hi=1)
        wt = rand(54, 3, 64, 3, 3, lo=-0.08, hi=0.08)
        b = rand(55, 3, lo=-0.1, hi=0.1)
        lr = rand(56, 1, 3, 6, 10)
        pc = ops.PackedConv(wt.to(DEV), b.to(DEV), L.CONV_3X3, L.ACT_NONE, L.EPI_OUT_NCHW_F32)
        y = pc(nhwc(x), impl=impl)
        y = ops.upsample(lr.to(DEV), s, L.UP_BICUBIC if mode == 'BD' else L.UP_BILINEAR, y=y, accumulate=True).cpu()
        up = K.bicubic_upsample(lr.numpy(), s) if mode == 'BD' else K.bilinear_upsample(lr.numpy(), s)
        ref = F.conv2d(f16(x), f16(wt), b, padding=1) + torch.from_numpy(up)
        out[f'out_{mode}{s}_rel'] = relmax(y.numpy(), ref.numpy())
        assert out[f'out_{mode}{s}_rel'] <= 1e-3, out
    return out


# =============================================================================== FRNet end to end
def _net(seed, scale, degradation, gain, nb=10):
    net = T.FRNet(3, 3, 64, nb, degradation, scale)
    p = O.make_frnet_params(seed, nb=nb, scale=scale, degradation=degradation, gain=gain)
    net.load_state_dict(p, strict=True)
    return net.to(DEV).eval(), p


def check_step_golden(tag='g15'):
    """FRNet.step vs the reference-generated fp32 fixture (4x BD, 18x28: reflect pad 2/4).

    Two bars: (a) north star -- rel-L2 <= 1e-3 against the fp32 reference for PyTorch-default
    (g1) and 1.5x (g15) weights; (b) implementation -- for every gain, incl. the chaotic 2x
    weights where the fp16 design itself sits 3e-3 from fp32, the GPU result must be no further
    from the fixture than 1.5x the CPU precision model (oracle/frnet_fp16emu.py) + 1e-4."""
    from oracle import frnet_fp16emu as E
    gain = {'g1': 1.0, 'g15': 1.5, 'g2': 2.0}[tag]
    g = np.load(os.path.join(G, f'step_bd4_18x28_{tag}.npz'))
    net, p = _net(11, 4, 'BD', gain)
    lr_curr, lr_prev, hr_prev = rand(1, 1, 3, 18, 28), rand(2, 1, 3, 18, 28), rand(3, 1, 3, 72, 112)
    flow = net.fnet(lr_curr.to(DEV), lr_prev.to(DEV)).cpu().numpy()
    hr = net.step(lr_curr.to(DEV), lr_prev.to(DEV), hr_prev.to(DEV)).cpu().numpy()
    with torch.no_grad():
        emu, emu_flow = E.step(p, lr_curr, lr_prev, hr_prev, 4, 'BD')
    base = K.bicubic_upsample(lr_curr.numpy(), 4)          # the part of the output that is not conv
    out = {'flow_abs': float(np.abs(flow - g['lr_flow']).max()),
           'flow_absmax_ref': float(np.abs(g['lr_flow']).max()),
           'hr_rel_l2': rell2(hr, g['hr_curr']), 'hr_rel_max': relmax(hr, g['hr_curr']),
           'emu_rel_l2': rell2(emu.numpy(), g['hr_curr']),
           'gpu_vs_emu_rel_l2': rell2(hr, emu.numpy()),
           'conv_part_rel_l2': rell2(hr - base, g['hr_curr'] - base)}
    if tag in ('g1', 'g15'):
        assert out['hr_rel_l2'] <= 1e-3, out                 # north-star tolerance (fp16 path)
        assert out['hr_rel_max'] <= 5e-3, out
    assert out['hr_rel_l2'] <= 1.5 * out['emu_rel_l2'] + 1e-4, out
    assert out['flow_abs'] <= 2e-3 * max(1.0, out['flow_absmax_ref']), out
    return out


def check_step_bi2():
    g = np.load(os.path.join(G, 'step_bi2_20x24_g15.npz'))
    net, p = _net(12, 2, 'BI', 1.5)
    hr = net.step(rand(4, 1, 3, 20, 24).to(DEV), rand(5, 1, 3, 20, 24).to(DEV),
                  rand(6, 1, 3, 40, 48).to(DEV)).cpu().numpy()
    out = {'hr_rel_l2': rell2(hr, g['hr_curr']), 'hr_rel_max': relmax(hr, g['hr_curr'])}
    assert out['hr_rel_l2'] <= 1e-3 and out['hr_rel_max'] <= 5e-3, out
    return out


def check_infer_sequence_golden():
    g = np.load(os.path.join(G, 'infer_seq_bd4_16x24_g15.npz'))
    net, p = _net(13, 4, 'BD', 1.5)
    clip = O.make_clip(7, 4, 3, 16, 24)
    seq = net.infer_sequence(clip, torch.device(DEV))
    assert seq.shape == g['hr_seq'].shape and seq.dtype == np.uint8
    d = np.abs(seq.astype(np.int32) - g['hr_seq'].astype(np.int32))
    out = {'max_lsb': int(d.max()), 'frac_diff': float((d != 0).mean())}
    # fp16 path vs fp32 reference after 8-bit quantisation over a 4-frame recurrence: <= 1 LSB
    assert out['max_lsb'] <= 1 and out['frac_diff'] <= 0.02, out
    # eval-mode forward dispatch (reference FRNet.forward -> infer_sequence)
    seq2 = net(clip, torch.device(DEV))
    assert np.array_equal(seq, seq2), 'infer_sequence must be deterministic'
    return out


def check_forward_sequence_golden():
    g = np.load(os.path.join(G, 'fwd_seq_bd4_16x16_g15.npz'))
    net, p = _net(14, 4, 'BD', 1.5)
    net.train()
    with torch.no_grad():
        d = net(rand(8, 1, 3, 3, 16, 16).to(DEV))
    out = {}
    for k in ('hr_data', 'hr_flow', 'lr_prev', 'lr_curr', 'lr_flow'):
        assert tuple(d[k].shape) == g[k].shape, k
        out[k] = rell2(d[k].cpu().numpy(), g[k])
    assert out['hr_data'] <= 1e-3 and out['lr_flow'] <= 1e-3 and out['hr_flow'] <= 1e-3, out
    assert out['lr_prev'] == 0.0 and out['lr_curr'] == 0.0
    # under autograd the same call trains (autograd.SequenceFunction): same forward values
    d2 = net(rand(8, 1, 3, 3, 16, 16).to(DEV))
    assert d2['hr_data'].requires_grad and d2['lr_flow'].requires_grad
    out['train_vs_nograd_hr'] = rell2(d2['hr_data'].detach().cpu().numpy(), d['hr_data'].cpu().numpy())
    # (identical kernels give exactly 0; the fused-tail inference path differs from the per-layer training path by
    # fp32 summation order, which the 1.5x-gain recurrence amplifies to the level of the fp16 design error)
    assert out['train_vs_nograd_hr'] <= 1e-3, out
    return out


def _psnr_y(a_u8, b_u8):
    """Y-channel PSNR of two uint8 HWC frames (reference metric_calculator.py:228-244 math:
    BT.601 luma from RGB, MSE over the frame)."""
    def y(x):
        x = x.astype(np.float64)
        return 16.0 + (65.481 * x[..., 0] + 128.553 * x[..., 1] + 24.966 * x[..., 2]) / 255.0
    mse = np.mean((y(a_u8) - y(b_u8)) ** 2)
    return float(10 * np.log10(255.0 ** 2 / max(mse, 1e-12)))


def check_step_vs_oracle_fullsize(n=1, h=134, w=320, gain=1.0, frames=3):
    """BASELINE size 3x134x320 -> 3x536x1280: `frames`-step recurrence from zero state on a moving
    clip against the CPU oracle (fp32) per frame (drift), plus the PSNR of both uint8 outputs
    against a synthetic ground truth (the bicubic-upsampled clip): |delta PSNR| <= 0.01 dB."""
    net, p = _net(5, 4, 'BD', gain)
    clip = O.make_clip(9, frames, 3, h, w)
    gt = np.clip(K.bicubic_upsample(clip.numpy(), 4), 0, 1)
    lr_prev = torch.zeros(1, 3, h, w)
    hr_prev = torch.zeros(1, 3, 4 * h, 4 * w)
    g_lr_prev, g_hr_prev = lr_prev.to(DEV), hr_prev.to(DEV)
    out = {}
    for i in range(frames):
        lr_curr = clip[i:i + 1]
        ref = O.frnet_step(p, lr_curr, lr_prev, hr_prev, 4, 'BD')
        got = net.step(lr_curr.to(DEV), g_lr_prev, g_hr_prev)
        out[f'rel_l2_f{i}'] = rell2(got.cpu().numpy(), ref.numpy())
        lr_prev, hr_prev = lr_curr, ref
        g_lr_prev, g_hr_prev = lr_curr.to(DEV), got
    gt_u8 = K.float32_to_uint8(gt[-1]).transpose(1, 2, 0)
    ref_u8 = K.float32_to_uint8(ref[0].numpy()).transpose(1, 2, 0)
    got_u8 = ops.float_to_uint8_nhwc(got)[0].cpu().numpy()
    out['psnr_ref_db'] = _psnr_y(ref_u8, gt_u8)
    out['psnr_gpu_db'] = _psnr_y(got_u8, gt_u8)
    out['u8_max_lsb'] = int(np.abs(ref_u8.astype(np.int32) - got_u8.astype(np.int32)).max())
    for i in range(frames):
        assert out[f'rel_l2_f{i}'] <= 1e-3, out
    assert abs(out['psnr_ref_db'] - out['psnr_gpu_db']) <= 0.01, out
    assert out['u8_max_lsb'] <= 1, out
    return out


def check_batch_consistency(n=3, h=24, w=40):
    """step() on a batch of clips == step() on each clip alone (lock-stepped clips are
    independent): bit exact."""
    net, p = _net(15, 4, 'BD', 1.5, nb=2)
    a, b, c = rand(60, n, 3, h, w).to(DEV), rand(61, n, 3, h, w).to(DEV), rand(62, n, 3, 4 * h, 4 * w).to(DEV)
    full = net.step(a, b, c)
    for i in range(n):
        one = net.step(a[i:i + 1], b[i:i + 1], c[i:i + 1])
        assert torch.equal(one[0], full[i]), f'clip {i} differs between batch and solo'
    return {}


def check_engine_matches_eager(n=2, t=5, h=24, w=40):
    """CUDA-graph clip engine == eager step loop, bit exact on the uint8 output."""
    net, p = _net(16, 4, 'BD', 1.5, nb=3)
    clips = torch.stack([O.make_clip(70 + i, t, 3, h, w) for i in range(n)])       # n,t,c,h,w
    got = T.infer_clips(net, clips, torch.device(DEV))
    lr_prev = torch.zeros(n, 3, h, w, device=DEV)
    hr_prev = torch.zeros(n, 3, 4 * h, 4 * w, device=DEV)
    for i in range(t):
        lr_curr = clips[:, i].to(DEV)
        hr = net.step(lr_curr, lr_prev, hr_prev)
        ref_u8 = ops.float_to_uint8_nhwc(hr).cpu().numpy()
        assert np.array_equal(got[:, i], ref_u8), f'frame {i}'
        lr_prev, hr_prev = lr_curr, hr
    assert got.shape == (n, t, 4 * h, 4 * w, 3)
    return {}


# =============================================================================== size-independent properties
def check_properties_fullsize(n=2, h=134, w=320):
    """BASELINE-size properties that need no oracle run: (1) the fused warp kernel with zero flow
    is an exact space_to_depth of hr_prev (bit exact after the fp16 rounding), (2) conv linearity
    conv(a+b) - conv(b) = conv(a) - bias-free part, within fp16 rounding, (3) the transposed conv's
    four parity outputs interleave without overlap or holes (every output pixel written exactly
    once: a poisoned buffer comes back fully overwritten), (4) step() is deterministic."""
    out = {}
    hr = rand(80, n, 3, 4 * h, 4 * w)
    lr = rand(81, n, 3, h, w)
    zero = torch.zeros(n, 2, 4 * h, 4 * w)
    x = ops.warp_s2d_concat_hrflow(hr.to(DEV), zero.to(DEV), lr.to(DEV), 4)
    ref = torch.cat([lr, torch.from_numpy(K.space_to_depth(hr.numpy(), 4))], 1)
    assert torch.equal(from_nhwc(x, 51), f16(ref)), 'zero-flow warp must be an exact space_to_depth'
    # linearity on a 64->64 conv without activation
    wt = rand(82, 64, 64, 3, 3, lo=-0.05, hi=0.05)
    pc = ops.PackedConv(wt.to(DEV), torch.zeros(64, device=DEV), L.CONV_3X3, L.ACT_NONE)
    a = nhwc(rand(83, 1, 64, h, w, lo=-1, hi=1), 64)
    b = nhwc(rand(84, 1, 64, h, w, lo=-1, hi=1), 64)
    ya, yb, yab = pc(a).float(), pc(b).float(), pc((a.float() + b.float()).half()).float()
    lin = float((yab - ya - yb).abs().max() / yab.abs().max())
    out['linearity_rel'] = lin
    assert lin <= 4e-3, out           # three fp16 roundings of O(1) values
    # transposed conv coverage
    pt = ops.PackedConv(rand(85, 64, 64, 3, 3, lo=-0.05, hi=0.05).to(DEV), torch.ones(64, device=DEV),
                        L.CONVT_3X3_S2, L.ACT_RELU)
    y = torch.full((1, 2 * h, 2 * w, 64), float('nan'), dtype=torch.float16, device=DEV)
    pt(a, y=y)
    assert not bool(torch.isnan(y).any()), 'transposed conv left output pixels unwritten'
    # determinism of the whole step
    net, p = _net(17, 4, 'BD', 1.0, nb=2)
    args = (rand(86, n, 3, h, w).to(DEV), rand(87, n, 3, h, w).to(DEV), rand(88, n, 3, 4 * h, 4 * w).to(DEV))
    assert torch.equal(net.step(*args), net.step(*args)), 'step() must be deterministic'
    return out


def check_ragged_sizes():
    """Sizes that are not multiples of the 16x8 tile, of 8 (FNet reflect pad) or of the 14x6 thin-head
    tile: step() against the CPU oracle."""
    out = {}
    for (hh, ww) in ((17, 23), (9, 8), (31, 50)):
        net, p = _net(18, 4, 'BD', 1.5, nb=2)
        a, b, c = rand(90, 1, 3, hh, ww), rand(91, 1, 3, hh, ww), rand(92, 1, 3, 4 * hh, 4 * ww)
        got = net.step(a.to(DEV), b.to(DEV), c.to(DEV)).cpu().numpy()
        ref = O.frnet_step(p, a, b, c, 4, 'BD').numpy()
        out[f'{hh}x{ww}'] = rell2(got, ref)
        assert out[f'{hh}x{ww}'] <= 1e-3, out
    return out


def check_bi2_fullsize(h=268, w=640):
    """BASELINE config 5 shape (2x BI, LR 3x268x640): one step against the CPU oracle."""
    net, p = _net(19, 2, 'BI', 1.0)
    a, b, c = rand(93, 1, 3, h, w), rand(94, 1, 3, h, w), rand(95, 1, 3, 2 * h, 2 * w)
    got = net.step(a.to(DEV), b.to(DEV), c.to(DEV)).cpu().numpy()
    ref = O.frnet_step(p, a, b, c, 2, 'BI').numpy()
    out = {'rel_l2': rell2(got, ref), 'rel_max': relmax(got, ref)}
    assert out['rel_l2'] <= 1e-3, out
    return out


# =============================================================================== benchmark workloads
def _clip_recurrence_vs_oracle(net, p, host_clips, scale, degradation, tag):
    """infer_sequence (graph ClipEngine, pinned host clips -> host uint8) against the CPU oracle
    recurrence run on the same clips: per-frame max LSB / differing fraction (drift over time)."""
    n, t = host_clips.shape[:2]
    seq = net.infer_sequence(host_clips, torch.device(DEV))          # [n,t,H,W,c] uint8
    c, h, w = host_clips.shape[2:]
    assert seq.shape == (n, t, scale * h, scale * w, c) and seq.dtype == np.uint8
    lr_prev = torch.zeros(n, c, h, w)
    hr_prev = torch.zeros(n, c, scale * h, scale * w)
    out = {'max_lsb': 0, 'frac_diff_per_frame': [], 'max_lsb_per_frame': []}
    for i in range(t):
        lr_curr = host_clips[:, i].contiguous()
        hr_prev = O.frnet_step(p, lr_curr, lr_prev, hr_prev, scale, degradation)
        lr_prev = lr_curr
        ref_u8 = np.stack([K.float32_to_uint8(hr_prev[k].numpy()).transpose(1, 2, 0) for k in range(n)])
        d = np.abs(seq[:, i].astype(np.int32) - ref_u8.astype(np.int32))
        out['max_lsb_per_frame'].append(int(d.max()))
        out['frac_diff_per_frame'].append(round(float((d != 0).mean()), 5))
    out['max_lsb'] = max(out['max_lsb_per_frame'])
    out['frac_diff'] = float(np.mean(out['frac_diff_per_frame']))
    # fp16 storage vs the fp32 oracle after 8-bit quantisation: never more than 1 LSB on any frame
    # of any clip, and only where a value sits next to a rounding boundary
    assert out['max_lsb'] <= 1 and max(out['frac_diff_per_frame']) <= 0.05, (tag, out)
    return out


def check_bench_workload_parity(n=4, t=10):
    """EXACTLY the e2e workload of bench.py: 4 lock-stepped clips x 10 frames of 3x134x320 from pinned
    host memory through FRNet.infer_sequence (CUDA-graph ClipEngine, H2D/D2H rings) -> uint8
    [n,t,536,1280,3], compared per clip and per frame with the CPU oracle recurrence."""
    import bench
    net = T.FRNet(3, 3, 64, 10, 'BD', 4)
    p = bench.make_params()
    net.load_state_dict(p, strict=True)
    net = net.to(DEV).eval()
    host = bench.synthetic_clips(n, t, seed=100).pin_memory()
    return _clip_recurrence_vs_oracle(net, p, host, 4, 'BD', 'bench 4xBD')


def check_bi2_workload_parity(n=1, t=5, h=268, w=640):
    """BASELINE config 5 at full size: 2x BI, LR 3x268x640 -> 3x536x1280, a t-frame clip through the
    same engine path, against the CPU oracle recurrence."""
    net, p = _net(19, 2, 'BI', 1.0)
    host = torch.stack([O.make_clip(40 + k, t, 3, h, w) for k in range(n)]).pin_memory()
    return _clip_recurrence_vs_oracle(net, p, host, 2, 'BI', 'config5 2xBI')


# The generator section of the reference's FRVSR YAMLs (experiments_BD/FRVSR/FRVSR_VimeoTecoGAN_4xSR_2GPU/
# {train,test}.yml), the keys define_generator reads.
FRVSR_OPT = {'scale': 4, 'dataset': {'degradation': {'type': 'BD', 'sigma': 1.5}},
             'model': {'generator': {'name': 'FRNet', 'in_nc': 3, 'out_nc': 3, 'nf': 64, 'nb': 10}}}


def check_reference_callers_integration():
    """Drop-in through the steps of the reference's inference callers: define_generator from the FRVSR test
    YAML, prepare_inference_data (thwc -> tchw) and infer() with its reflect temporal padding of 5 frames
    (base_model.py:87-122,230-251, vsr_model.py:97-113), compared with the sequence the same callers produced
    with the reference generator on the CPU (tests/golden/callers_infer_bd4_18x28_g15.npz, every 14th
    element); then main.profile's FLOP / parameter report (main.py:210-244) and one step() on the generator's
    own dummy data."""
    g = np.load(os.path.join(G, 'callers_infer_bd4_18x28_g15.npz'))
    net = T.define_generator(FRVSR_OPT).to(DEV)
    assert isinstance(net, T.FRNet)
    net.load_state_dict(O.make_frnet_params(23, gain=1.5), strict=True)
    clip = O.make_clip(11, 9, 3, 18, 28)                       # tchw; 18x28 exercises the reflect flow pad
    lr_data = clip.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)   # thwc as the datasets deliver it
    n_pad = 5
    lr_data = torch.cat([lr_data[1:1 + n_pad].flip(0), lr_data], 0)
    net.eval()
    got_seq = net(lr_data, torch.device(DEV))[n_pad:]
    assert got_seq.shape == tuple(g['shape']) == (9, 72, 112, 3) and got_seq.dtype == np.uint8
    d = np.abs(got_seq.reshape(-1)[::14].astype(np.int32) - g['hr_seq_sample'].astype(np.int32))
    out = {'infer_max_lsb': int(d.max()), 'infer_frac_diff': float((d != 0).mean())}
    assert out['infer_max_lsb'] <= 1 and out['infer_frac_diff'] <= 0.03, out

    # main.profile: the FLOP / parameter report, and the step() it times on generate_dummy_data
    net = T.define_generator(FRVSR_OPT).to(DEV)
    gflops, params = net.profile((3, 134, 320), DEV)
    assert list(gflops) == list(params) == ['FNet', 'SRNet'], (gflops, params)
    report = [f'{gflops["FNet"]:.3f}', f'{gflops["SRNet"]:.3f}', f'{sum(gflops.values()):.3f}',
              f'{sum(params.values()) / 1e6:.3f}']
    assert report == ['10.511', '83.927', '94.438', '2.589'], report
    net.eval()
    with torch.no_grad():
        hr = net.step(*net.generate_dummy_data((3, 134, 320), DEV))
    assert tuple(hr.shape) == (1, 3, 536, 1280) and bool(torch.isfinite(hr).all()), hr.shape
    return out


def check_autograd_guards():
    """Ops must never silently cut the graph: inputs that require grad either get a backward kernel
    (backward_warp, upsample_func, space_to_depth, fnet, forward_sequence) or raise (step, SRNet.forward,
    gradients w.r.t. the LR frames)."""
    x = rand(1, 1, 3, 16, 16).to(DEV).requires_grad_(True)
    y = T.space_to_depth(x, 4)
    assert y.requires_grad
    y.sum().backward()
    assert torch.equal(x.grad, torch.ones_like(x))
    net, _ = _net(3, 4, 'BD', 1.0, nb=2)
    n_raised = 0
    for fn in (lambda: net.step(x[:, :, :8, :8], x[:, :, :8, :8].detach(), rand(2, 1, 3, 32, 32).to(DEV)),
               lambda: net.fnet(x, x.detach()),
               lambda: net.train().forward_sequence(x[None])):
        try:
            fn()
        except NotImplementedError:
            n_raised += 1
    assert n_raised == 3, n_raised
    return {'raised': n_raised}


# =============================================================================== backward kernels
def _conv_grads_ref(x, wt, kind, gy):
    """torch CPU autograd of conv3x3 / convT3x3s2 on fp16-rounded operands: (dx, dw)"""
    x = f16(x).clone().requires_grad_(True)
    w = f16(wt).clone().requires_grad_(True)
    if kind == L.CONV_3X3:
        y = F.conv2d(x, w, None, 1, 1)
    else:
        y = F.conv_transpose2d(x, w, None, 2, 1, output_padding=1)
    dx, dw = torch.autograd.grad(y, [x, w], f16(gy))
    return dx, dw


def check_conv_dgrad(impl='tcgen05', kind=None, cin=64, cout=64, h=20, w=24, n=2, cin_real=None, cout_real=None,
                     mask_act=None, residual=False, seed=300):
    """data gradient of a conv layer (PackedDgrad: flipped-tap conv / stride-2 conv over dz, optional
    + residual and * act'(mask)) against torch CPU autograd."""
    kind = L.CONV_3X3 if kind is None else kind
    cin_real, cout_real = cin_real or cin, cout_real or cout
    x = rand(seed, n, cin_real, h, w, lo=-1, hi=1)
    wshape = (cout_real, cin_real, 3, 3) if kind == L.CONV_3X3 else (cin_real, cout_real, 3, 3)
    wt = rand(seed + 1, *wshape, lo=-0.1, hi=0.1)
    up = 1 if kind == L.CONV_3X3 else 2
    gy = rand(seed + 2, n, cout_real, up * h, up * w, lo=-1, hi=1)
    dx_ref, _ = _conv_grads_ref(x, wt, kind, gy)
    fwd = ops.PackedConv(wt.to(DEV), torch.zeros(cout_real).to(DEV), kind, L.ACT_NONE)
    dg = ops.PackedDgrad(fwd, wt.to(DEV))
    res = rand(seed + 3, n, cin_real, h, w, lo=-1, hi=1) if residual else None
    msk = rand(seed + 4, n, cin_real, h, w, lo=-1, hi=1) if mask_act is not None else None
    got = dg(nhwc(gy, ops.pad64(cout_real)), residual=nhwc(res, dg.cout) if residual else None,
             mask=nhwc(msk, dg.cout) if msk is not None else None, mask_act=mask_act or L.ACT_NONE, impl=impl)
    torch.cuda.synchronize()
    ref = dx_ref
    if residual:
        ref = ref + f16(res)
    if msk is not None:
        slope = 0.0 if mask_act == L.ACT_RELU else 0.2
        ref = ref * torch.where(f16(msk) > 0, torch.ones_like(ref), torch.full_like(ref, slope))
    got_f = from_nhwc(got, cin_real)
    out = {'rel_l2': rell2(got_f.numpy(), ref.numpy()), 'rel_max': relmax(got_f.numpy(), ref.numpy())}
    assert out['rel_l2'] <= 2e-3, out                  # fp16 output rounding of a K<=2304 contraction
    if dg.cout > cin_real:
        assert float(got[..., cin_real:].abs().max()) == 0.0, 'pad channels of dx must be zero'
    return out


def check_wgrad(kind=None, cin=64, cout=64, h=20, w=24, n=2, cin_real=None, cout_real=None, seed=320, flags=(0,)):
    """weight gradient (tcgen05 GEMM over pixels, MN-major operands) against torch CPU autograd and the
    CUDA-core cross-check; `flags` = TG_WGRAD_FLAGS variants to report (only the first must pass)."""
    kind = L.CONV_3X3 if kind is None else kind
    cin_real, cout_real = cin_real or cin, cout_real or cout
    x = rand(seed, n, cin_real, h, w, lo=-1, hi=1)
    wshape = (cout_real, cin_real, 3, 3) if kind == L.CONV_3X3 else (cin_real, cout_real, 3, 3)
    wt = rand(seed + 1, *wshape, lo=-0.1, hi=0.1)
    up = 1 if kind == L.CONV_3X3 else 2
    gy = rand(seed + 2, n, cout_real, up * h, up * w, lo=-1, hi=1)
    _, dw_ref = _conv_grads_ref(x, wt, kind, gy)
    fwd = ops.PackedConv(wt.to(DEV), torch.zeros(cout_real).to(DEV), kind, L.ACT_NONE)
    xg, dzg = nhwc(x, fwd.cin), nhwc(gy, ops.pad64(cout_real))
    out = {}
    dw = torch.zeros(wshape, device=DEV)
    ops.wgrad(fwd, xg, dzg, dw, impl='simt')
    torch.cuda.synchronize()
    out['simt_rel_l2'] = rell2(dw.cpu().numpy(), dw_ref.numpy())
    assert out['simt_rel_l2'] <= 1e-4, out
    prev = os.environ.get('TG_WGRAD_FLAGS')
    try:
        for fl in flags:
            os.environ['TG_WGRAD_FLAGS'] = str(fl)
            dw = torch.zeros(wshape, device=DEV)
            sc = ops.GradScale(DEV).from_amax(gy.to(DEV))          # exercises the 1/scale epilogue too
            dzs = ops.grad_pack(gy.to(DEV), scale=sc, cpad=ops.pad64(cout_real))
            ops.wgrad(fwd, xg, dzs, dw, scale=sc)
            ops.wgrad(fwd, xg, dzs, dw, scale=sc)                   # accumulates: 2x
            torch.cuda.synchronize()
            got = dw.cpu().numpy() / 2
            out[f'tc_rel_l2_flags{fl}'] = rell2(got, dw_ref.numpy())
            if fl == flags[0] and out[f'tc_rel_l2_flags{fl}'] > 1e-3:      # bring-up aid: where is it wrong?
                r = dw_ref.numpy()
                out['per_tap_rel_l2'] = [round(rell2(got[:, :, t // 3, t % 3], r[:, :, t // 3, t % 3]), 4) for t in range(9)]
                out['transposed_rel_l2'] = rell2(got.transpose(1, 0, 2, 3), r) if got.shape[0] == got.shape[1] else None
                out['flipped_rel_l2'] = rell2(got[:, :, ::-1, ::-1], r)
                out['norm_ratio'] = float(np.linalg.norm(got) / np.linalg.norm(r))
    finally:
        if prev is None:
            os.environ.pop('TG_WGRAD_FLAGS', None)
        else:
            os.environ['TG_WGRAD_FLAGS'] = prev
    assert out[f'tc_rel_l2_flags{flags[0]}'] <= 1e-3, out
    db = torch.zeros(cout_real, device=DEV)
    ops.bias_grad(dzg, db)
    torch.cuda.synchronize()
    out['bias_rel_l2'] = rell2(db.cpu().numpy(), f16(gy).sum((0, 2, 3)).numpy())
    assert out['bias_rel_l2'] <= 1e-4, out
    # bias gradient fused into the wgrad launch (conv layers: the spare half of the last tap pair reads ones)
    db2, dw2 = torch.zeros(cout_real, device=DEV), torch.zeros(wshape, device=DEV)
    ops.wgrad(fwd, xg, dzg, dw2, db=db2)
    torch.cuda.synchronize()
    out['fused_bias_rel_l2'] = rell2(db2.cpu().numpy(), f16(gy).sum((0, 2, 3)).numpy())
    out['fused_dw_rel_l2'] = rell2(dw2.cpu().numpy(), dw_ref.numpy())
    assert out['fused_bias_rel_l2'] <= 1e-4 and out['fused_dw_rel_l2'] <= 1e-3, out
    return out


def check_backward_elementwise():
    """warp / upsample / pool / x2-bilinear / tanh-head derivatives against torch CPU autograd."""
    from oracle import frnet_torchref as R
    out = {}
    # ---- backward_warp: d/dx (scatter) and d/dflow (gather), incl. out-of-range flow (zero coordinate grad)
    x = rand(1, 2, 3, 21, 26).requires_grad_(True)
    fl = rand(2, 2, 2, 21, 26, lo=-4, hi=4)
    fl[0, :, 0, 0] = torch.tensor([-50.0, 50.0])
    fl = fl.requires_grad_(True)
    gy = rand(3, 2, 3, 21, 26, lo=-1, hi=1)
    y = R.warp(x, fl)
    gx_ref, gf_ref = torch.autograd.grad(y, [x, fl], gy)
    gx, gf = ops.backward_warp_bwd(x.detach().to(DEV), fl.detach().to(DEV), gy.to(DEV))
    out['warp_dx'] = rell2(gx.cpu().numpy(), gx_ref.numpy())
    out['warp_dflow'] = rell2(gf.cpu().numpy(), gf_ref.numpy())
    assert out['warp_dx'] <= 1e-4 and out['warp_dflow'] <= 2e-3, out      # closed-form grid vs the normalised round trip
    # through the public op + autograd
    xg, fg = x.detach().to(DEV).requires_grad_(True), fl.detach().to(DEV).requires_grad_(True)
    (T.backward_warp(xg, fg) * gy.to(DEV)).sum().backward()
    out['warp_public_dx'] = rell2(xg.grad.cpu().numpy(), gx_ref.numpy())
    assert out['warp_public_dx'] <= 1e-4 and rell2(fg.grad.cpu().numpy(), gf_ref.numpy()) <= 2e-3, out
    # ---- fused warp + s2d + concat backward
    for s_ in (4, 2):
        h, w = 9, 13
        hp = rand(10, 2, 3, s_ * h, s_ * w).requires_grad_(True)
        hf = rand(11, 2, 2, s_ * h, s_ * w, lo=-3, hi=3).requires_grad_(True)
        lrc = rand(12, 2, 3, h, w)
        cin = (s_ * s_ + 1) * 3
        g = rand(13, 2, cin, h, w, lo=-1, hi=1)
        xx = torch.cat([lrc, R.s2d(R.warp(hp, hf), s_)], 1)
        ghp_ref, ghf_ref = torch.autograd.grad(xx, [hp, hf], f16(g))
        d_hp = torch.zeros(2, 3, s_ * h, s_ * w, device=DEV)
        d_hf = torch.empty(2, 2, s_ * h, s_ * w, device=DEV)
        ops.warp_s2d_concat_bwd(nhwc(g), hp.detach().to(DEV), hf.detach().to(DEV), s_, d_hr_prev=d_hp, d_hr_flow=d_hf)
        out[f'fused_warp_s{s_}_dhr'] = rell2(d_hp.cpu().numpy(), ghp_ref.numpy())
        out[f'fused_warp_s{s_}_dflow'] = rell2(d_hf.cpu().numpy(), ghf_ref.numpy())
        assert out[f'fused_warp_s{s_}_dhr'] <= 1e-4 and out[f'fused_warp_s{s_}_dflow'] <= 2e-3, out
    # ---- upsample_func backward (bicubic x4, bicubic x2, bilinear x2, bilinear x4), ragged tile sizes
    for s_, deg, mode in ((4, 'BD', L.UP_BICUBIC), (2, 'BD', L.UP_BICUBIC), (2, 'BI', L.UP_BILINEAR), (4, 'BI', L.UP_BILINEAR)):
        xs = rand(20, 2, 2, 19, 37).requires_grad_(True)
        p = {'upsample_func.kernels': torch.from_numpy(K.bicubic_kernels(s_))}
        yy = R.upsample(p, xs, s_, deg)
        gg = rand(21, *yy.shape, lo=-1, hi=1)
        ref, = torch.autograd.grad(yy, [xs], gg)
        got = ops.upsample_bwd(gg.to(DEV), s_, mode, mul=1.0)
        out[f'upsample_bwd_{deg}{s_}'] = rell2(got.cpu().numpy(), ref.numpy())
        assert out[f'upsample_bwd_{deg}{s_}'] <= 1e-5, out
    xg = rand(22, 1, 2, 8, 8).to(DEV).requires_grad_(True)
    (T.BicubicUpsampler(4).to(DEV)(xg)).sum().backward()
    assert abs(float(xg.grad.sum()) - 16 * 2 * 64) <= 1e-2            # rows of the filter sum to 1
    # ---- maxpool backward fused with LeakyReLU' (odd sizes: last row / column gets no gradient)
    xm = rand(30, 2, 64, 9, 11, lo=-1, hi=1)
    pre = f16(xm).clone().requires_grad_(True)
    act = F.leaky_relu(pre, 0.2)
    pooled = F.max_pool2d(f16(act).detach().clone().requires_grad_(True), 2, 2)
    a2 = f16(act).detach().clone().requires_grad_(True)
    gp = rand(31, 2, 64, 4, 5, lo=-1, hi=1)
    ref_a, = torch.autograd.grad(F.max_pool2d(a2, 2, 2), [a2], f16(gp))
    ref = ref_a * torch.where(f16(act) > 0, torch.ones_like(ref_a), torch.full_like(ref_a, 0.2))
    got = ops.maxpool2x2_bwd(nhwc(f16(act).detach()), nhwc(gp), L.ACT_LRELU02)
    out['maxpool_bwd'] = rell2(from_nhwc(got, 64).numpy(), f16(ref.detach()).numpy())
    assert out['maxpool_bwd'] <= 1e-3, out
    # ---- x2 bilinear backward fused with LeakyReLU'
    m = rand(40, 2, 64, 7, 10, lo=-1, hi=1)
    mm = f16(m).clone().requires_grad_(True)
    up = F.interpolate(mm, scale_factor=2, mode='bilinear', align_corners=False)
    gu = rand(41, 2, 64, 14, 20, lo=-1, hi=1)
    ref_m, = torch.autograd.grad(up, [mm], f16(gu))
    ref = ref_m * torch.where(f16(m) > 0, torch.ones_like(ref_m), torch.full_like(ref_m, 0.2))
    got = ops.upsample2x_bwd(nhwc(gu), nhwc(m), L.ACT_LRELU02)
    out['upsample2x_bwd'] = rell2(from_nhwc(got, 64).numpy(), ref.numpy())
    assert out['upsample2x_bwd'] <= 1e-3, out
    # ---- flow head: d(24 tanh z) with the device-chosen loss scale
    z = rand(50, 2, 2, 8, 16, lo=-2, hi=2).requires_grad_(True)
    flow = torch.tanh(z) * 24
    gf = rand(51, 2, 2, 8, 16, lo=-1e-6, hi=1e-6)          # tiny, like a mean-reduced loss gradient
    ref, = torch.autograd.grad(flow, [z], gf)
    sc = ops.GradScale(DEV)
    dz = ops.flow_head_bwd(gf.to(DEV), flow.detach().to(DEV), sc)
    torch.cuda.synchronize()
    scale = float(sc.ws[0])
    out['flow_head_scale_log2'] = float(np.log2(scale))
    out['flow_head_bwd'] = rell2(from_nhwc(dz, 2).numpy() / scale, ref.numpy())
    assert out['flow_head_bwd'] <= 1e-3 and scale > 1e3, out
    return out


def _seq_loss(d, seed):
    rng = np.random.default_rng(seed)
    r1 = torch.from_numpy(rng.uniform(-1, 1, size=tuple(d['hr_data'].shape)).astype(np.float32)).to(d['hr_data'].device)
    r2 = torch.from_numpy(rng.uniform(-1, 1, size=tuple(d['lr_flow'].shape)).astype(np.float32)).to(d['hr_data'].device)
    return (d['hr_data'] * r1).sum() + 0.05 * (d['lr_flow'] * r2).sum()


def check_sequence_grads_golden(loss_mul=1.0):
    """The generator BACKWARD against (a) gradients the reference itself produced (loss.backward() through
    its FRNet.forward_sequence, oracle/gen_golden.py `grads`) and (b) the CPU precision model of this very
    design (oracle/gen_emu_grads.py: the same orchestration over tests/fake_ops.py with fp16 storage).
    Tolerances: (a) the fp16 FORWARD (weights + activations) moves the gradients of this random-projection
    loss by a few percent -- measured with the model: 3-5 % rel-L2, the fp16 gradient storage adds 1e-3
    (tests/test_training_orchestration_cpu.py) -- norms <= 5e-2, whole gradients <= 6e-2; (b) only the
    accumulation order differs: <= 1.5e-2.  loss_mul = 1e-7 ~ a mean-reduced loss: exercises the device-side
    loss scale."""
    g = np.load(os.path.join(G, 'fwd_seq_grads_bd4_16x16_nb2_g15.npz'))
    e = np.load(os.path.join(G, 'fwd_seq_grads_bd4_16x16_nb2_g15_fp16emu.npz'))
    net = T.FRNet(3, 3, 64, 2, 'BD', 4)
    net.load_state_dict(O.make_frnet_params(15, nb=2, scale=4, degradation='BD', gain=1.5), strict=True)
    net = net.to(DEV).train()
    d = net(rand(9, 1, 3, 3, 16, 16).to(DEV))
    loss = _seq_loss(d, 16)
    (loss * loss_mul).backward()
    torch.cuda.synchronize()
    out = {'loss_rel': abs(float(loss) - float(g['loss'])) / abs(float(g['loss']))}
    assert out['loss_rel'] <= 1e-3, out
    named = dict(net.named_parameters())
    names = [str(k) for k in g['names']]
    for tag, fx in (('ref', g), ('emu', e)):
        worst = 0.0
        for k, nrm in zip(names, fx['norms']):
            assert named[k].grad is not None, f'no gradient for {k}'
            err = abs(float(named[k].grad.norm()) / loss_mul - nrm) / max(nrm, 1e-12)
            if err > worst:
                worst, out[f'{tag}_worst_norm_param'] = err, k
        out[f'{tag}_worst_norm_rel'] = worst
        for k in fx.files:
            if k.startswith('g:'):
                out[f'{tag}_rel_l2 ' + k[2:]] = rell2(named[k[2:]].grad.cpu().numpy() / loss_mul, fx[k])
    assert out['ref_worst_norm_rel'] <= 5e-2 and out['emu_worst_norm_rel'] <= 3e-2, out
    assert all(v <= 6e-2 for kk, v in out.items() if kk.startswith('ref_rel_l2 ')), out
    assert all(v <= 4e-2 for kk, v in out.items() if kk.startswith('emu_rel_l2 ')), out
    return out


def check_fnet_autograd_public():
    """net_G.fnet(x1, x2) called bare under autograd (the ST-discriminator's call, tecogan_nets.py:420)
    against torch CPU autograd through the operator port."""
    from oracle import frnet_torchref as R
    p = O.make_frnet_params(31, nb=2, gain=1.5)
    net = T.FRNet(3, 3, 64, 2, 'BD', 4)
    net.load_state_dict(p, strict=True)
    net = net.to(DEV).train()
    x1, x2 = rand(60, 2, 3, 24, 40), rand(61, 2, 3, 24, 40)
    r = rand(62, 2, 2, 24, 40, lo=-1, hi=1)
    flow = net.fnet(x1.to(DEV), x2.to(DEV))
    (flow * r.to(DEV)).sum().backward()
    q = {k: v.clone().requires_grad_(k.startswith('fnet.')) for k, v in p.items()}
    ref_flow = R.fnet(q, x1, x2)
    names = [k for k in q if q[k].requires_grad]
    refs = torch.autograd.grad((ref_flow * r).sum(), [q[k] for k in names])
    named = dict(net.named_parameters())
    out = {'flow_rel_l2': rell2(flow.detach().cpu().numpy(), ref_flow.detach().numpy())}
    worst = 0.0
    for k, gr in zip(names, refs):
        e = rell2(named[k].grad.cpu().numpy(), gr.numpy())
        if e > worst:
            worst, out['worst_param'] = e, k
    out['worst_grad_rel_l2'] = worst
    assert out['flow_rel_l2'] <= 1e-3 and worst <= 6e-2, out      # fp16 forward, see check_sequence_grads_golden
    assert all(v.grad is None for k, v in named.items() if k.startswith('srnet.')), 'srnet must not receive gradients'
    return out


def _charbonnier(x, y, eps=1e-6):
    """CharbonnierLoss(reduction='mean') of the reference (models/optim/losses.py)"""
    d = x - y
    return torch.sqrt(d * d + eps).mean()


def bd_training_data(gt, scale=4, sigma=1.5):
    """prepare_training_data of the reference for BD (base_model.py:42-85): the LR clip blurred and subsampled
    on the device from the GT clip [n,t,c,H,W], and the GT without its border of int(3 sigma) pixels."""
    border = int(sigma * 3.0)
    n, t, c, gt_h, gt_w = gt.shape
    lr_h, lr_w = (gt_h - 2 * border) // scale, (gt_w - 2 * border) // scale
    gt = gt.view(n * t, c, gt_h, gt_w)
    lr_data = T.downsample_bd(gt, T.create_kernel(sigma).to(gt.device), scale, False).view(n, t, c, lr_h, lr_w)
    gt = gt[..., border:border + scale * lr_h, border:border + scale * lr_w]
    return lr_data, gt.reshape(n, t, c, scale * lr_h, scale * lr_w)


def frvsr_train_step(model, gt):
    """One iteration of the reference's FRVSR training loop (FRVSR train.yml; vsr_model.py:50-95), restated
    around `model` (the generator, or DistributedDataParallel wrapping it) for a GT clip on its device:
    Charbonnier pixel loss + Charbonnier warping loss through backward_warp, one Adam step (lr 1e-4, betas
    (0.9, 0.999)).  Returns the logged losses."""
    lr_data, gt = bd_training_data(gt)
    optim_G = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=0, betas=(0.9, 0.999))
    model.train()
    optim_G.zero_grad()
    d = model(lr_data)
    loss_pix = _charbonnier(d['hr_data'], gt)
    loss_warp = _charbonnier(T.backward_warp(d['lr_prev'], d['lr_flow']), d['lr_curr'])
    log = {'l_pix_G': loss_pix.item(), 'l_warp_G': loss_warp.item()}
    (loss_pix + loss_warp).backward()
    optim_G.step()
    return log


def ddp_wrap(net):
    """base_model.model_to_device for dist=True"""
    return torch.nn.parallel.DistributedDataParallel(torch.nn.SyncBatchNorm.convert_sync_batchnorm(net),
                                                     device_ids=[torch.cuda.current_device()])


def check_reference_training_integration(ddp=False):
    """One iteration of the reference's FRVSR training loop (frvsr_train_step) around define_generator's FRNet
    on the GPU, compared with the same iteration of the reference loop and generator on the CPU
    (tests/golden/train_frvsr_bd4_nb2_g15.npz): logged losses, gradient norms, two whole gradients and the
    direction of the Adam step.  ddp=True wraps the generator in DistributedDataParallel (NCCL, world size 1
    here; 2 ranks in tests/ddp_train_check.py) as base_model.model_to_device does."""
    import torch.distributed as dist
    g = np.load(os.path.join(G, 'train_frvsr_bd4_nb2_g15.npz'))
    p = O.make_frnet_params(41, nb=2, gain=1.5)
    gt = rand(70, 2, 4, 3, 72, 72)                            # [n,t,c,H+8,W+8] -> LR 16x16 after the BD border
    opt = {**FRVSR_OPT, 'model': {'generator': {**FRVSR_OPT['model']['generator'], 'nb': 2}}}
    net = T.define_generator(opt).to(DEV)
    net.load_state_dict(p, strict=True)
    if ddp and not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29533')
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        got_log = frvsr_train_step(ddp_wrap(net) if ddp else net, gt.to(DEV))
        torch.cuda.synchronize()
    finally:
        if ddp and dist.is_initialized():
            dist.destroy_process_group()
    got_g = {k: v.grad.detach().cpu() for k, v in net.named_parameters()}
    got_w = {k: v.detach().cpu() for k, v in net.named_parameters()}
    ref_log = dict(zip([str(k) for k in g['log_keys']], g['log_values']))
    assert sorted(ref_log) == sorted(got_log), (ref_log, got_log)
    out = {}
    for k in ref_log:
        out['log_' + k] = abs(got_log[k] - ref_log[k]) / max(abs(ref_log[k]), 1e-12)
        assert out['log_' + k] <= 2e-3, (k, got_log[k], ref_log[k])
    names = [str(k) for k in g['names']]
    assert sorted(names) == sorted(got_g)
    worst = 0.0
    for k, nrm in zip(names, g['norms']):
        e = abs(float(got_g[k].norm()) - nrm) / max(nrm, 1e-20)
        if e > worst:
            worst, out['worst_norm_param'] = e, k
    out['worst_grad_norm_rel'] = worst
    out['grad_rel_l2_conv_in'] = rell2(got_g['srnet.conv_in.0.weight'].numpy(), _stored(g, 'g:srnet.conv_in.0.weight'))
    out['grad_rel_l2_fnet_e1'] = rell2(got_g['fnet.encoder1.0.weight'].numpy(), _stored(g, 'g:fnet.encoder1.0.weight'))
    assert worst <= 5e-2 and out['grad_rel_l2_conv_in'] <= 6e-2 and out['grad_rel_l2_fnet_e1'] <= 6e-2, out
    # one Adam step moved every weight by ~lr (1e-4) in both runs, in the same direction almost everywhere:
    # compared at sampled positions where the reference gradient is large (Adam's first step = lr*sign(g))
    agree, off = [], 0
    for k, cnt in zip(names, g['adam_count']):
        idx = torch.from_numpy(g['adam_idx'][off:off + cnt].astype(np.int64))
        d_got = (got_w[k] - p[k]).reshape(-1)[idx]
        agree.append(float((torch.sign(d_got).numpy() == g['adam_sign'][off:off + cnt]).mean()))
        off += cnt
    out['adam_step_sign_agreement_min'] = min(agree)
    assert min(agree) >= 0.95, out
    return out


def _stored(g, key):
    """a fixture array, rescaled when it was stored as fp16 relative to its largest magnitude"""
    x = g[key].astype(np.float64)
    return x * float(g[key + '_scale']) if key + '_scale' in g.files else x


def check_reference_gan_training_integration():
    """BASELINE config 3 in miniature: one iteration of the reference's TecoGAN training loop (VSRGANModel.train:
    adaptive ST-discriminator, VGG perceptual loss, ping-pong, warping and GAN losses; vsrgan_model.py:98-286)
    with nb=2, 4-frame clips and 32x32 GT crops, replayed at the generator's boundary.  The reference's own
    iteration on the CPU (tests/golden/train_tecogan_bd4_nb2_t4_32x32.npz) gives d loss_G / d hr_data and
    d loss_G / d lr_flow -- the only generator outputs the loss reaches, as the discriminator detaches the
    flows it takes from hr_flow -- together with its logged losses and generator gradients.  Here
    define_generator's FRNet runs forward_sequence on the same ping-pong clip on the GPU; the losses that need
    neither discriminator nor VGG are recomputed from its outputs, and the two cotangents are propagated
    through its backward: logged losses, every gradient norm and the conv_in / conv_out gradients."""
    g = np.load(os.path.join(G, 'train_tecogan_bd4_nb2_t4_32x32.npz'))
    t, crop, border = 4, 32, int(1.5 * 3.0)
    opt = {**FRVSR_OPT, 'model': {'generator': {**FRVSR_OPT['model']['generator'], 'nb': 2}}}
    net = T.define_generator(opt).to(DEV)
    assert isinstance(net, T.FRNet)
    net.load_state_dict(O.make_frnet_params(43, nb=2, gain=1.0), strict=True)
    lr_data, gt = bd_training_data(rand(80, 1, t, 3, crop + 2 * border, crop + 2 * border).to(DEV))
    lr_data = torch.cat([lr_data, lr_data.flip(1)[:, 1:]], 1)      # ping-pong: (0,..,t-1,..,0)
    gt = torch.cat([gt, gt.flip(1)[:, 1:]], 1)
    net.train()
    d = net(lr_data)
    with torch.no_grad():
        got_log = {'l_pix_G': _charbonnier(d['hr_data'], gt).item(),
                   'l_warp_G': _charbonnier(T.backward_warp(d['lr_prev'], d['lr_flow']), d['lr_curr']).item(),
                   'l_pp_G': 0.5 * _charbonnier(d['hr_data'][:, :t - 1], d['hr_data'][:, t:].flip(1)).item()}
    cot_hr = torch.from_numpy(_stored(g, 'cot_hr_data').astype(np.float32)).to(DEV)
    cot_flow = torch.from_numpy(g['cot_lr_flow']).to(DEV)
    assert tuple(d['hr_data'].shape) == tuple(cot_hr.shape) and tuple(d['lr_flow'].shape) == tuple(cot_flow.shape)
    torch.autograd.backward([d['hr_data'], d['lr_flow']], [cot_hr, cot_flow])
    torch.cuda.synchronize()
    ref_log = dict(zip([str(k) for k in g['log_keys']], g['log_values']))
    out = {}
    for k, v in got_log.items():
        out['log_' + k] = abs(v - ref_log[k]) / max(abs(ref_log[k]), 1e-6)
        assert out['log_' + k] <= 5e-3, (k, v, ref_log[k], out)
    named = dict(net.named_parameters())
    names = [str(k) for k in g['names']]
    assert sorted(names) == sorted(named)
    worst = 0.0
    for k, nrm in zip(names, g['norms']):
        e = abs(float(named[k].grad.norm()) - nrm) / max(nrm, 1e-20)
        if e > worst:
            worst, out['worst_norm_param'] = e, k
    out['worst_grad_norm_rel'] = worst
    out['grad_rel_l2_conv_out'] = rell2(named['srnet.conv_out.weight'].grad.cpu().numpy(), _stored(g, 'g:srnet.conv_out.weight'))
    out['grad_rel_l2_conv_in'] = rell2(named['srnet.conv_in.0.weight'].grad.cpu().numpy(), _stored(g, 'g:srnet.conv_in.0.weight'))
    assert worst <= 6e-2 and out['grad_rel_l2_conv_out'] <= 3e-2 and out['grad_rel_l2_conv_in'] <= 6e-2, out
    return out


def check_st_discriminator_input():
    """tg_st_disc_input (f3) against the reference's own SpatioTemporalDiscriminator.forward_sequence: its
    input tensor captured at conv_in for use_pp_crit = True (flows taken from the generator's hr_flow) and
    the gradient w.r.t. the frames (tests/golden/st_disc_input_bd4_n2t7_32x32.npz: norms and every 26th
    element)."""
    g = np.load(os.path.join(G, 'st_disc_input_bd4_n2t7_32x32.npz'))
    n, T_, c, s_, h = 2, 7, 3, 4, 8
    H = s_ * h
    data = rand(90, n, T_, c, H, H)
    bi = rand(91, n, T_, c, H, H)
    hr_flow = rand(93, n, T_ - 1, 2, H, H, lo=-3, hi=3)
    # the same flows merge the reference builds (tecogan_nets.py:408-431)
    t = T_ // 3 * 3
    bw = hr_flow[:, 0:t:3]
    fw = hr_flow.flip(1)[:, 1:t:3]
    merge = torch.stack([bw, torch.zeros_like(bw), fw], dim=2).view(n * t, 2, H, H)
    dg = data.to(DEV).requires_grad_(True)
    got = T.st_discriminator_input(dg, bi.to(DEV), merge.to(DEV), H, 0.75)
    assert tuple(got.shape) == tuple(g['x_shape']) == (n * t // 3, 27, H, H)
    gw = rand(94, *got.shape, lo=-1, hi=1)
    (got * gw.to(DEV)).sum().backward()
    x = got.detach().cpu().numpy()
    gx = dg.grad.cpu().numpy()
    out = {'value_max_abs': float(np.abs(x.reshape(-1)[::26] - g['x_sample']).max()),
           'value_norm_rel': abs(float(np.linalg.norm(x)) - float(g['x_norm'])) / float(g['x_norm']),
           'grad_rel_l2': rell2(gx.reshape(-1)[::26], g['grad_sample']),
           'grad_norm_rel': abs(float(np.linalg.norm(gx)) - float(g['grad_norm'])) / float(g['grad_norm'])}
    assert out['value_max_abs'] <= 1e-4 and out['value_norm_rel'] <= 1e-4, out
    assert out['grad_rel_l2'] <= 1e-4 and out['grad_norm_rel'] <= 1e-4, out
    return out


def check_conv_pool_epilogue(cin=64, cout=64, h=37, w=45, n=2, a_mode=None, seed=500):
    """TG_EPI_NHWC_F16_POOL2 (MaxPool2d(2,2) folded into the conv epilogue by warp shuffles) must equal the
    separate maxpool kernel applied to the plain conv output bit for bit (odd sizes: floor pooling)."""
    x = rand(seed, n, cin, h, w, lo=-1, hi=1)
    wt = rand(seed + 1, cout, cin, 3, 3, lo=-0.1, hi=0.1)
    b = rand(seed + 2, cout, lo=-0.2, hi=0.2)
    pc = ops.PackedConv(wt.to(DEV), b.to(DEV), L.CONV_3X3, L.ACT_LRELU02)
    xg = nhwc(x, ops.pad64(cin))
    ref = ops.maxpool2x2(pc(xg, a_mode=a_mode))
    got = torch.full((n, h // 2, w // 2, pc.cout), float('nan'), dtype=torch.float16, device=DEV)
    pc(xg, y=got, a_mode=a_mode, pool=True)
    torch.cuda.synchronize()
    assert not torch.isnan(got).any(), 'pooled epilogue left pixels unwritten'
    assert torch.equal(got, ref), float((got.float() - ref.float()).abs().max())
    return {'bit_exact': True, 'shape': list(got.shape)}


def check_fused_tail(scale=4, n=2, h=20, w=26, with_lr=True, seed=400, accumulate=False):
    """tg_convT_convout_tcgen05 (last transposed conv + ReLU + conv_out + upsample_func(lr) + uint8 in one
    launch) against the same four stages run as separate kernels, and against torch CPU fp32."""
    mid_h, mid_w = h, w                               # input of the last transposed conv
    lr_scale = scale
    x = rand(seed, n, 64, mid_h, mid_w, lo=-1, hi=1)
    wt = rand(seed + 1, 64, 64, 3, 3, lo=-0.08, hi=0.08)
    bu = rand(seed + 2, 64, lo=-0.2, hi=0.2)
    wo = rand(seed + 3, 3, 64, 3, 3, lo=-0.08, hi=0.08)
    bo = rand(seed + 4, 3, lo=-0.2, hi=0.2)
    assert (2 * mid_h) % lr_scale == 0 and (2 * mid_w) % lr_scale == 0
    lr = rand(seed + 5, n, 3, 2 * mid_h // lr_scale, 2 * mid_w // lr_scale)
    up = ops.PackedConv(wt.to(DEV), bu.to(DEV), L.CONVT_3X3_S2, L.ACT_RELU)
    oc = ops.PackedConv(wo.to(DEV), bo.to(DEV), L.CONV_3X3, L.ACT_NONE, L.EPI_OUT_NCHW_F32)
    mode = L.UP_BICUBIC if scale == 4 else L.UP_BILINEAR
    xg = nhwc(x)
    # separate kernels
    ref = oc(up(xg))
    if with_lr:
        ops.upsample(lr.to(DEV), lr_scale, mode, y=ref, accumulate=True)
    ref_u8 = ops.float_to_uint8_nhwc(ref)
    # fused (output buffers poisoned first: every pixel must be written exactly once)
    got = torch.full((n, 3, 2 * mid_h, 2 * mid_w), float('nan'), device=DEV)
    got_u8 = torch.full((n, 2 * mid_h, 2 * mid_w, 3), 77, dtype=torch.uint8, device=DEV)
    if accumulate:       # y pre-filled with the residual, the kernel adds conv + bias onto it (no uint8 inside)
        ops.upsample(lr.to(DEV), lr_scale, mode, y=got)
        ops.fused_tail(up, oc, xg, None, lr_scale, mode, y=got, accumulate=True)
        ops.float_to_uint8_nhwc(got, got_u8)
    else:
        ops.fused_tail(up, oc, xg, lr.to(DEV) if with_lr else None, lr_scale, mode, y=got, y_u8=got_u8)
    torch.cuda.synchronize()
    assert not torch.isnan(got).any(), 'fused tail left output pixels unwritten'
    out = {'vs_separate_max_abs': float((got - ref).abs().max()), 'vs_separate_rel_l2': rell2(got.cpu().numpy(), ref.cpu().numpy())}
    du8 = (got_u8.int() - ref_u8.int()).abs()
    out['u8_max_lsb'] = int(du8.max())
    out['u8_frac_diff'] = float((du8 != 0).float().mean())
    # torch CPU fp32 on the fp16-rounded operands
    t = F.relu(F.conv_transpose2d(f16(x), f16(wt), bu, 2, 1, output_padding=1))
    tr = F.conv2d(f16(t), f16(wo), bo, 1, 1)
    if with_lr:
        tr = tr + torch.from_numpy(K.bicubic_upsample(lr.numpy(), lr_scale) if scale == 4 else K.bilinear_upsample(lr.numpy(), lr_scale))
    out['vs_torch_rel_l2'] = rell2(got.cpu().numpy(), tr.numpy())
    assert out['vs_separate_max_abs'] <= 2e-5 and out['u8_max_lsb'] <= 1 and out['u8_frac_diff'] <= 1e-4, out
    assert out['vs_torch_rel_l2'] <= 1e-3, out
    return out


# =============================================================================== backward kernels at training shapes
# The unit checks above give every persistent CTA of the backward kernels at most one 16x8 tile.  The checks
# below run them at the shapes of training (10 residual blocks, 19-frame ping-pong clips, 64x64 LR crops), where
# a CTA walks many tiles: the smem stage ring wraps, the phase bit flips, later tiles accumulate onto earlier
# ones, and the fused bias gradient reads its ones block from every stage.  The references are exact: every
# product of two fp16 values is exact in fp64, so a float64 reference on the very fp16 operands handed to the
# kernel leaves only the kernel's fp32 summation error, and one dropped or doubled tile out of T moves the
# result by ~1/sqrt(T) -- orders of magnitude above the bars.

WG_STAGES_SMEM = 232448          # tg_wgrad_tcgen05: dynamic smem per CTA


def _wgrad_plan(kind, cin, cout, n, h, w, max_ctas=0, with_db=False, sms=148):
    """Tile count, CTAs per (ci chunk, co chunk) pair, tiles per CTA and smem stage count, as tg_wgrad_tcgen05
    computes them on the host (cin / cout = stored channel counts)."""
    tiles = -(-w // 8) * -(-h // 16) * n
    pairs = (cin // 64) * (cout // 64)
    budget = max_ctas if 0 < max_ctas < sms else sms
    budget = max(budget, pairs)
    cpp = min(budget // pairs, tiles)
    conv = kind == L.CONV_3X3
    box_w, box_h = (10, 18) if conv else (9, 17)
    stage = (box_w * box_h * 128 + 1023) // 1024 * 1024 + (1 if conv else 4) * 16384
    ones = 3072 if (conv and with_db) else 0
    stages = min((WG_STAGES_SMEM - 2048 - ones) // stage, 6)
    return {'tiles': tiles, 'pairs': pairs, 'ctas_per_pair': cpp, 'tiles_per_cta': tiles / cpp,
            'max_tiles_per_cta': -(-tiles // cpp), 'stages': stages}


def _dgrad_plan(cout, n, h, w, max_ctas=0, sms=148):
    """Tiles per CTA of tg_conv_tcgen05 for a data gradient (h, w = the size of dx, cout = its stored channels):
    output channels above 64 split the tiles over cout/64 CTA groups."""
    n_split = cout // 64 if cout > 64 else 1
    tiles = -(-w // 8) * -(-h // 16) * n * n_split
    grid = max_ctas if max_ctas > 0 else sms
    grid = min(grid, tiles)
    grid -= grid % n_split
    grid = max(grid, n_split)
    return {'tiles': tiles, 'grid': grid, 'tiles_per_cta': tiles / grid, 'max_tiles_per_cta': -(-tiles // grid)}


def _host_scale(amax, target=256.0):
    """2^clamp(floor(log2(target / amax)), -24, 24): the loss scale scale_from_amax_kernel picks"""
    e = int(np.floor(np.log2(target / amax)))
    return float(2.0 ** max(-24, min(24, e)))


def _conv_bwd64(g, x, w, kind, weight_grad):
    """d/dW (weight_grad) or d/dx of conv3x3 (pad 1) / convT3x3s2 (pad 1, output_padding 1) in float64 for the output
    gradient g, through the kernel torch autograd runs (aten.convolution_backward); only the shapes of the
    operand not differentiated against are used."""
    conv = kind == L.CONV_3X3
    st = [1, 1] if conv else [2, 2]
    op = [0, 0] if conv else [1, 1]
    mask = [False, True, False] if weight_grad else [True, False, False]
    r = torch.ops.aten.convolution_backward(g, x, w, None, st, [1, 1], [1, 1], not conv, op, 1, mask)
    return r[1] if weight_grad else r[0]


def _wgrad_ref64(x16, dz16, kind, inv_scale, chunk=4):
    """dW, db (float64) of a conv3x3 / convT3x3s2 layer from the fp16 operands handed to the kernel: x16 = its
    input [n,cin_real,h,w], dz16 = the loss-scaled gradient of its output [n,cout_real,oh,ow]; times 1/scale."""
    n, ci = x16.shape[:2]
    co = dz16.shape[1]
    wshape = (co, ci, 3, 3) if kind == L.CONV_3X3 else (ci, co, 3, 3)
    dw = torch.zeros(wshape, dtype=torch.float64)
    with torch.no_grad():
        for i in range(0, n, chunk):                       # chunks bound the im2col buffers
            dw += _conv_bwd64(dz16[i:i + chunk].double(), x16[i:i + chunk].double(), dw, kind, True)
        db = dz16.double().sum((0, 2, 3))
    return dw * inv_scale, db * inv_scale


def _dact64(mask16, mask_act):
    slope = 0.0 if mask_act == L.ACT_RELU else 0.2
    m = mask16.double()
    return torch.where(m > 0, torch.ones_like(m), torch.full_like(m, slope))


def _dgrad_ref64(dz16, w, kind, residual16=None, mask16=None, mask_act=None, chunk=4):
    """float64 data gradient of a conv layer, (d/dx [+ residual]) * act'(mask), from the fp16 operands handed to
    the kernel: dz16 [n,cout_real,oh,ow], w = the layer weight (the kernel packs it as fp16), residual16 /
    mask16 [n,cin_real,h,w]."""
    w64 = f16(w).double()
    up = 1 if kind == L.CONV_3X3 else 2
    n, _, oh, ow = dz16.shape
    cin = w.shape[1] if kind == L.CONV_3X3 else w.shape[0]
    with torch.no_grad():
        y = torch.cat([_conv_bwd64(dz16[i:i + chunk].double(),
                                   torch.empty(min(chunk, n - i), cin, oh // up, ow // up, dtype=torch.float64),
                                   w64, kind, False) for i in range(0, n, chunk)])
        if residual16 is not None:
            y = y + residual16.double()
        if mask16 is not None:
            y = y * _dact64(mask16, mask_act)
    return y


def _tile_mask(shape, img, ty, tx, up):
    """[n,1,oh,ow] float64 mask of one 16x8 pixel tile of image img (up = 2: the tile seen at the convT output)"""
    m = torch.zeros(shape[0], 1, shape[2], shape[3], dtype=torch.float64)
    m[img, :, up * 16 * ty:up * 16 * (ty + 1), up * 8 * tx:up * 8 * (tx + 1)] = 1.0
    return m


def _dgrad_metric(got, ref):
    """max over elements of |got - ref| / (1 fp16 ulp(|ref|) + 1e-5 max|ref|): <= 1 is the bar"""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float64)
    tol = ulp + 1e-5 * np.abs(ref).max()
    return float((np.abs(got - ref) / tol).max())


# wgrad cases: (kind, cin_real, cout_real, n, h, w) with h, w = the layer INPUT size; runs = max_ctas values
WGRAD_CASES = {
    # SRNet residual conv over 2 clips x 19 frames of 64x64: ~8 tiles per CTA, the 5-stage ring wraps
    'srnet_conv': dict(kind=L.CONV_3X3, cin_real=64, cout_real=64, n=38, h=64, w=64, runs=(0,), seed=600),
    # conv_out 64->3 over 38 HR frames of 256x256: ~131 tiles per CTA
    'conv_out': dict(kind=L.CONV_3X3, cin_real=64, cout_real=3, n=38, h=256, w=256, runs=(0,), seed=610),
    # the two transposed convs (dz at 2x): the 2-stage ring wraps many times
    'convT_64': dict(kind=L.CONVT_3X3_S2, cin_real=64, cout_real=64, n=38, h=64, w=64, runs=(0,), seed=620),
    'convT_128': dict(kind=L.CONVT_3X3_S2, cin_real=64, cout_real=64, n=38, h=128, w=128, runs=(0,), seed=630),
    # FNet on 36 frame pairs at LR 64x64; 2-4 tiles per CTA on the default grid, many at max_ctas=8
    'fnet_enc1_0': dict(kind=L.CONV_3X3, cin_real=6, cout_real=32, n=36, h=64, w=64, runs=(0, 8), seed=640),
    'fnet_dec1_0': dict(kind=L.CONV_3X3, cin_real=128, cout_real=256, n=36, h=8, w=8, runs=(0, 8), seed=650),
    'fnet_dec1_2': dict(kind=L.CONV_3X3, cin_real=256, cout_real=256, n=36, h=8, w=8, runs=(0, 8), seed=660),
    'fnet_dec2_0': dict(kind=L.CONV_3X3, cin_real=256, cout_real=128, n=36, h=16, w=16, runs=(0, 8), seed=670),
    'fnet_flow_2': dict(kind=L.CONV_3X3, cin_real=32, cout_real=2, n=36, h=64, w=64, runs=(0, 8), seed=680),
    # ragged 37x29, few CTAs: the ring wraps cheaply and the bias descriptor visits every stage index
    'max_ctas_sweep': dict(kind=L.CONV_3X3, cin_real=64, cout_real=64, n=5, h=37, w=29, runs=(1, 2, 3, 5, 7), seed=690),
}

WG_BAR_L2, WG_BAR_MAX, WG_BAR_DB = 1e-4, 1e-3, 1e-4


def wgrad_case_operands(case):
    """Host operands of a wgrad case: x16 [n,cin_real,h,w] fp16, the fp32 gradient gy of the layer output (tiny,
    like a mean-reduced loss: amax ~1e-8, so the 2^24 cap of the loss scale is active), the scale the device will
    pick, and dz16 = fp16(gy * scale) as grad_pack stores it."""
    c = WGRAD_CASES[case]
    up = 1 if c['kind'] == L.CONV_3X3 else 2
    x16 = rand(c['seed'], c['n'], c['cin_real'], c['h'], c['w'], lo=-1, hi=1).half()
    gy = rand(c['seed'] + 1, c['n'], c['cout_real'], up * c['h'], up * c['w'], lo=-1e-8, hi=1e-8)
    scale = _host_scale(float(gy.abs().max()))
    return x16, gy, scale, (gy * scale).half()


def wgrad_detection_power(case, x16=None, dz16=None, scale=None, ref=None):
    """rel-L2 of the exact reference with the contribution of one 16x8 tile (the last tile of the last image)
    removed, against the full reference: what a kernel that dropped that tile would score, for dW and db."""
    c = WGRAD_CASES[case]
    if x16 is None:
        x16, _, scale, dz16 = wgrad_case_operands(case)
    if ref is None:
        ref = _wgrad_ref64(x16, dz16, c['kind'], 1.0 / scale)
    up = 1 if c['kind'] == L.CONV_3X3 else 2
    n = c['n']
    m = _tile_mask(dz16.shape, 0, -(-c['h'] // 16) - 1, -(-c['w'] // 8) - 1, up)[:1]
    part = _wgrad_ref64(x16[n - 1:n], (dz16[n - 1:n].double() * m).half(), c['kind'], 1.0 / scale)
    return {'dw_rel_l2': rell2((ref[0] - part[0]).numpy(), ref[0].numpy()),
            'db_rel_l2': rell2((ref[1] - part[1]).numpy(), ref[1].numpy())}


def check_wgrad_multitile(case):
    """tg_wgrad_tcgen05 at a training shape against the exact float64 reference (_wgrad_ref64) on the operands
    handed to the kernel: the scale the device chose and the dz grad_pack stored are first checked to be the
    host's, bit for bit.  dw / db are pre-filled (the kernel accumulates).  Bars: dW rel-L2 <= 1e-4 and
    per-element |err| <= 1e-3 max|ref|, fused db rel-L2 <= 1e-4 (fp32 accumulation of exact fp16 products: the
    only error is the fp32 summation; measured on a B200, 1.5e-6 at 8 tiles per CTA and 2.2e-5 at 144, as the
    running sums of a CTA grow).  The CUDA-core kernel is reported as a second opinion."""
    c = WGRAD_CASES[case]
    kind, n, h, w = c['kind'], c['n'], c['h'], c['w']
    up = 1 if kind == L.CONV_3X3 else 2
    x16, gy, scale, dz16 = wgrad_case_operands(case)
    ref_dw, ref_db = ref = _wgrad_ref64(x16, dz16, kind, 1.0 / scale)
    det = wgrad_detection_power(case, x16, dz16, scale, ref)
    out = {'detect_drop_tile_dw': det['dw_rel_l2'], 'detect_drop_tile_db': det['db_rel_l2'], 'scale_log2': float(np.log2(scale))}
    assert det['dw_rel_l2'] > 10 * WG_BAR_L2 and det['db_rel_l2'] > 10 * WG_BAR_DB, out
    wshape = tuple(ref_dw.shape)
    fwd = ops.PackedConv(torch.zeros(wshape, device=DEV), torch.zeros(c['cout_real'], device=DEV), kind, L.ACT_NONE)
    cpad = ops.pad64(c['cout_real'])
    sc = ops.GradScale(DEV).from_amax(gy.to(DEV))
    dzs = ops.grad_pack(gy.to(DEV), scale=sc, cpad=cpad)
    xg = nhwc(x16.float(), fwd.cin)
    torch.cuda.synchronize()
    assert float(sc.ws[0]) == scale and float(sc.ws[1]) == 1.0 / scale, (float(sc.ws[0]), scale)
    host_dz = torch.zeros(n, up * h, up * w, cpad, dtype=torch.float16)
    host_dz[..., :c['cout_real']] = dz16.permute(0, 2, 3, 1)
    assert torch.equal(dzs.cpu(), host_dz), 'grad_pack output differs from fp16(g * scale)'
    del host_dz
    rmax = float(ref_dw.abs().max())
    pre_dw = rand(c['seed'] + 2, *wshape, lo=-1, hi=1) * rmax
    pre_db = rand(c['seed'] + 3, c['cout_real'], lo=-1, hi=1) * float(ref_db.abs().max())
    first = None
    for mc in c['runs']:
        plan = _wgrad_plan(kind, fwd.cin, cpad, n, h, w, mc, with_db=kind == L.CONV_3X3, sms=ops.sm_count())
        dw, db = pre_dw.to(DEV), pre_db.to(DEV)
        ops.wgrad(fwd, xg, dzs, dw, scale=sc, db=db, max_ctas=mc)
        torch.cuda.synchronize()
        got_dw = dw.cpu().double() - pre_dw.double()
        got_db = db.cpu().double() - pre_db.double()
        r = {'tiles_per_cta': round(plan['tiles_per_cta'], 2), 'stages': plan['stages'],
             'dw_rel_l2': rell2(got_dw.numpy(), ref_dw.numpy()),
             'dw_rel_max': float((got_dw - ref_dw).abs().max()) / rmax,
             'db_rel_l2': rell2(got_db.numpy(), ref_db.numpy())}
        if first is None:
            first = (got_dw, got_db)
        elif case == 'max_ctas_sweep':   # grids of 2..7 CTAs: only the order of the fp32 sums and atomics differs
            r['vs_first_run_rel_l2'] = max(rell2(got_dw.numpy(), first[0].numpy()), rell2(got_db.numpy(), first[1].numpy()))
            assert r['vs_first_run_rel_l2'] <= 1e-5, (case, mc, r)
        out[f'max_ctas{mc}'] = r
        assert r['dw_rel_l2'] <= WG_BAR_L2 and r['dw_rel_max'] <= WG_BAR_MAX and r['db_rel_l2'] <= WG_BAR_DB, (case, mc, r)
        if case == 'max_ctas_sweep':
            assert plan['ctas_per_pair'] == mc, (case, mc, plan)
        if mc == 0 and case.startswith('fnet_'):
            assert plan['tiles_per_cta'] >= 2, (case, mc, plan)                 # FNet's few tiles on the default grid
        else:
            assert plan['tiles_per_cta'] > plan['stages'], (case, mc, plan)     # the ring wraps on every CTA
    # the CUDA-core kernel on the same operands (reported)
    dw = torch.zeros(wshape, device=DEV)
    ops.wgrad(fwd, xg, dzs, dw, scale=sc, impl='simt')
    torch.cuda.synchronize()
    out['simt_dw_rel_l2'] = rell2(dw.cpu().numpy(), ref_dw.numpy())
    return out


# dgrad cases: the forward layer (kind, cin_real, cout_real), n images of h x w (= the size of dx), the
# derivative mask, a residual; every case runs on the default grid and on the few CTAs of `runs`
DGRAD_CASES = {
    # SRNet residual conv, halo BWD instance with ReLU' mask and the skip gradient
    'srnet_halo': dict(kind=L.CONV_3X3, cin_real=64, cout_real=64, n=8, h=64, w=64, act=L.ACT_RELU, residual=True,
                       runs=(0, 3), seed=700),
    # conv_out: dz has 3 real channels (k-step skip), ReLU' of the last transposed conv; ~28 tiles per CTA
    'conv_out': dict(kind=L.CONV_3X3, cin_real=64, cout_real=3, n=8, h=256, w=256, act=L.ACT_RELU, residual=False,
                     runs=(0, 7), seed=710),
    # transposed convs: a stride-2 conv over dz (CONV_3X3_S2, tap mode)
    'convT_256_to_128': dict(kind=L.CONVT_3X3_S2, cin_real=64, cout_real=64, n=8, h=128, w=128, act=L.ACT_RELU,
                             residual=False, runs=(0, 5), seed=720),
    'convT_128_to_64': dict(kind=L.CONVT_3X3_S2, cin_real=64, cout_real=64, n=8, h=64, w=64, act=L.ACT_RELU,
                            residual=False, runs=(0, 3), seed=730),
    # FNet decoder2.0 256->128 at 16x16: dx has 256 channels = 4 CTA groups
    'fnet_dec2_0': dict(kind=L.CONV_3X3, cin_real=256, cout_real=128, n=36, h=16, w=16, act=L.ACT_LRELU02,
                        residual=False, runs=(0, 2), seed=740),
}


def dgrad_case_operands(case):
    """weight [fp32, the layer's layout], dz16 [n,cout_real,oh,ow], residual16 / mask16 [n,cin_real,h,w] (fp16)"""
    c = DGRAD_CASES[case]
    up = 1 if c['kind'] == L.CONV_3X3 else 2
    n, ci, co, h, w, s = c['n'], c['cin_real'], c['cout_real'], c['h'], c['w'], c['seed']
    wshape = (co, ci, 3, 3) if c['kind'] == L.CONV_3X3 else (ci, co, 3, 3)
    wt = rand(s, *wshape, lo=-0.1, hi=0.1)
    dz16 = rand(s + 1, n, co, up * h, up * w, lo=-1, hi=1).half()
    res16 = rand(s + 2, n, ci, h, w, lo=-1, hi=1).half() if c['residual'] else None
    mask16 = rand(s + 3, n, ci, h, w, lo=-1, hi=1).half()
    return wt, dz16, res16, mask16


def dgrad_detection_power(case, ref=None):
    """the per-element metric of the exact reference with one output tile (the last tile of the last image)
    zeroed, against the full reference: what a kernel that skipped that tile would score"""
    c = DGRAD_CASES[case]
    if ref is None:
        wt, dz16, res16, mask16 = dgrad_case_operands(case)
        ref = _dgrad_ref64(dz16, wt, c['kind'], res16, mask16, c['act'])
    m = 1.0 - _tile_mask(ref.shape, ref.shape[0] - 1, -(-c['h'] // 16) - 1, -(-c['w'] // 8) - 1, 1)
    return _dgrad_metric((ref * m).numpy(), ref.numpy())


def check_dgrad_multitile(case):
    """PackedDgrad (the BWD instances of tg_conv_tcgen05 with the DRELU / DLRELU mask epilogue) at a training shape
    against the exact float64 reference (_dgrad_ref64).  The output is poisoned with NaN first, so every element
    must be written.  Per-element bar: |got - ref| <= 1 fp16 ulp(|ref|) + 1e-5 max|ref| -- the output is rounded
    to fp16, nothing looser is justified.  A tile is computed by one CTA with the same MMAs in the same order
    whichever CTA it is, so the runs on different grids must agree bit for bit."""
    c = DGRAD_CASES[case]
    kind = c['kind']
    wt, dz16, res16, mask16 = dgrad_case_operands(case)
    ref = _dgrad_ref64(dz16, wt, kind, res16, mask16, c['act'])
    out = {'detect_zero_tile': dgrad_detection_power(case, ref)}
    assert out['detect_zero_tile'] > 10, out
    epi = L.EPI_OUT_NCHW_F32 if c['cout_real'] <= 3 else L.EPI_NHWC_F16        # conv_out is a thin NCHW head
    fwd = ops.PackedConv(wt.to(DEV), torch.zeros(c['cout_real'], device=DEV), kind, L.ACT_NONE, epi)
    dg = ops.PackedDgrad(fwd, wt.to(DEV))
    n, h, w = c['n'], c['h'], c['w']
    dzg = nhwc(dz16.float(), dg.cin)
    res = nhwc(res16.float(), dg.cout) if res16 is not None else None
    msk = nhwc(mask16.float(), dg.cout)
    ci = c['cin_real']
    first = None
    for mc in c['runs']:
        plan = _dgrad_plan(dg.cout, n, h, w, mc, sms=ops.sm_count())
        y = torch.full((n, h, w, dg.cout), float('nan'), dtype=torch.float16, device=DEV)
        dg(dzg, y=y, residual=res, mask=msk, mask_act=c['act'], max_ctas=mc)
        torch.cuda.synchronize()
        assert not bool(torch.isnan(y).any()), f'{case} max_ctas={mc}: dgrad left output elements unwritten'
        if dg.cout > ci:
            assert float(y[..., ci:].abs().max()) == 0.0, 'pad channels of dx must be zero'
        got = from_nhwc(y, ci).double()
        r = {'tiles_per_cta': round(plan['tiles_per_cta'], 2), 'ulp_metric': _dgrad_metric(got.numpy(), ref.numpy()),
             'rel_l2': rell2(got.numpy(), ref.numpy())}
        out[f'max_ctas{mc}'] = r
        assert r['ulp_metric'] <= 1.0, (case, mc, r)
        assert mc == 0 or plan['tiles_per_cta'] > 6, (case, mc, plan)          # many tiles per CTA
        if first is None:
            first = y
        else:
            assert torch.equal(y, first), f'{case}: max_ctas={mc} differs from the default grid'
    return out


# =============================================================================== elementwise backward past one grid pass
GRID_STRIDE_ITEMS = 148 * 32 * 256         # items one pass of the backward kernels' capped grid-stride loop covers


def check_backward_elementwise_large():
    """The grid-stride elementwise backward kernels at sizes above one pass of their capped grid (148*32 blocks x 256
    threads), with the decisive values at the LAST indices, against float64 / exact host references."""
    out = {}
    # ---- loss scale: amax over 38x3x256x256 with the largest |value| last; exact power of two
    shape = (38, 3, 256, 256)
    assert int(np.prod(shape)) > GRID_STRIDE_ITEMS
    for tag, amax in (('clamped', 1.3e-8), ('free', 3.7)):
        a = rand(800, *shape, lo=-0.5 * amax, hi=0.5 * amax)
        a.view(-1)[-1] = -amax
        sc = ops.GradScale(DEV).from_amax(a.to(DEV))
        torch.cuda.synchronize()
        want = _host_scale(float(np.float32(amax)))
        out[f'scale_log2_{tag}'] = float(np.log2(float(sc.ws[0])))
        assert float(sc.ws[0]) == want and float(sc.ws[1]) == 1.0 / want, (tag, float(sc.ws[0]), want)
        assert (want == 2.0 ** 24) == (tag == 'clamped')
    # ---- grad_pack (a + b) * scale -> NHWC fp16 and grad_unpack back to NCHW fp32 / scale (accumulating)
    n, c, h, w = 38, 3, 256, 256
    a, b = rand(801, n, c, h, w, lo=-1e-8, hi=1e-8), rand(802, n, c, h, w, lo=-1e-8, hi=1e-8)
    a[-1, -1, -1, -1], b[-1, -1, -1, -1] = 3e-8, 1e-8          # the largest value: last element of the last pass
    sc = ops.GradScale(DEV).from_amax(a.to(DEV), b.to(DEV))
    pk = ops.grad_pack(a.to(DEV), b.to(DEV), scale=sc, cpad=64)
    torch.cuda.synchronize()
    s = float(sc.ws[0])
    assert s == _host_scale(max(float(a.abs().max()), float(b.abs().max()))), s
    want = ((a + b) * s).half()
    got = pk.cpu()
    assert torch.equal(got[..., :c], want.permute(0, 2, 3, 1)), 'grad_pack differs from fp16((a + b) * scale)'
    assert float(got[..., c:].abs().max()) == 0.0, 'grad_pack pad channels must be zero'
    base = rand(803, n, c, h, w, lo=-1, hi=1)
    y = base.to(DEV)
    ops.grad_unpack(pk, c, scale=sc, y=y, accumulate=True)
    torch.cuda.synchronize()
    ref = base.double() + want.double() / s
    out['grad_unpack_max_abs'] = float((y.cpu().double() - ref).abs().max())
    assert torch.equal(y.cpu(), base + want.float() / s), 'grad_unpack must be exact: fp16 * 2^-k + fp32 in fp32'
    out['grad_pack_roundtrip_rel_l2'] = rell2((want.double() / s).numpy(), (a.double() + b.double()).numpy())
    assert out['grad_pack_roundtrip_rel_l2'] <= 1e-3, out          # fp16 rounding of the scaled values
    del a, b, pk, y, base, want, got
    # ---- bias gradient over 40x256x256 = 2.6 M pixels (the transposed-conv path), pre-filled db, loss scale
    npx_n = 40
    dz = torch.empty(npx_n, 256, 256, 64, dtype=torch.float16).uniform_(-1, 1, generator=torch.Generator().manual_seed(804))
    dz[-1, -1, -1, 5] = 2000.0                             # decisive value in the very last pixel
    assert npx_n * 256 * 256 > 2 * GRID_STRIDE_ITEMS
    sc = ops.GradScale(DEV).from_amax(torch.full((1, 1, 1, 1), 1.5, device=DEV))
    db = torch.linspace(-1, 1, 64).to(DEV)
    ops.bias_grad(dz.to(DEV), db, sc)
    torch.cuda.synchronize()
    s = float(sc.ws[0])
    assert s == _host_scale(1.5) == 128.0, s
    ref = torch.linspace(-1, 1, 64).double() + dz.sum((0, 1, 2), dtype=torch.float64) / s
    out['bias_grad_rel_l2'] = rell2(db.cpu().numpy(), ref.numpy())
    out['bias_grad_ch5_rel'] = abs(float(db[5]) - float(ref[5])) / abs(float(ref[5]))
    assert out['bias_grad_rel_l2'] <= 1e-5 and out['bias_grad_ch5_rel'] <= 1e-5, out
    del dz
    # ---- fused warp + s2d + concat backward on 24 HR frames of 256x256 (1.57 M pixels), loss-scaled gx
    from oracle import frnet_torchref as R
    n, S, h, w = 24, 4, 64, 64
    assert n * S * h * S * w > GRID_STRIDE_ITEMS
    hp = rand(805, n, 3, S * h, S * w)
    hf = rand(806, n, 2, S * h, S * w, lo=-3, hi=3)
    hf[-1, :, -1, -1] = torch.tensor([-40.0, -70.0])           # the last pixel samples far across the frame
    # flows on a 2^-12 grid offset by 2^-13: x + flow is exact in fp32 and never within 2^-13 of a pixel line, where
    # the flow gradient of bilinear sampling jumps (else the fp32 rounding of the coordinate moves ~1 pixel in 3e4
    # to the neighbouring cell, an O(1) change that is the conditioning of the operation, not a kernel error)
    hf = torch.floor(hf * 4096.0) / 4096.0 + 1.0 / 8192.0
    g = rand(807, n, 51, h, w, lo=-1e-8, hi=1e-8)
    g[-1, :, -1, -1] *= 50.0
    sc = ops.GradScale(DEV).from_amax(g.to(DEV))
    s = float(sc.ws[0])
    assert s == _host_scale(float(g.abs().max())), s
    g16 = (g * s).half()
    hp64 = hp.double().requires_grad_(True)
    hf64 = hf.double().requires_grad_(True)
    xx = R.s2d(R.warp(hp64, hf64), S)
    ghp_ref, ghf_ref = torch.autograd.grad(xx, [hp64, hf64], g16[:, 3:].double() / s)
    pre = rand(808, n, 3, S * h, S * w, lo=-1e-8, hi=1e-8)
    d_hp = pre.to(DEV)
    d_hf = torch.full((n, 2, S * h, S * w), float('nan'), device=DEV)
    ops.warp_s2d_concat_bwd(nhwc(g16.float()), hp.to(DEV), hf.to(DEV), S, d_hr_prev=d_hp, d_hr_flow=d_hf, scale=sc)
    torch.cuda.synchronize()
    got_hp = d_hp.cpu().double() - pre.double()
    out['fused_warp_dhr_rel_l2'] = rell2(got_hp.numpy(), ghp_ref.numpy())
    out['fused_warp_dflow_rel_l2'] = rell2(d_hf.cpu().numpy(), ghf_ref.numpy())
    out['fused_warp_dhr_last_img_rel_l2'] = rell2(got_hp[-1].numpy(), ghp_ref[-1].numpy())
    assert out['fused_warp_dhr_rel_l2'] <= 1e-4 and out['fused_warp_dhr_last_img_rel_l2'] <= 1e-4, out
    assert out['fused_warp_dflow_rel_l2'] <= 1e-4, out          # same sample points: the closed form is exact
    return out


# =============================================================================== full-depth BPTT
def _frvsr_losses(d, gt, warp):
    """the FRVSR training losses of frvsr_train_step: Charbonnier pixel loss + Charbonnier warping loss"""
    return _charbonnier(d['hr_data'], gt), _charbonnier(warp(d['lr_prev'], d['lr_flow']), d['lr_curr'])


def _record_max(store, key, fn):
    def wrapped(*args, **kwargs):
        y = fn(*args, **kwargs)
        store[key] = max(store.get(key, 0.0), float(y.float().abs().max()))
        return y
    return wrapped


def check_sequence_grads_full_depth(n=2, t=10, lr=32, seed=41):
    """The generator backward at full depth: define_generator(FRVSR_OPT) (10 residual blocks, 4x BD), 2 clips of a
    10-frame ping-pong (19 frames), LR 32x32, the FRVSR losses, forward + backward without the optimizer step, on
    (a) the GPU, (b) the fp16 CPU precision model (tests/fake_ops.py on a separate FRNet, installed only inside a
    MonkeyPatch context) and (c) R.forward_sequence in float64.  Bars: every gradient finite; per parameter,
    rel-L2(a, c) <= 1.5 rel-L2(b, c) + 2e-3 (the pattern of check_step_golden); rel-L2(a, b) <= 1e-2; the logged
    losses within 1e-3 of (c).  fp16 headroom: the largest |value| PackedDgrad and grad_pack store on the GPU must
    be finite and <= 2^12 (fp16 max is 65504).  Measured on a B200: rel-L2(a, b) <= 3.0e-3, at most 0.51 of the
    bar against (c), losses within 1.5e-5, largest stored fp16 gradient 37 (the CPU model's too)."""
    import pytest
    from oracle import frnet_torchref as R
    here = os.path.dirname(os.path.abspath(__file__))
    if here not in sys.path:
        sys.path.insert(0, here)
    import fake_ops
    P = 'tecogan-pytorch_b200.'
    autograd, networks, net_utils = (sys.modules[P + m] for m in ('autograd', 'networks', 'net_utils'))
    p = O.make_frnet_params(seed, gain=1.0)
    lr_data, gt = bd_training_data(rand(72, n, t, 3, 4 * lr + 8, 4 * lr + 8).to(DEV))
    lr_data = torch.cat([lr_data, lr_data.flip(1)[:, 1:]], 1)          # ping-pong: 2t - 1 frames
    gt = torch.cat([gt, gt.flip(1)[:, 1:]], 1)
    assert tuple(lr_data.shape) == (n, 2 * t - 1, 3, lr, lr)
    out = {}
    # (a) the GPU, recording the largest fp16 gradient the dgrad launches and grad_pack store
    net = T.define_generator(FRVSR_OPT).to(DEV)
    net.load_state_dict(p, strict=True)
    net.train()
    head = {}
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(ops.PackedDgrad, '__call__', _record_max(head, 'dgrad', ops.PackedDgrad.__call__))
        mp.setattr(ops, 'grad_pack', _record_max(head, 'grad_pack', ops.grad_pack))
        lp, lw = _frvsr_losses(net(lr_data), gt, T.backward_warp)
        (lp + lw).backward()
        torch.cuda.synchronize()
    log_a = {'l_pix_G': lp.item(), 'l_warp_G': lw.item()}
    names = [k for k, _ in net.named_parameters()]
    ga = {k: v.grad.detach().cpu().double() if v.grad is not None else None for k, v in net.named_parameters()}
    out['fp16_headroom_gpu'] = dict(head)
    # (b) the fp16 CPU precision model on its own FRNet and CPU tensors
    lr_cpu, gt_cpu = lr_data.cpu(), gt.cpu()
    head_b = {}
    with pytest.MonkeyPatch.context() as mp:
        fake_ops.install(mp, ops, networks, net_utils, autograd)
        mp.setattr(fake_ops, 'STORAGE', torch.float16)
        mp.setattr(autograd, '_ACT_DTYPE', torch.float16)
        mp.setattr(ops.PackedDgrad, '__call__', _record_max(head_b, 'dgrad', ops.PackedDgrad.__call__))
        mp.setattr(ops, 'grad_pack', _record_max(head_b, 'grad_pack', ops.grad_pack))
        net_b = T.FRNet(3, 3, 64, 10, 'BD', 4)
        net_b.load_state_dict(p, strict=True)
        net_b.train()
        lp_b, lw_b = _frvsr_losses(net_b(lr_cpu), gt_cpu, T.backward_warp)
        (lp_b + lw_b).backward()
    gb = {k: v.grad.detach().double() for k, v in net_b.named_parameters()}
    out['fp16_headroom_cpu_model'] = dict(head_b)
    # (c) float64 through the reference's operators
    q = {k: v.double().requires_grad_(k in names) for k, v in p.items()}
    lp_c, lw_c = _frvsr_losses(R.forward_sequence(q, lr_cpu.double(), 4, 'BD', nb=10), gt_cpu.double(), R.warp)
    gc = dict(zip(names, torch.autograd.grad(lp_c + lw_c, [q[k] for k in names])))
    log_c = {'l_pix_G': lp_c.item(), 'l_warp_G': lw_c.item()}
    for k in log_c:
        out['log_rel_' + k] = abs(log_a[k] - log_c[k]) / abs(log_c[k])
        assert out['log_rel_' + k] <= 1e-3, out
    missing = [k for k in names if ga[k] is None or not bool(torch.isfinite(ga[k]).all())]
    assert not missing, f'missing or non-finite gradients: {missing}'
    worst_c, worst_b, used = 0.0, 0.0, 0.0
    for k in names:
        e_ac, e_bc, e_ab = (rell2(ga[k].numpy(), gc[k].numpy()), rell2(gb[k].numpy(), gc[k].numpy()),
                            rell2(ga[k].numpy(), gb[k].numpy()))
        if e_ac > worst_c:
            worst_c, out['worst_vs_fp64'] = e_ac, (k, e_ac, e_bc)
        if e_ab > worst_b:
            worst_b, out['worst_vs_cpu_model'] = e_ab, (k, e_ab)
        used = max(used, e_ac / (1.5 * e_bc + 2e-3))
        assert e_ac <= 1.5 * e_bc + 2e-3, (k, e_ac, e_bc, out)
    out['worst_fraction_of_fp64_bar'] = used
    assert worst_b <= 1e-2, out
    h = max(head.values())
    assert np.isfinite(h) and h <= 2.0 ** 12, out
    return out


CHECKS = {
    'warp_hrflow_s4': lambda: check_warp_hrflow(4),
    'warp_hrflow_s2': lambda: check_warp_hrflow(2, h=9, w=70),
    'warp_lrflow_bd4': lambda: check_warp_lrflow(4, 'BD'),
    'warp_lrflow_bi2': lambda: check_warp_lrflow(2, 'BI', h=20, w=24),
    'pool_upsample': check_pool_upsample,
    'module_ops': check_module_ops,
    'downsample_bd': check_downsample_bd,
    'conv_simt_64': lambda: check_conv('simt'),
    'conv_simt_pad': lambda: check_conv('simt', cin=64, cout=64, cin_real=51, cout_real=32, act=L.ACT_LRELU02),
    'conv_simt_convT': lambda: check_conv('simt', kind=L.CONVT_3X3_S2),
    'conv_simt_res': lambda: check_conv('simt', act=L.ACT_NONE, residual=True),
    'conv_simt_256': lambda: check_conv('simt', cin=256, cout=128, h=9, w=12),
    'epilogues_simt': lambda: check_conv_epilogues('simt'),
    'conv_tc_tap_64': lambda: check_conv('tcgen05', L.AMODE_TAP),
    'conv_tc_halo_64': lambda: check_conv('tcgen05', L.AMODE_HALO),
    'conv_tc_halo_res': lambda: check_conv('tcgen05', L.AMODE_HALO, act=L.ACT_NONE, residual=True),
    'conv_tc_tap_convT': lambda: check_conv('tcgen05', L.AMODE_TAP, kind=L.CONVT_3X3_S2),
    'conv_tc_halo_convT': lambda: check_conv('tcgen05', L.AMODE_HALO, kind=L.CONVT_3X3_S2),
    'conv_tc_tap_128_256': lambda: check_conv('tcgen05', L.AMODE_TAP, cin=128, cout=256, h=16, w=40),
    'conv_tc_tap_256_256': lambda: check_conv('tcgen05', L.AMODE_TAP, cin=256, cout=256, h=16, w=40),
    'conv_tc_tap_256_128': lambda: check_conv('tcgen05', L.AMODE_TAP, cin=256, cout=128, h=33, w=80, n=1),
    'conv_tc_tap_64_128': lambda: check_conv('tcgen05', None, cin=64, cout=128, h=33, w=80, n=2),
    'conv_tc_nsplit_res': lambda: check_conv('tcgen05', None, cin=128, cout=128, h=17, w=20, act=L.ACT_NONE, residual=True),
    'conv_tc_auto_128_256': lambda: check_conv('tcgen05', None, cin=128, cout=256, h=16, w=40),
    'conv_tc_auto_pad': lambda: check_conv('tcgen05', None, cin=64, cout=64, cin_real=51, cout_real=32, act=L.ACT_LRELU02),
    'epilogues_tc': lambda: check_conv_epilogues('tcgen05'),
    'conv_tc_vs_simt_tap_full': lambda: check_conv_vs_simt(L.AMODE_TAP),
    'conv_tc_vs_simt_halo_full': lambda: check_conv_vs_simt(L.AMODE_HALO),
    'conv_tc_vs_simt_halo_convT_full': lambda: check_conv_vs_simt(L.AMODE_HALO, kind=L.CONVT_3X3_S2),
    'conv_tc_vs_simt_halo_2cta': lambda: check_conv_vs_simt(L.AMODE_HALO, h=64, w=64, n=2, max_ctas=3),
    'conv_issue_variants_64': lambda: check_conv_issue_variants(residual=True),
    'conv_issue_variants_thin_6_32': lambda: check_conv_issue_variants(cin_real=6, cout_real=32),
    'conv_issue_variants_thin_32_64': lambda: check_conv_issue_variants(cin_real=32, cout_real=64, h=33, w=80),
    'conv_issue_variants_convT': lambda: check_conv_issue_variants(kind=L.CONVT_3X3_S2, h=24, w=40, n=2),
    'conv_chain_vs_reference': check_conv_chain_vs_reference,
    'conv_chain_1tile': lambda: check_conv_chain(n=1, h=16, w=8, blocks=1),
    'conv_chain_ragged_repeat': lambda: check_conv_chain(n=2, h=37, w=29, blocks=2, repeats=3),
    'conv_chain_few_ctas': lambda: check_conv_chain(n=3, h=50, w=44, blocks=3, max_ctas=5, repeats=2),
    'conv_chain_full': lambda: check_conv_chain(n=4, h=134, w=320, blocks=10, repeats=2),
    'conv_chain_24_layers': check_conv_chain_plain,
    'conv_chain_two_tiles_per_cta': lambda: check_conv_chain(n=1, h=134, w=320, blocks=4, max_ctas=0, repeats=2, seed=120),
    'step_golden_g1': lambda: check_step_golden('g1'),
    'step_golden_g15': lambda: check_step_golden('g15'),
    'step_golden_g2_stress': lambda: check_step_golden('g2'),
    'step_bi2_golden': check_step_bi2,
    'infer_sequence_golden': check_infer_sequence_golden,
    'forward_sequence_golden': check_forward_sequence_golden,
    'batch_consistency': check_batch_consistency,
    'engine_matches_eager': check_engine_matches_eager,
    'properties_fullsize': check_properties_fullsize,
    'ragged_sizes': check_ragged_sizes,
    'bi2_fullsize': check_bi2_fullsize,
    'step_vs_oracle_fullsize': check_step_vs_oracle_fullsize,
    'bench_workload_parity': check_bench_workload_parity,
    'bi2_workload_parity': check_bi2_workload_parity,
    'reference_callers_integration': check_reference_callers_integration,
    'conv_pool_epilogue_halo': check_conv_pool_epilogue,
    'conv_pool_epilogue_128_tap': lambda: check_conv_pool_epilogue(cin=128, cout=128, h=33, w=80, n=1, seed=510),
    'conv_pool_epilogue_fullres': lambda: check_conv_pool_epilogue(h=134, w=320, n=2, seed=520),
    'fused_tail_bd4': lambda: check_fused_tail(4),
    'fused_tail_bd4_ragged_1img': lambda: check_fused_tail(4, n=1, h=30, w=14, seed=410),
    'fused_tail_bd4_big': lambda: check_fused_tail(4, n=2, h=64, w=46, seed=420),
    'fused_tail_bi2': lambda: check_fused_tail(2, n=3, h=21, w=33, seed=430),
    'fused_tail_accumulate_bd4': lambda: check_fused_tail(4, n=2, h=34, w=22, seed=450, accumulate=True),
    'fused_tail_accumulate_bi2': lambda: check_fused_tail(2, n=1, h=17, w=31, seed=460, accumulate=True),
    'fused_tail_no_residual': lambda: check_fused_tail(4, with_lr=False, h=18, w=8, seed=440),
    'autograd_guards': check_autograd_guards,
    'dgrad_simt_conv': lambda: check_conv_dgrad('simt'),
    'dgrad_simt_convT': lambda: check_conv_dgrad('simt', kind=L.CONVT_3X3_S2, h=10, w=12),
    'dgrad_tc_conv': lambda: check_conv_dgrad('tcgen05'),
    'dgrad_tc_conv_mask_res': lambda: check_conv_dgrad('tcgen05', mask_act=L.ACT_RELU, residual=True, h=37, w=29),
    'dgrad_tc_conv_lrelu_256_128': lambda: check_conv_dgrad('tcgen05', cin=128, cout=256, h=16, w=40, mask_act=L.ACT_LRELU02),
    'dgrad_tc_conv_thin': lambda: check_conv_dgrad('tcgen05', cin=64, cout=64, cin_real=32, cout_real=2, mask_act=L.ACT_LRELU02),
    'dgrad_tc_convT': lambda: check_conv_dgrad('tcgen05', kind=L.CONVT_3X3_S2, h=21, w=12, mask_act=L.ACT_RELU),
    'dgrad_tc_convT_fullrow': lambda: check_conv_dgrad('tcgen05', kind=L.CONVT_3X3_S2, h=64, w=64, n=1),
    'wgrad_conv': lambda: check_wgrad(flags=(0, 1, 2, 3)),
    'wgrad_conv_ragged': lambda: check_wgrad(h=37, w=29, n=3),
    'wgrad_conv_thin': lambda: check_wgrad(cin_real=51, cout_real=3, h=24, w=40),
    'wgrad_conv_128_256': lambda: check_wgrad(cin=128, cout=256, h=16, w=40),
    'wgrad_convT': lambda: check_wgrad(kind=L.CONVT_3X3_S2, h=18, w=20, flags=(0, 1, 2, 3)),
    'wgrad_convT_ragged': lambda: check_wgrad(kind=L.CONVT_3X3_S2, h=21, w=13, n=3),
    'backward_elementwise': check_backward_elementwise,
    'fnet_autograd_public': check_fnet_autograd_public,
    'sequence_grads_golden': check_sequence_grads_golden,
    'sequence_grads_golden_tiny_loss': lambda: check_sequence_grads_golden(1e-7),
    'reference_training_integration': check_reference_training_integration,
    'st_discriminator_input': check_st_discriminator_input,
    'reference_gan_training_integration': check_reference_gan_training_integration,
    'reference_training_integration_ddp': lambda: check_reference_training_integration(ddp=True),
    'step_vs_oracle_fullsize_g15': lambda: check_step_vs_oracle_fullsize(gain=1.5, frames=2),
    'wgrad_multitile_srnet_conv': lambda: check_wgrad_multitile('srnet_conv'),
    'wgrad_multitile_conv_out': lambda: check_wgrad_multitile('conv_out'),
    'wgrad_multitile_convT_64': lambda: check_wgrad_multitile('convT_64'),
    'wgrad_multitile_convT_128': lambda: check_wgrad_multitile('convT_128'),
    'wgrad_multitile_fnet_enc1_0': lambda: check_wgrad_multitile('fnet_enc1_0'),
    'wgrad_multitile_fnet_dec1_0': lambda: check_wgrad_multitile('fnet_dec1_0'),
    'wgrad_multitile_fnet_dec1_2': lambda: check_wgrad_multitile('fnet_dec1_2'),
    'wgrad_multitile_fnet_dec2_0': lambda: check_wgrad_multitile('fnet_dec2_0'),
    'wgrad_multitile_fnet_flow_2': lambda: check_wgrad_multitile('fnet_flow_2'),
    'wgrad_multitile_max_ctas_sweep': lambda: check_wgrad_multitile('max_ctas_sweep'),
    'dgrad_multitile_srnet_halo': lambda: check_dgrad_multitile('srnet_halo'),
    'dgrad_multitile_conv_out': lambda: check_dgrad_multitile('conv_out'),
    'dgrad_multitile_convT_256_to_128': lambda: check_dgrad_multitile('convT_256_to_128'),
    'dgrad_multitile_convT_128_to_64': lambda: check_dgrad_multitile('convT_128_to_64'),
    'dgrad_multitile_fnet_dec2_0': lambda: check_dgrad_multitile('fnet_dec2_0'),
    'backward_elementwise_large': check_backward_elementwise_large,
    'sequence_grads_full_depth': check_sequence_grads_full_depth,
}
