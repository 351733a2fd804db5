"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(skycrapers/TecoGAN-PyTorch @ 903b070) on seeded inputs:

    TECOGAN_REFERENCE=<checkout of the reference> python oracle/gen_golden.py [integration]

Import recipe = SURVEY.md section 9 (two module stubs, no edits to the reference).
Inputs and weights are NOT stored: they are regenerated from seeds by
oracle.frnet_oracle.make_frnet_params / numpy default_rng, so the fixtures hold
only the reference's outputs.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def import_reference():
    import refimport                                        # SURVEY.md section 9 recipe, no reference edits
    return refimport.import_generator()


def rand(seed, *shape, lo=0.0, hi=1.0):
    return torch.from_numpy(np.random.default_rng(seed).uniform(lo, hi, size=shape).astype(np.float32))


def gen_downsample_bd(data_utils, out_dir):
    """BD degradation of the data side (SURVEY 8-f2): create_kernel + downsample_bd
    (codes/utils/data_utils.py:11-53) -- the reference calls scipy.signal.gaussian, an alias that
    newer scipy only keeps under scipy.signal.windows."""
    import scipy.signal
    if not hasattr(scipy.signal, 'gaussian'):
        scipy.signal.gaussian = scipy.signal.windows.gaussian
    kern = data_utils.create_kernel(1.5)                      # [3,3,9,9]
    a = data_utils.downsample_bd(rand(30, 2, 3, 36, 44), kern, 4, pad_data=True)
    b = data_utils.downsample_bd(rand(31, 1, 3, 41, 45), kern, 4, pad_data=False)
    c = data_utils.downsample_bd(rand(32, 1, 3, 27, 30), kern, 2, pad_data=True)
    np.savez_compressed(os.path.join(out_dir, 'downsample_bd.npz'), kernel=kern.numpy(),
                        s4_pad=a.numpy(), s4_valid=b.numpy(), s2_pad=c.numpy())


GRAD_FULL = ('fnet.encoder1.0.weight', 'fnet.flow.2.weight', 'fnet.flow.2.bias', 'srnet.conv_in.0.weight',
             'srnet.resblocks.1.conv.2.bias', 'srnet.conv_up.2.bias', 'srnet.conv_out.weight', 'srnet.conv_out.bias')


def gen_sequence_grads(FRNet, out_dir):
    from oracle.frnet_oracle import make_frnet_params
    net = FRNet(3, 3, 64, 2, 'BD', 4)
    net.load_state_dict(make_frnet_params(15, nb=2, scale=4, degradation='BD', gain=1.5), strict=True)
    net.train()
    lr_data = rand(9, 1, 3, 3, 16, 16).requires_grad_(True)
    d = net.forward_sequence(lr_data)
    rng = np.random.default_rng(16)
    r1 = torch.from_numpy(rng.uniform(-1, 1, size=tuple(d['hr_data'].shape)).astype(np.float32))
    r2 = torch.from_numpy(rng.uniform(-1, 1, size=tuple(d['lr_flow'].shape)).astype(np.float32))
    loss = (d['hr_data'] * r1).sum() + 0.05 * (d['lr_flow'] * r2).sum()
    loss.backward()
    named = dict(net.named_parameters())
    out = {'loss': np.float32(loss.item()), 'd_lr_data': lr_data.grad.numpy(),
           'names': np.array(list(named)), 'norms': np.array([float(v.grad.norm()) for v in named.values()], np.float64)}
    for k in GRAD_FULL:
        out['g:' + k] = named[k].grad.numpy()
    np.savez_compressed(os.path.join(out_dir, 'fwd_seq_grads_bd4_16x16_nb2_g15.npz'), **out)
    print('sequence grads: loss', loss.item(), 'max |d lr_data|', float(lr_data.grad.abs().max()))


# Fixtures of the integration checks hold strided samples (every SAMPLE_STRIDE-th element of the flattened
# output) so that they stay small; the tests take the same elements of their own result.
SAMPLE_STRIDE = {'callers': 14, 'st_disc': 26, 'full_size': 241}
ADAM_SAMPLES = 256          # per parameter: positions of the sign check of the first Adam step


def gen_callers_infer(out_dir):
    """The reference's inference callers on the CPU: VSRModel from the FRVSR test YAML (reflect temporal
    padding, 5 frames) -> prepare_inference_data -> infer(), reference generator with seeded weights."""
    import copy
    import yaml
    import refimport
    from oracle.frnet_oracle import make_frnet_params, make_clip
    models, _ = refimport.import_models()
    yml = os.path.join(refimport.root_dir(), 'experiments_BD', 'FRVSR', 'FRVSR_VimeoTecoGAN_4xSR_2GPU', 'test.yml')
    opt = yaml.safe_load(open(yml))
    opt['model']['generator'].pop('load_path', None)
    opt.update({'dist': False, 'is_train': False, 'rank': 0, 'world_size': 1, 'device': 'cpu'})
    m = models.vsr_model.VSRModel(copy.deepcopy(opt))
    m.net_G.load_state_dict(make_frnet_params(23, gain=1.5), strict=True)
    m.prepare_inference_data({'lr': make_clip(11, 9, 3, 18, 28).permute(0, 2, 3, 1).contiguous()})
    seq = m.infer()
    np.savez_compressed(os.path.join(out_dir, 'callers_infer_bd4_18x28_g15.npz'), shape=np.array(seq.shape),
                        hr_seq_sample=seq.reshape(-1)[::SAMPLE_STRIDE['callers']])
    print('callers infer', seq.shape, seq.dtype)


def gen_frvsr_train_step(out_dir):
    """One iteration of the reference's FRVSR training loop (VSRModel.train, FRVSR train.yml, nb=2) with the
    reference generator on the CPU: logged losses, every parameter gradient's norm, two whole gradients (conv_in
    as fp16 relative to its largest magnitude) and the sign of the first Adam step at sampled large-gradient positions of every parameter."""
    import copy
    import yaml
    import refimport
    from oracle.frnet_oracle import make_frnet_params
    models, _ = refimport.import_models()
    yml = os.path.join(refimport.root_dir(), 'experiments_BD', 'FRVSR', 'FRVSR_VimeoTecoGAN_4xSR_2GPU', 'train.yml')
    opt = yaml.safe_load(open(yml))
    opt['model']['generator']['nb'] = 2
    opt.update({'dist': False, 'is_train': True, 'rank': 0, 'world_size': 1, 'device': 'cpu'})
    opt['train']['ckpt_dir'] = '/tmp'
    p = make_frnet_params(41, nb=2, gain=1.5)
    m = models.vsr_model.VSRModel(copy.deepcopy(opt))
    m.net_G.load_state_dict(p, strict=True)
    m.prepare_training_data({'gt': rand(70, 2, 4, 3, 72, 72)})
    m.train()
    named = dict(m.net_G.named_parameters())
    idx, sign, count = [], [], []
    for k, v in named.items():
        g = v.grad.detach().reshape(-1)
        big = torch.nonzero(g.abs() > 0.1 * g.abs().max())[:, 0]
        sel = big[::max(1, len(big) // ADAM_SAMPLES)][:ADAM_SAMPLES]
        idx.append(sel.numpy().astype(np.int32))
        sign.append(torch.sign(v.detach().reshape(-1)[sel] - p[k].reshape(-1)[sel]).numpy().astype(np.int8))
        count.append(len(sel))
    out = {'log_keys': np.array(list(m.log_dict)), 'log_values': np.array(list(m.log_dict.values()), np.float64),
           'names': np.array(list(named)), 'norms': np.array([float(v.grad.norm()) for v in named.values()], np.float64),
           'adam_idx': np.concatenate(idx), 'adam_sign': np.concatenate(sign), 'adam_count': np.array(count, np.int32)}
    out['g:fnet.encoder1.0.weight'] = named['fnet.encoder1.0.weight'].grad.numpy()
    out['g:srnet.conv_in.0.weight'], out['g:srnet.conv_in.0.weight_scale'] = _f16_scaled(
        named['srnet.conv_in.0.weight'].grad.numpy())
    np.savez_compressed(os.path.join(out_dir, 'train_frvsr_bd4_nb2_g15.npz'), **out)
    print('frvsr train step', dict(m.log_dict))


# TecoGAN training step of the GAN fixture: 4-frame clips (ping-pong: 7 frames), 32x32 GT crops, nb=2
TECOGAN_STEP = dict(t=4, crop=32, seed_gt=80, seed_params=43)


def _f16_scaled(x):
    """x as fp16 after division by max|x| (keeps small gradients out of the fp16 subnormal range)"""
    s = float(np.abs(x).max())
    return (x / s).astype(np.float16), np.float64(s)


def gen_tecogan_train_step(out_dir):
    """One iteration of the reference's TecoGAN training loop (VSRGANModel.train: adaptive ST-discriminator
    update, then pixel + warping + VGG feature + ping-pong + GAN losses for the generator) with the reference
    generator on the CPU.  Stored: the logged losses, every generator gradient's norm, the conv_in / conv_out
    gradients, and the cotangents d loss_G / d hr_data and d loss_G / d lr_flow -- the only two generator
    outputs the loss reaches (the discriminator detaches the flows it takes from hr_flow)."""
    import refimport
    from oracle.frnet_oracle import make_frnet_params
    cfg = TECOGAN_STEP
    opt = refimport.training_opt('tecogan', device='cpu', nb=2)
    opt['dataset']['train']['crop_size'] = cfg['crop']
    opt['train']['tempo_extent'] = cfg['t']
    m = refimport.build_training_model(opt)
    m.net_G.load_state_dict(make_frnet_params(cfg['seed_params'], nb=2, gain=1.0), strict=True)
    cot = {}
    forward = m.net_G.forward

    def capturing_forward(*args, **kwargs):
        d = forward(*args, **kwargs)
        for key in ('hr_data', 'lr_flow'):
            d[key].register_hook(lambda g, key=key: cot.__setitem__(key, g.detach().clone() + cot.get(key, 0)))
        return d

    m.net_G.forward = capturing_forward
    gt_hw = cfg['crop'] + 2 * int(1.5 * 3.0)
    m.prepare_training_data({'gt': rand(cfg['seed_gt'], 1, cfg['t'], 3, gt_hw, gt_hw)})
    m.train()
    named = dict(m.net_G.named_parameters())
    cot_hr, cot_hr_scale = _f16_scaled(cot['hr_data'].numpy())
    g_in, g_in_scale = _f16_scaled(named['srnet.conv_in.0.weight'].grad.numpy())
    out = {'log_keys': np.array(list(m.log_dict)), 'log_values': np.array(list(m.log_dict.values()), np.float64),
           'names': np.array(list(named)), 'norms': np.array([float(v.grad.norm()) for v in named.values()], np.float64),
           'cot_hr_data': cot_hr, 'cot_hr_data_scale': cot_hr_scale, 'cot_lr_flow': cot['lr_flow'].numpy(),
           'g:srnet.conv_out.weight': named['srnet.conv_out.weight'].grad.numpy(),
           'g:srnet.conv_in.0.weight': g_in, 'g:srnet.conv_in.0.weight_scale': g_in_scale}
    np.savez_compressed(os.path.join(out_dir, 'train_tecogan_bd4_nb2_t4_32x32.npz'), **out)
    print('tecogan train step', dict(m.log_dict), {k: tuple(v.shape) for k, v in cot.items()})


def gen_st_disc_input(out_dir):
    """The input tensor of the reference's SpatioTemporalDiscriminator (forward_sequence with use_pp_crit,
    captured at conv_in) and its gradient w.r.t. the frames for a seeded cotangent."""
    FRNet, _, _ = import_reference()
    from models.networks.tecogan_nets import SpatioTemporalDiscriminator
    n, t, c, s, h = 2, 7, 3, 4, 8
    H = s * h
    D = SpatioTemporalDiscriminator(in_nc=3, spatial_size=H, tempo_range=3, degradation='BD', scale=4)
    captured = {}

    class _Stop(Exception):
        pass

    class _Capture(torch.nn.Module):
        def forward(self, x):
            captured['x'] = x
            raise _Stop()

    D.conv_in = _Capture()
    data = rand(90, n, t, c, H, H).requires_grad_(True)
    args = {'net_G': None, 'lr_data': rand(92, n, t, c, h, h), 'bi_data': rand(91, n, t, c, H, H),
            'hr_flow': rand(93, n, t - 1, 2, H, H, lo=-3, hi=3), 'use_pp_crit': True, 'crop_border_ratio': 0.75}
    try:
        D.forward_sequence(data, args)
    except _Stop:
        pass
    x = captured['x']
    gx, = torch.autograd.grad(x, [data], rand(94, *x.shape, lo=-1, hi=1))
    st = SAMPLE_STRIDE['st_disc']
    x, gx = x.detach().numpy(), gx.numpy()
    np.savez_compressed(os.path.join(out_dir, 'st_disc_input_bd4_n2t7_32x32.npz'),
                        x_shape=np.array(x.shape), x_sample=x.reshape(-1)[::st], x_norm=np.linalg.norm(x),
                        grad_sample=gx.reshape(-1)[::st], grad_norm=np.linalg.norm(gx))
    print('st disc input', x.shape)


def gen_step_full_size(out_dir):
    """FRNet.step at the benchmark size 3x134x320 -> 3x536x1280 (4x BD, 2x-gain weights)."""
    from oracle.frnet_oracle import make_frnet_params
    FRNet, _, _ = import_reference()
    net = FRNet(3, 3, 64, 10, 'BD', 4)
    net.load_state_dict(make_frnet_params(5, gain=2.0), strict=True)
    net.eval()
    with torch.no_grad():
        hr = net.step(rand(1, 1, 3, 134, 320), rand(2, 1, 3, 134, 320), rand(3, 1, 3, 536, 1280)).numpy()
    np.savez_compressed(os.path.join(out_dir, 'step_bd4_134x320_g2_sample.npz'), shape=np.array(hr.shape),
                        hr_sample=hr.reshape(-1)[::SAMPLE_STRIDE['full_size']], hr_absmax=np.abs(hr).max())
    print('full-size step', hr.shape)


def gen_integration(out_dir):
    gen_callers_infer(out_dir)
    gen_frvsr_train_step(out_dir)
    gen_tecogan_train_step(out_dir)
    gen_st_disc_input(out_dir)
    gen_step_full_size(out_dir)


def main():
    from oracle.frnet_oracle import make_frnet_params, make_clip
    FRNet, net_utils, data_utils = import_reference()
    out_dir = os.path.join(ROOT, 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)
    torch.set_num_threads(8)
    if sys.argv[1:] == ['integration']:              # only the integration fixtures
        return gen_integration(out_dir)
    gen_downsample_bd(data_utils, out_dir)
    if sys.argv[1:] == ['bd']:                       # only this fixture
        return
    if sys.argv[1:] == ['grads']:
        return gen_sequence_grads(FRNet, out_dir)

    def ref_model(scale, degradation, seed, gain, nb=10):
        net = FRNet(3, 3, 64, nb, degradation, scale)
        sd = make_frnet_params(seed, nb=nb, scale=scale, degradation=degradation, gain=gain)
        net.load_state_dict(sd, strict=True)
        return net.eval()

    # ---- 1. FRNet.step, 4x BD, size not a multiple of 8 (reflect pad 2 rows / 4 cols)
    for tag, gain in (('g1', 1.0), ('g15', 1.5), ('g2', 2.0)):
        net = ref_model(4, 'BD', seed=11, gain=gain)
        lr_curr, lr_prev = rand(1, 1, 3, 18, 28), rand(2, 1, 3, 18, 28)
        hr_prev = rand(3, 1, 3, 72, 112)
        with torch.no_grad():
            lr_flow = net.fnet(lr_curr, lr_prev)
            hr = net.step(lr_curr, lr_prev, hr_prev)
        np.savez_compressed(os.path.join(out_dir, f'step_bd4_18x28_{tag}.npz'),
                            lr_flow=lr_flow.numpy(), hr_curr=hr.numpy(),
                            meta=np.array([4, 11, 1, 2, 3], dtype=np.int64), gain=np.float32(gain))
        print(tag, 'flow absmax', float(lr_flow.abs().max()), 'hr range', float(hr.min()), float(hr.max()))

    # ---- 2. FRNet.step, 2x BI (bilinear upsample_func), pad 4 rows
    net = ref_model(2, 'BI', seed=12, gain=1.5)
    lr_curr, lr_prev = rand(4, 1, 3, 20, 24), rand(5, 1, 3, 20, 24)
    hr_prev = rand(6, 1, 3, 40, 48)
    with torch.no_grad():
        lr_flow = net.fnet(lr_curr, lr_prev)
        hr = net.step(lr_curr, lr_prev, hr_prev)
    np.savez_compressed(os.path.join(out_dir, 'step_bi2_20x24_g15.npz'),
                        lr_flow=lr_flow.numpy(), hr_curr=hr.numpy(), gain=np.float32(1.5))

    # ---- 3. FRNet.infer_sequence (uint8 THWC), 4x BD, 4 frames of a moving clip
    net = ref_model(4, 'BD', seed=13, gain=1.5)
    clip = make_clip(7, 4, 3, 16, 24)
    with torch.no_grad():
        seq = net.infer_sequence(clip, torch.device('cpu'))
    np.savez_compressed(os.path.join(out_dir, 'infer_seq_bd4_16x24_g15.npz'), hr_seq=seq)
    print('infer_sequence', seq.shape, seq.dtype)

    # ---- 4. FRNet.forward_sequence (training forward), 4x BD, n=1 t=3 16x16
    net = ref_model(4, 'BD', seed=14, gain=1.5)
    lr_data = rand(8, 1, 3, 3, 16, 16)
    net.train()
    with torch.no_grad():
        d = net.forward_sequence(lr_data)
    np.savez_compressed(os.path.join(out_dir, 'fwd_seq_bd4_16x16_g15.npz'),
                        **{k: v.numpy() for k, v in d.items()})

    # ---- 4b. gradients of forward_sequence (generator backward, SURVEY 8-f1), nb=2 to keep it small:
    # loss = <hr_data, R1> + 0.05 <lr_flow, R2>; stored: loss, d/d lr_data, a few whole parameter
    # gradients and the L2 norm of every parameter gradient
    gen_sequence_grads(FRNet, out_dir)

    # ---- 5. functional ops
    x = rand(20, 2, 3, 20, 24)
    flow = rand(21, 2, 2, 20, 24, lo=-4.0, hi=4.0)
    flow[0, :, 0, 0] = torch.tensor([-30.0, 40.0])   # far out of range -> border clamp
    warped = net_utils.backward_warp(x, flow)
    s2d4 = net_utils.space_to_depth(rand(22, 2, 3, 16, 24), 4)
    s2d2 = net_utils.space_to_depth(rand(22, 2, 3, 16, 24), 2)
    bic4 = net_utils.BicubicUpsampler(4)(rand(23, 1, 3, 9, 11))
    bic2 = net_utils.BicubicUpsampler(2)(rand(23, 1, 3, 9, 11))
    bil4 = net_utils.get_upsampling_func(4, 'BI')(rand(23, 1, 3, 9, 11))
    bil2 = net_utils.get_upsampling_func(2, 'BI')(rand(23, 1, 3, 9, 11))
    q_in = np.concatenate([np.arange(-3, 520, dtype=np.float32) / np.float32(510.0),   # x.5 ties
                           np.random.default_rng(24).uniform(-0.2, 1.2, 1000).astype(np.float32)])
    q = data_utils.float32_to_uint8(q_in)
    convt = torch.nn.ConvTranspose2d(8, 8, 3, 2, 1, output_padding=1)
    wt = rand(25, 8, 8, 3, 3, lo=-1, hi=1)
    bt = rand(26, 8, lo=-1, hi=1)
    with torch.no_grad():
        convt.weight.copy_(wt)
        convt.bias.copy_(bt)
        ct = convt(rand(27, 1, 8, 5, 7))
    np.savez_compressed(os.path.join(out_dir, 'ops.npz'),
                        warped=warped.numpy(), s2d4=s2d4.numpy(), s2d2=s2d2.numpy(),
                        bic4=bic4.numpy(), bic2=bic2.numpy(), bil4=bil4.numpy(), bil2=bil2.numpy(),
                        q_in=q_in, q=q, convt=ct.numpy())

    # ---- 6. the reference's callers, training step, discriminator input and the full-size step
    gen_integration(out_dir)
    print('done ->', out_dir)


if __name__ == '__main__':
    main()
