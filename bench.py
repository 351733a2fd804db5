#!/usr/bin/env python
"""bench.py -- HR frames/sec of the FRNet hot path at 4x BD, LR 3x134x320 -> HR 3x536x1280.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|eager-gpu]
                    [--dump-outputs DIR]   (writes the last timed step's outputs as DIR/*.npy)

Workload (BASELINE.json configs[1]): TecoGAN 4x BD inference, synthetic 3x134x320 clips, 4 clips
lock-stepped per GPU.  One "step" = one recurrent frame of all 4 clips on one GPU = 4 HR frames.
N > 1: launched by torchrun, one rank per GPU; clips shard across ranks with no data-path
collective (the recurrence keeps a clip on one device) -> weak scaling.

Prints ONE JSON line (rank 0):
  value      whole-job HR frames/s with inputs resident in HBM (CUDA-graph replay of the step,
             timed with CUDA events, max over ranks)
  e2e        the same metric through the reference-facing call FRNet.infer_sequence() with HOST
             buffers: per step the H2D copy of the LR frames and the D2H copy of the uint8 HR
             frames are inside the timed region
  roofline   the dominant kernel (conv_chain_kernel: SRNet conv_in + 10 residual blocks = 21 convs
             64->64 in one persistent tcgen05 launch) timed live with CUDA events against the measured
             tensor peak; `traffic` = its DRAM bytes from one ncu --set full capture
  roofline_conv_single  one residual conv 64->64 as its own launch (conv_tcgen05_kernel)
  roofline_warp*  the fused warp+space_to_depth+concat kernel against the HBM roofline
  cpu_baseline   the reference's CPU path (oracle/frnet_torchref.py: same PyTorch CPU library
             ops as the reference) on the box's host cores, bounded sample (rank 0, N=1)

--impl reference times ONLY that CPU path with the same metric/unit (rank 0 alone).
--impl eager-gpu is a second REFERENCE arm (context, not part of the contract, never what `value`
measures): the same port of the reference's operator sequence, executed by PyTorch's CUDA library
kernels on the same GPU instead of the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The two inference workloads of BASELINE.json; --workload selects one (default: the headline bd4).
WORKLOADS = {
    # configs[1]: TecoGAN 4x BD inference, synthetic 3x134x320, batch=4 lock-stepped clips per B200
    'bd4': dict(lr=(3, 134, 320), scale=4, degradation='BD', clips_per_gpu=4,
                flop_per_frame=94.438e9,          # reference counter, SURVEY.md 8-d (FNet 10.511 + SRNet 83.927)
                warp_bytes_per_frame=22983680,    # SURVEY.md 8-d byte formula, fp32
                metric='hr_frames_per_sec_4xBD_3x134x320',
                name='TecoGAN 4x BD inference, synthetic 3x134x320 -> 3x536x1280, batch=4 lock-stepped clips per '
                     'B200 (BASELINE.json configs[1]); clips shard across GPUs, no collective'),
    # configs[4]: TecoGAN 2x BI inference, synthetic 3x268x640 LR, 30-frame clips, sequence-sharded over GPUs
    'bi2': dict(lr=(3, 268, 640), scale=2, degradation='BI', clips_per_gpu=2,
                flop_per_frame=313.916e9,         # FNet 43.019 + SRNet 270.897
                warp_bytes_per_frame=26071040,
                metric='hr_frames_per_sec_2xBI_3x268x640',
                name='TecoGAN 2x BI inference, synthetic 3x268x640 -> 3x536x1280, 30-frame clips, 2 lock-stepped '
                     'clips per B200 (BASELINE.json configs[4]); clips round-robin over GPUs (main.py:169), '
                     'no collective'),
}
WL = WORKLOADS['bd4']                # set by main()
LR, SCALE, CLIPS_PER_GPU = WL['lr'], WL['scale'], WL['clips_per_gpu']
RES_CONV_FLOP_PER_PX = 2 * 9 * 64 * 64
PUBLISHED_FPS_1080TI = 27.0            # resources/benchmark.png (GTX 1080 Ti, batch 1, 4x BD 134x320)


WL_KEY = 'bd4'


def select_workload(name):
    global WL, WL_KEY, LR, SCALE, CLIPS_PER_GPU
    WL_KEY = name
    WL = WORKLOADS[name]
    LR, SCALE, CLIPS_PER_GPU = WL['lr'], WL['scale'], WL['clips_per_gpu']


def workload_config(world):
    """`config` of the JSON line -- identical for our arm and the reference arm."""
    return {'workload': WL['name'], 'clips_per_gpu': CLIPS_PER_GPU, 'frames_per_step': CLIPS_PER_GPU * world,
            'weights': 'seeded random init (no checkpoint)',
            'l2': 'inputs larger than L2: ~1.3 GB of activations per step >> 126 MB, no explicit flush'}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        d = json.load(open(path))
        return {'hbm_gbs': d['hbm_gbs'], 'tflops_burst': d['bf16_tflops'],
                'tflops_sustained': d['bf16_tflops_sustained'], 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'tflops_burst': 1590.0, 'tflops_sustained': 1400.0, 'src': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                 '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def make_params():
    import synthetic
    return synthetic.make_frnet_params(0, scale=SCALE, degradation=WL['degradation'], gain=1.0)


def synthetic_clips(n, t, seed=0):
    """n smooth translating clips [n,t,c,h,w] of the selected workload (SURVEY.md 8-d) -- synthetic data."""
    import torch
    import synthetic
    base = synthetic.make_clip(seed, min(t, 12), *LR)    # generate 12 frames, then ping-pong in time
    idx = [i % max(1, 2 * len(base) - 2) for i in range(t)]
    idx = [i if i < len(base) else 2 * len(base) - 2 - i for i in idx]
    one = base[idx]
    return torch.stack([torch.roll(one, shifts=17 * k, dims=-1) for k in range(n)])


# =============================================================================== reference arm
def _host_threads(threads=None):
    """torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use the host cores this
    process may run on (affinity mask, capped at 64: oversubscribing oneDNN's OpenMP pool stalls)."""
    import torch
    if threads is None and torch.get_num_threads() == 1:
        try:
            threads = min(64, len(os.sched_getaffinity(0)))
        except Exception:
            threads = None
    if threads:
        torch.set_num_threads(threads)
    return torch.get_num_threads()


def reference_net(device):
    """The UNMODIFIED reference FRNet (the checkout named by $TECOGAN_REFERENCE, see refimport.py) holding
    the benchmark's seeded weights; None when it is not available."""
    import refimport
    if not refimport.available():
        return None
    FRNet, _, _ = refimport.import_generator()
    net = FRNet(in_nc=3, out_nc=3, nf=64, nb=10, degradation=WL['degradation'], scale=SCALE)
    net.load_state_dict(make_params(), strict=True)
    return net.to(device).eval()


def cpu_reference_fps(steps, warmup, n=None):
    """The reference's own CPU path: FRNet.step on `n` lock-stepped clip-frames per step (default: the
    workload's clips_per_gpu, i.e. the SAME step as our arm), fp32, all host threads.  Falls back to the
    operator-for-operator port (oracle/frnet_torchref.py) when TECOGAN_REFERENCE is not set."""
    import torch
    n = CLIPS_PER_GPU if n is None else n
    cores = _host_threads()
    g = torch.Generator().manual_seed(0)
    lr_curr = torch.rand(n, *LR, generator=g)
    lr_prev = torch.rand(n, *LR, generator=g)
    hr_prev = torch.rand(n, LR[0], SCALE * LR[1], SCALE * LR[2], generator=g)
    net = reference_net('cpu')
    if net is not None:
        kind = 'reference'
        step = lambda a, b, c: net.step(a, b, c)
    else:
        from oracle import frnet_torchref as R
        p = make_params()
        kind = 'port'
        step = lambda a, b, c: R.step(p, a, b, c, SCALE, WL['degradation'])
    with torch.no_grad():
        for _ in range(warmup):
            step(lr_curr, lr_prev, hr_prev)
        t0 = time.perf_counter()
        for _ in range(steps):
            hr_prev = step(lr_curr, lr_prev, hr_prev)
        dt = time.perf_counter() - t0
    return n * steps / dt, dt, cores, kind


def run_reference(args, rank):
    if rank != 0:
        return
    n = CLIPS_PER_GPU
    fps, dt, cores, kind = cpu_reference_fps(args.steps, max(args.warmup, 1))
    src = ('unmodified reference FRNet.step from $TECOGAN_REFERENCE (codes/models/networks/tecogan_nets.py:227-252)'
           if kind == 'reference' else 'port oracle/frnet_torchref.py (TECOGAN_REFERENCE not set)')
    sample = (f'{args.steps} steps x {n} lock-stepped clip-frames {"x".join(map(str, LR))} -> x{SCALE} '
              f'(the same step as the GPU arm), {src}, fp32, {cores} host threads')
    line = {
        'impl': 'reference', 'metric': WL['metric'], 'value': fps, 'unit': 'frames/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.gpus),
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def eager_gpu_results(steps, warmup):
    """Context comparator: the UNMODIFIED reference FRNet ($TECOGAN_REFERENCE) on the same B200 through
    PyTorch's CUDA library kernels (cuDNN), same lock-stepped step, CUDA events: fp32, TF32 and fp16
    autocast.  Answers "what does the stock reference get on this GPU" (no B200 number is published)."""
    import torch
    dev = torch.device('cuda', torch.cuda.current_device())
    net = reference_net(dev)
    if net is None:
        return {'unavailable': 'TECOGAN_REFERENCE not set'}
    torch.backends.cudnn.benchmark = True                      # codes/main.py:216
    g = torch.Generator().manual_seed(0)
    n = CLIPS_PER_GPU
    base = [torch.rand(n, *LR, generator=g).to(dev), torch.rand(n, *LR, generator=g).to(dev),
            torch.rand(n, LR[0], SCALE * LR[1], SCALE * LR[2], generator=g).to(dev)]
    out = {}
    for name, tf32, amp in (('fp32', False, False), ('tf32', True, False), ('fp16_autocast', True, True)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        lr_curr, lr_prev, hr_prev = base
        try:
            with torch.no_grad(), torch.autocast('cuda', dtype=torch.float16, enabled=amp):
                for _ in range(max(warmup, 3)):
                    hr_prev = net.step(lr_curr, lr_prev, hr_prev).float()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    hr_prev = net.step(lr_curr, lr_prev, hr_prev).float()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {'ms_per_step': ms, 'frames_per_s': n * 1e3 / ms}
        except Exception as exc:                               # a mode the stock code cannot run
            out[name] = {'error': f'{type(exc).__name__}: {exc}'[:200]}
    torch.backends.cudnn.allow_tf32 = True
    return {'clips_per_step': n, 'steps': steps, 'unit': 'frames/s', 'results': out,
            'note': 'unmodified reference FRNet.step on PyTorch CUDA library kernels (cuDNN), device-resident '
                    'inputs, no uint8/H2D/D2H; includes the reference\'s own CPU-built warp grid + H2D '
                    '(net_utils.py:62-64)'}


def run_eager_gpu(args, rank):
    if rank != 0:
        return
    import torch
    torch.cuda.set_device(0)
    res = eager_gpu_results(args.steps, args.warmup)
    res.update({'impl': 'eager-gpu', 'metric': WL['metric'], 'device': torch.cuda.get_device_name(0)})
    print(json.dumps(res), flush=True)



# =============================================================================== training workloads
# BASELINE.json configs[2] / [3]: TecoGAN 4x BD training (G + D + ping-pong), synthetic REDS-shape 10-frame
# 3x64x64 LR crops, batch 32 per B200; N > 1 = DDP over NCCL (gradient all-reduce), weak scaling.
# The loop is the REFERENCE's own (VSRGANModel.train from $TECOGAN_REFERENCE: discriminator, VGG, losses and
# optimisers stay PyTorch -- SURVEY.md section 2 puts them out of scope); the generator is this repo's
# (forward + backward on the library's kernels) or, for the comparison arms, the reference's.
TRAIN = dict(lr=(3, 64, 64), scale=4, t=10, batch=32, border=4,
             metric={'tecogan': 'train_frames_per_sec_TecoGAN_4xBD_64x64', 'frvsr': 'train_frames_per_sec_FRVSR_4xBD_64x64'})


def train_config(model, batch, world):
    return {'workload': f'{"TecoGAN (G + ST-discriminator + VGG + ping-pong)" if model == "tecogan" else "FRVSR (generator only)"} '
                        f'4x BD training, synthetic REDS-shape {TRAIN["t"]}-frame 3x64x64 LR crops (GT 264x264 incl. the BD '
                        f'border), reference training loop ($TECOGAN_REFERENCE) with the generator under test; DDP/NCCL gradient '
                        f'all-reduce for N > 1 (BASELINE.json configs[2]/[3])',
            'batch_per_gpu': batch, 'global_batch': batch * world, 'frames_per_step': batch * TRAIN['t'] * world,
            'weights': 'seeded random init (no checkpoint; VGG19 = random weights of the same architecture)',
            'l2': 'activations of one step (tens of GB) >> 126 MB L2, no explicit flush'}


def _train_model(model, device, generator, dist_on, rank, world):
    import refimport
    opt = refimport.training_opt(model, device=str(device), dist=dist_on, rank=rank, world_size=world)
    opt['dataset']['train']['crop_size'] = TRAIN['scale'] * TRAIN['lr'][1]
    define_generator = None
    if generator == 'ours':
        import tecogan_b200 as T
        define_generator = T.define_generator
    m = refimport.build_training_model(opt, define_generator)
    m.get_bare_model(m.net_G).load_state_dict(make_params(), strict=True)
    return m


def _train_steps(m, data, steps, sync):
    t0 = time.perf_counter()
    for _ in range(steps):
        m.prepare_training_data({'gt': data})        # H2D of the batch when `data` is pinned host memory
        m.train()                                    # one full iteration (forward, D step, G step)
    sync()
    return time.perf_counter() - t0


def _generator_only_ms(generator, device, batch, reps=3):
    """forward_sequence + backward of the generator alone (19-frame ping-pong sequence as the TecoGAN loop
    feeds it): the part of the step this repo implements, ours vs the reference generator on cuDNN."""
    import torch
    import refimport
    if generator == 'ours':
        import tecogan_b200 as T
        net = T.FRNet(3, 3, 64, 10, 'BD', 4)
    else:
        FRNet, _, _ = refimport.import_generator()
        net = FRNet(in_nc=3, out_nc=3, nf=64, nb=10, degradation='BD', scale=4)
    net.load_state_dict(make_params(), strict=True)
    net = net.to(device).train()
    g = torch.Generator().manual_seed(1)
    lr = torch.rand(batch, 2 * TRAIN['t'] - 1, *TRAIN['lr'], generator=g).to(device)
    out = []
    for i in range(reps + 1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d = net(lr)
        (d['hr_data'].mean() + 0.1 * d['lr_flow'].mean()).backward()
        e1.record()
        torch.cuda.synchronize()
        net.zero_grad(set_to_none=True)
        if i:
            out.append(e0.elapsed_time(e1))
    del net, lr, d
    torch.cuda.empty_cache()
    return statistics.median(out)


def time_train_kernels(dev, pk, batch):
    """Live CUDA-event timing of the two tensor-core kernels of the backward on the training shapes: the weight
    gradient of a 64->64 residual conv over all T*n images of a step (one launch per layer and step) and its data
    gradient on one frame's batch.  FLOPs by the reference counter's convention (2*9*Cin*Cout per pixel)."""
    import torch
    ops = sys.modules['tecogan-pytorch_b200.ops']
    L = sys.modules['tecogan-pytorch_b200.lib']
    c, h, w = TRAIN['lr']
    T_ = 2 * TRAIN['t'] - 1
    wt = torch.randn(64, 64, 3, 3, device=dev) * 0.04
    pc = ops.PackedConv(wt, torch.zeros(64, device=dev), L.CONV_3X3, L.ACT_RELU)
    dgr = ops.PackedDgrad(pc, wt)
    out = {}
    n_img = T_ * batch
    xs = [torch.randn(n_img, h, w, 64, device=dev).half() for _ in range(2)]         # 2 x 319 MB > L2
    dzs = [torch.randn(n_img, h, w, 64, device=dev).half() for _ in range(2)]
    dw = torch.zeros(64, 64, 3, 3, device=dev)
    t = _time_graph(lambda i: ops.wgrad(pc, xs[i], dzs[i], dw), 2, 6, torch)
    fl = RES_CONV_FLOP_PER_PX * n_img * h * w
    out['roofline_wgrad'] = {'kernel': f'wgrad_tcgen05_kernel<conv3x3> (64->64, {n_img} images {h}x{w} = one layer of one step)',
                             'bound': 'tensor', 'achieved': fl / t / 1e12, 'peak': pk['tflops_burst'], 'unit': 'TFLOP/s',
                             'frac': fl / t / 1e12 / pk['tflops_burst'], 'us_per_launch': t * 1e6, 'flop_per_launch': fl,
                             'traffic': ncu_traffic('wgrad_train')[0], 'traffic_src': ncu_traffic('wgrad_train')[1],
                             'how': '6 launches in one CUDA graph over 2 rotating operand sets (1.3 GB > L2), CUDA events'}
    nb = 8
    xd = [torch.randn(batch, h, w, 64, device=dev).half() for _ in range(nb)]
    yd = [torch.empty_like(v) for v in xd]
    md = [torch.randn(batch, h, w, 64, device=dev).half() for _ in range(nb)]
    t = _time_graph(lambda i: dgr(xd[i], y=yd[i], mask=md[i], mask_act=L.ACT_RELU), nb, 40, torch)
    fl = RES_CONV_FLOP_PER_PX * batch * h * w
    out['roofline_dgrad'] = {'kernel': f'conv_tcgen05_kernel<conv3x3, halo, BWD> (dgrad 64->64 * ReLU\'(mask), {batch} images {h}x{w})',
                             'bound': 'tensor', 'achieved': fl / t / 1e12, 'peak': pk['tflops_burst'], 'unit': 'TFLOP/s',
                             'frac': fl / t / 1e12 / pk['tflops_burst'], 'us_per_launch': t * 1e6, 'flop_per_launch': fl,
                             'traffic': None, 'how': f'40 launches in one CUDA graph over {nb} rotating buffer sets, CUDA events'}
    return out


def run_train(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    model = 'frvsr' if args.workload == 'train-frvsr' else 'tecogan'
    impl = args.impl
    K, Wm = args.steps, max(args.warmup, 1)
    import refimport
    if not refimport.available():
        sys.exit(f'bench.py --workload {args.workload} drives the reference\'s own training loop (VSRModel / '
                 f'VSRGANModel, discriminator, VGG, losses): set {refimport.ENV} to the root of a TecoGAN-PyTorch checkout')
    if impl == 'reference':
        # the reference's own training step on the host cores: a bounded sample (1 clip per step)
        if rank != 0:
            return
        cores = _host_threads()
        n = 1
        m = _train_model(model, 'cpu', 'reference', False, 0, 1)
        data = torch.rand(n, TRAIN['t'], 3, 264, 264, generator=torch.Generator().manual_seed(0))
        steps = K
        _train_steps(m, data, 1, lambda: None)
        dt = _train_steps(m, data, steps, lambda: None)
        fps = n * TRAIN['t'] * steps / dt
        line = {'impl': 'reference', 'metric': TRAIN['metric'][model], 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
                'steps': steps, 'warmup': 1, 'ms_per_step': 1e3 * dt / steps, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': train_config(model, args.batch or TRAIN['batch'], args.gpus),
                'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'reference',
                                 'sample': f'{steps} training iterations of {n} clip ({TRAIN["t"]} frames, 64x64 LR) with the unmodified '
                                           f'reference ($TECOGAN_REFERENCE) on {cores} host threads -- a bounded sample of the batch'},
                'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line), flush=True)
        return
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback exists)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')
        dist.init_process_group('nccl', device_id=dev)
    ops = None
    if impl == 'ours':
        import tecogan_b200 as T  # noqa: F401
        ops = sys.modules['tecogan-pytorch_b200.ops']
    torch.backends.cudnn.benchmark = True
    batch = args.batch or TRAIN['batch']
    m = _train_model(model, dev, 'ours' if impl == 'ours' else 'reference', world > 1, rank, world)
    g = torch.Generator().manual_seed(100 + rank)
    host = torch.rand(batch, TRAIN['t'], 3, 264, 264, generator=g).pin_memory()
    resident = host.to(dev)
    sync = lambda: torch.cuda.synchronize()
    _train_steps(m, resident, Wm, sync)
    torch.cuda.reset_peak_memory_stats()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ops.LAUNCH_COUNT if ops else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    _train_steps(m, resident, K, sync)
    e1.record()
    torch.cuda.synchronize()
    launches = (ops.LAUNCH_COUNT - l0) if ops else 0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    value = world * batch * TRAIN['t'] * K / (float(ms.item()) * 1e-3)
    # end to end: the batch comes from pinned host memory every iteration (H2D inside the timed region);
    # the losses the loop logs come back through .item() (D2H)
    if world > 1:
        dist.barrier()
    dt = torch.tensor([_train_steps(m, host, K, sync)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e = world * batch * TRAIN['t'] * K / float(dt.item())
    clocks = sampler.stop() if rank == 0 else None
    peak_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    log = {k: float(v) for k, v in m.log_dict.items()}
    line = None
    if rank == 0:
        line = {'metric': TRAIN['metric'][model], 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
                'ms_per_step': float(ms.item()) / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f16' if impl == 'ours' else 'f32', 'data': 'synthetic', 'config': train_config(model, batch, world),
                'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': host.numel() * 4, 'd2h_bytes_per_step': 4 * len(log),
                        'api': 'reference VSR(GAN)Model.prepare_training_data(pinned gt) + .train() with define_generator = tecogan_b200'},
                'gpu_launches': launches, 'launches_per_step': launches / K if K else 0, 'clocks': clocks,
                'peak_memory_gb': peak_gb, 'last_log': log,
                'generator': 'tecogan_b200 (fp16 tcgen05 forward + backward)' if impl == 'ours' else 'reference FRNet on cuDNN (fp32/TF32)'}
        if impl != 'ours':
            line['impl'] = 'eager-gpu'
    del m
    torch.cuda.empty_cache()
    if rank == 0 and impl == 'ours':
        line.update(time_train_kernels(dev, peaks(), batch))
    if rank == 0 and world == 1 and impl == 'ours' and not args.no_eager:
        gb = min(batch, 8)
        ours_ms = _generator_only_ms('ours', dev, gb)
        ref_ms = _generator_only_ms('reference', dev, gb)
        line['generator_fwd_bwd'] = {'batch': gb, 'frames': 2 * TRAIN['t'] - 1, 'ours_ms': ours_ms, 'reference_cudnn_ms': ref_ms,
                                     'speedup': ref_ms / ours_ms,
                                     'note': 'forward_sequence + backward of the generator alone on the same B200'}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)


# =============================================================================== our arm
def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, taken from the latest
    `ncu --set full` capture summarised in profiles/ncu_traffic.json (written by
    tools/summarize_ncu.py --traffic-json from the .ncu-rep of the CURRENT kernels); None when that
    kernel has no capture -- never a remembered constant."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        ent = json.load(open(path)).get(kernel_key)
    except Exception:
        ent = None
    if not ent:
        return None, None
    return float(ent['dram_bytes_per_launch']), ent.get('src')



def _time_graph(fn, nbuf, reps, torch):
    """Average device time of one fn(i) launch: `reps` launches over `nbuf` rotating buffer sets are
    captured in a CUDA graph (so the number is the kernel, not the Python launch rate) and the
    replay is timed with CUDA events; 3 untimed replays first."""
    for i in range(nbuf):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps):
            fn(i % nbuf)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def time_kernels(dev, pk):
    """Live CUDA-event timing of the two roofline kernels on rotating buffers larger than L2."""
    import torch
    import tecogan_b200 as T
    ops = sys.modules['tecogan-pytorch_b200.ops']
    L = sys.modules['tecogan-pytorch_b200.lib']
    n, (c, h, w) = CLIPS_PER_GPU, LR
    out = {}
    reps = 60
    mb = n * h * w * 128 / 1e6                    # one 64-channel fp16 activation map of a step, MB
    # ---- dominant kernel: SRNet residual-block conv 64->64 (+bias, ReLU), n frames per launch
    wt = torch.randn(64, 64, 3, 3, device=dev) * 0.04
    pc = ops.PackedConv(wt, torch.zeros(64, device=dev), L.CONV_3X3, L.ACT_RELU)
    nbuf = max(3, int(220 / mb) + 1)            # bd4: 10 x (22 MB in + 22 MB out) = 440 MB > 126 MB L2
    xs = [torch.randn(n, h, w, 64, device=dev).half() for _ in range(nbuf)]
    ys = [torch.empty_like(x) for x in xs]
    t_conv = _time_graph(lambda i: pc(xs[i], y=ys[i]), nbuf, reps, torch)
    flops = RES_CONV_FLOP_PER_PX * n * h * w
    out['roofline'] = {
        'kernel': f'conv_tcgen05_kernel<conv3x3, halo> (SRNet resblock conv 64->64, {n} frames/launch)',
        'bound': 'tensor', 'achieved': flops / t_conv / 1e12, 'peak': pk['tflops_burst'], 'unit': 'TFLOP/s',
        'frac': flops / t_conv / 1e12 / pk['tflops_burst'],
        'traffic': ncu_traffic('conv_single_' + WL_KEY)[0], 'traffic_src': ncu_traffic('conv_single_' + WL_KEY)[1],
        'us_per_launch': t_conv * 1e6, 'flop_per_launch': flops,
        'peak_src': pk['src'] + ' burst (kernel timed alone)',
        'how': f'{reps} launches in one CUDA graph, {nbuf} rotating in/out pairs ({2 * nbuf * mb:.0f} MB > L2), CUDA events'}
    out['roofline_conv_single'] = out['roofline']
    # ---- dominant kernel of the step: conv_in + 10 residual blocks as ONE persistent launch
    if ops.chain_enabled():
        nl = 21
        pcs = [ops.PackedConv(torch.randn(64, 64, 3, 3, device=dev) * 0.04, torch.zeros(64, device=dev), L.CONV_3X3,
                              L.ACT_RELU if (i == 0 or i % 2 == 1) else L.ACT_NONE) for i in range(nl)]
        specs = [(pcs[0], 0, 1, None)]
        for b in range(10):
            specs += [(pcs[1 + 2 * b], 1, 2, None), (pcs[2 + 2 * b], 2, 1, 1)]
        chain = ops.ConvChain(specs)
        nb3 = min(3, nbuf)                       # bd4: 3 x (22 MB in + 2 x 22 MB work) = 198 MB > 126 MB L2
        sets = [[xs[i], ys[i], torch.empty_like(xs[i])] for i in range(nb3)]
        creps = 12
        t_chain = _time_graph(lambda i: chain(sets[i]), nb3, creps, torch)
        cflops = flops * nl
        out['roofline'] = {
            'kernel': 'conv_chain_kernel (SRNet conv_in + 10 residual blocks = 21 convs 64->64 in one persistent '
                      f'launch, {n} frames/launch)',
            'bound': 'tensor', 'achieved': cflops / t_chain / 1e12, 'peak': pk['tflops_burst'], 'unit': 'TFLOP/s',
            'frac': cflops / t_chain / 1e12 / pk['tflops_burst'],
            'traffic': ncu_traffic('conv_chain_' + WL_KEY)[0], 'traffic_src': ncu_traffic('conv_chain_' + WL_KEY)[1],
            'us_per_launch': t_chain * 1e6, 'us_per_layer': t_chain * 1e6 / nl, 'flop_per_launch': cflops,
            'peak_src': pk['src'] + ' burst (kernel timed alone)',
            'how': f'{creps} launches in one CUDA graph, {nb3} rotating buffer sets ({3 * nb3 * mb:.0f} MB > L2), CUDA events'}
        del sets
    del xs, ys
    # ---- fused warp + space_to_depth + concat, HR flow given (BASELINE.md byte formula)
    H, W = SCALE * h, SCALE * w
    nb2 = 6                                      # bd4: 6 x 4 frames x ~20 MB = 470 MB > L2
    hp = [torch.rand(n, c, H, W, device=dev) for _ in range(nb2)]
    fl = [(torch.rand(n, 2, H, W, device=dev) - 0.5) * 6 for _ in range(nb2)]
    lr = [torch.rand(n, c, h, w, device=dev) for _ in range(nb2)]
    oo = [torch.empty(n, h, w, 64, dtype=torch.float16, device=dev) for _ in range(nb2)]
    lf = [(torch.rand(n, 2, h // 8 * 8, w // 8 * 8, device=dev) - 0.5) * 2 for _ in range(nb2)]
    up_mode = L.UP_BICUBIC if WL['degradation'] == 'BD' else L.UP_BILINEAR
    for variant in ('hrflow', 'lrflow'):
        if variant == 'hrflow':
            call = lambda i: ops.warp_s2d_concat_hrflow(hp[i], fl[i], lr[i], SCALE, out=oo[i])
        else:
            call = lambda i: ops.warp_s2d_concat_lrflow(hp[i], lf[i], lr[i], SCALE, up_mode, out=oo[i])
        t = _time_graph(call, nb2, reps, torch)
        alg = WL['warp_bytes_per_frame'] * n
        moved = n * (c * H * W * 4 + (2 * H * W * 4 if variant == 'hrflow' else 2 * (h // 8 * 8) * (w // 8 * 8) * 4)
                     + c * h * w * 4 + h * w * 64 * 2)
        out['roofline_warp' if variant == 'hrflow' else 'roofline_warp_fused_lrflow'] = {
            'kernel': f'warp_s2d_concat_kernel<{SCALE},{variant}> ({n} frames/launch)', 'bound': 'hbm',
            'achieved': alg / t / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': alg / t / 1e9 / pk['hbm_gbs'],
            'traffic': ncu_traffic(f'warp_{variant}_' + WL_KEY)[0], 'traffic_src': ncu_traffic(f'warp_{variant}_' + WL_KEY)[1],
            'us_per_launch': t * 1e6, 'algorithmic_bytes_per_launch': alg,
            'bytes_actually_moved_per_launch': moved, 'moved_gbs': moved / t / 1e9,
            'peak_src': pk['src'], 'how': f'{reps} launches in one CUDA graph, {nb2} rotating buffer sets > L2'}
    return out


DUMP_U8_SAMPLES = 1 << 20


def dump_outputs(out_dir, hr, u8):
    """What the last timed step handed its caller: the HR frames hr_curr [n,c,H,W] (fp32, whole) and the
    quantised frames [n,H,W,c] (uint8 -> float32, a fixed seeded sample of DUMP_U8_SAMPLES elements, with
    their flat indices) -- together under 64 MB, so two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    u8 = u8.cpu().numpy().reshape(-1)
    idx = np.sort(np.random.default_rng(0).choice(u8.size, size=min(DUMP_U8_SAMPLES, u8.size), replace=False))
    np.save(os.path.join(out_dir, 'hr_curr.npy'), hr.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, 'hr_u8_sample.npy'), u8[idx].astype(np.float32))
    np.save(os.path.join(out_dir, 'hr_u8_sample_index.npy'), idx.astype(np.float64))


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import tecogan_b200 as T
    ops = sys.modules['tecogan-pytorch_b200.ops']

    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback exists)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')          # keep stdout to the one JSON line
        dist.init_process_group('nccl', device_id=dev)
    pk = peaks()

    net = T.FRNet(3, 3, 64, 10, WL['degradation'], SCALE)
    net.load_state_dict(make_params(), strict=True)
    net = net.to(dev).eval()
    n, (c, h, w) = CLIPS_PER_GPU, LR
    K, Wm = args.steps, max(args.warmup, 3)

    # ---------------- device-resident throughput: graph replay of the recurrent step
    eng = T.ClipEngine(net, n, c, h, w, dev)
    clips = synthetic_clips(n, 8, seed=rank).to(dev)           # [n,8,c,h,w] resident in HBM
    frames = clips.transpose(0, 1).contiguous()

    def step(i):
        p = i & 1
        eng.lr[p].copy_(frames[i % frames.shape[0]])           # device->device, 2 MB
        eng.run_frame(p)

    eng.reset()
    for i in range(Wm):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.LAUNCH_COUNT
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(K):
        step(Wm + i)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * n * K / (ms_max * 1e-3)
    launches_per_step = eng.launches_per_step + 0               # kernels inside one graph replay
    gpu_launches = launches_per_step * K
    if args.dump_outputs and rank == 0:
        p_last = (Wm + K - 1) & 1
        dump_outputs(args.dump_outputs, eng.hr[p_last], eng.u8[p_last])

    if args.profile_only:          # under ncu: only the step loop, no JSON line
        if rank == 0:
            sampler.stop()
        return
    # ---------------- sustained: >= args.sustain_s seconds of back-to-back steps (clocks settle under load)
    sustained = None
    if args.sustain_s > 0:
        n_sus = max(K, int(args.sustain_s / (ms_max / K * 1e-3)) + 1)
        sus_sampler = ClockSampler(local_rank)
        if world > 1:
            dist.barrier()
        if rank == 0:
            sus_sampler.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s0.record()
        for i in range(n_sus):
            step(i)
        s1.record()
        torch.cuda.synchronize()
        ts = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        if rank == 0:
            sus_ms = float(ts.item())
            sustained = {'value': world * n * n_sus / (sus_ms * 1e-3), 'unit': 'frames/s', 'steps': n_sus,
                         'seconds': sus_ms * 1e-3, 'ms_per_step': sus_ms / n_sus, 'clocks': sus_sampler.stop(),
                         'model_tflops': world * n * n_sus / (sus_ms * 1e-3) * WL['flop_per_frame'] / 1e12 / world,
                         'how': 'same device-resident step loop as `value`, run for >= %.0f s' % args.sustain_s}

    # ---------------- end to end through FRNet.infer_sequence with host buffers
    t_e2e = K if WL_KEY == 'bd4' else 30                   # config 5 is quoted on 30-frame clips
    host_clips = synthetic_clips(n, t_e2e, seed=100 + rank).pin_memory()     # [n,T,c,h,w] pinned
    net.infer_sequence(host_clips[:, :4], dev)                                # warm-up
    net.infer_sequence(host_clips, dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    w0 = time.perf_counter()
    seq = net.infer_sequence(host_clips, dev)                                 # uint8 [n,T,H,W,c] on host
    torch.cuda.synchronize()
    w1 = time.perf_counter()
    assert seq.shape == (n, t_e2e, SCALE * h, SCALE * w, c) and str(seq.dtype) == 'uint8'
    te = torch.tensor([w1 - w0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * n * t_e2e / float(te.item())
    clocks = sampler.stop() if rank == 0 else None     # sampled over both timed regions

    line = None
    if rank == 0:
        del eng, clips, frames
        T.engine.release_engines(net)
        torch.cuda.empty_cache()
        roof = time_kernels(dev, pk)
        cpu, eager = None, None
        if world == 1:
            steps_cpu = 6 if WL_KEY == 'bd4' else 3
            fps, dt, cores, kind = cpu_reference_fps(steps_cpu, 1)
            cpu = {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
                   'sample': f'{steps_cpu} steps x {n} lock-stepped clip-frames {"x".join(map(str, LR))} (fp32, '
                             + ('unmodified reference FRNet.step from $TECOGAN_REFERENCE' if kind == 'reference' else
                                'port oracle/frnet_torchref.py') + f'), {dt:.1f} s of CPU work'}
            if not args.no_eager:
                eager = eager_gpu_results(10, 3)
        line = {
            'metric': WL['metric'], 'value': value, 'unit': 'frames/s', 'n_gpus': world,
            'steps': K, 'warmup': Wm, 'ms_per_step': ms_max / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': (value / PUBLISHED_FPS_1080TI) if WL_KEY == 'bd4' else None, 'dtype': 'f16',
            'data': 'synthetic',
            'config': workload_config(world),
            'notes': {
                'l2': 'per-step working set ~1.3 GB of activations (HR 64-channel map alone 351 MB for 4 frames) '
                      '>> 126 MB L2; no explicit flush', 'conv_impl': ops.default_conv_impl(),
                'baseline_note': 'vs_baseline = value / 27 FPS published for 1x GTX 1080 Ti, batch 1, 4x BD '
                                 '(resources/benchmark.png); no B200 number is published'},
            'gflop_per_frame': WL['flop_per_frame'] / 1e9,
            'model_tflops': value * WL['flop_per_frame'] / 1e12 / world,
            'model_tensor_frac_of_sustained': value * WL['flop_per_frame'] / 1e12 / world / pk['tflops_sustained'],
            'e2e': {'value': e2e_val, 'unit': 'frames/s', 'h2d_bytes_per_step': n * c * h * w * 4,
                    'd2h_bytes_per_step': n * SCALE * h * SCALE * w * c, 'steps': t_e2e,
                    'api': 'FRNet.infer_sequence(lr_data[n,t,c,h,w] pinned host) -> uint8 ndarray [n,t,H,W,c]'},
            'gpu_launches': gpu_launches, 'launches_per_step': launches_per_step,
            'clocks': clocks,
        }
        line.update(roof)
        if sustained is not None:
            line['sustained'] = sustained
        if cpu is not None:
            line['cpu_baseline'] = cpu
        if eager is not None:
            line['gpu_eager_baseline'] = eager
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50,
                    help='timed steps (recurrent frames of the lock-stepped clips, or training iterations); also the '
                         'frames of the e2e clip for bd4 -- bi2\'s e2e block always runs its 30-frame clips (config 5)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'eager-gpu'])
    ap.add_argument('--workload', default='bd4', choices=sorted(WORKLOADS) + ['train', 'train-frvsr'],
                    help='bd4 = BASELINE configs[1] (headline); bi2 = configs[4] (2x BI 268x640, 30-frame clips); '
                         'train = configs[2]/[3] (TecoGAN training step, DDP for N > 1); train-frvsr = generator-only losses')
    ap.add_argument('--batch', type=int, default=0, help='training workloads: clips per GPU (default 32)')
    ap.add_argument('--sustain-s', type=float, default=3.0, help='seconds of the sustained block (0 = skip)')
    ap.add_argument('--no-eager', action='store_true', help='skip the gpu_eager_baseline block (N=1 only)')
    ap.add_argument('--profile-only', action='store_true',
                    help='run only the device-resident step loop (for ncu captures); prints nothing')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last timed step as DIR/<name>.npy '
                         '(inference workloads of --impl ours; rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.workload.startswith('train')):
        ap.error('--dump-outputs writes the outputs of the timed inference step: --impl ours, --workload bd4 or bi2')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.workload.startswith('train'):
        return run_train(args, rank, world, local_rank)
    select_workload(args.workload)
    if args.impl == 'reference':
        return run_reference(args, rank)
    if args.impl == 'eager-gpu':
        return run_eager_gpu(args, rank)
    run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
