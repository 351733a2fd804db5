"""2-rank DDP check of the training path on real GPUs (run by hand on a 2-GPU box; the 1-GPU pytest suite covers
DDP with world size 1 in `reference_training_integration_ddp`):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tests/ddp_train_check.py

Each rank runs one iteration of the reference's FRVSR training loop (gpu_checks.frvsr_train_step, nb=2) around
tecogan_b200's generator wrapped in DistributedDataParallel as base_model.model_to_device wraps it, on DIFFERENT
clips; the ranks then verify that (a) every parameter gradient is finite and identical on both ranks (NCCL
all-reduce happened on gradients our backward kernels produced), (b) it equals the mean of the two single-rank
gradients computed without DDP on the same clips, (c) the updated weights agree across ranks.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = f'cuda:{local}'
    dist.init_process_group('nccl', device_id=torch.device(dev))
    import gpu_checks
    import synthetic
    import tecogan_b200 as T
    p = synthetic.make_frnet_params(41, nb=2, gain=1.5)
    clips = [torch.from_numpy(np.random.default_rng(70 + r).uniform(0, 1, (2, 4, 3, 72, 72)).astype(np.float32))
             for r in range(world)]

    def run(use_ddp, data):
        net = T.FRNet(3, 3, 64, 2, 'BD', 4).to(dev)
        net.load_state_dict(p, strict=True)
        log = gpu_checks.frvsr_train_step(gpu_checks.ddp_wrap(net) if use_ddp else net, data.to(dev))
        return ({k: v.grad.detach().clone() for k, v in net.named_parameters()},
                {k: v.detach().clone() for k, v in net.named_parameters()}, log)

    g_ddp, w_ddp, log = run(True, clips[rank])
    singles = [run(False, clips[r])[0] for r in range(world)]
    worst_sync, worst_mean, worst_w = 0.0, 0.0, 0.0
    for k, g in g_ddp.items():
        assert torch.isfinite(g).all(), k
        gathered = [torch.empty_like(g) for _ in range(world)]
        dist.all_gather(gathered, g)
        worst_sync = max(worst_sync, float((gathered[0] - gathered[1]).abs().max()))
        mean = sum(s[k] for s in singles) / world
        worst_mean = max(worst_mean, float((g - mean).norm() / mean.norm().clamp_min(1e-20)))
        wg = [torch.empty_like(w_ddp[k]) for _ in range(world)]
        dist.all_gather(wg, w_ddp[k])
        worst_w = max(worst_w, float((wg[0] - wg[1]).abs().max()))
    if rank == 0:
        print({'world': world, 'grad_max_abs_diff_across_ranks': worst_sync, 'ddp_vs_mean_of_single_rank_rel_l2': worst_mean,
               'weights_max_abs_diff_across_ranks': worst_w, 'log': log})
    # fp32 atomics make the backward's summation order non-deterministic: tolerance, not bit equality, vs the mean
    assert worst_sync == 0.0 and worst_w == 0.0 and worst_mean <= 2e-3, (worst_sync, worst_w, worst_mean)
    dist.destroy_process_group()
    if rank == 0:
        print('DDP_TRAIN_CHECK_OK')


if __name__ == '__main__':
    main()
