"""Multi-GPU correctness + timing check (run under torchrun on the GPU box):
   torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/mgpu_check.py
Checks after a few epochs that every rank holds byte-identical parameters, Adam moments, lr and (pooled) running stats,
for the eager and the CUDA-graph update paths, and prints per-epoch device time."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def main():
    rank, local_rank, world = bench.dist_info()
    torch.cuda.set_device(local_rank)
    dev = f'cuda:{local_rank}'
    out = {}
    ref_flat = None
    for mode, graph, fused, split in (('nccl_eager', False, False, False), ('nccl_graph', True, False, False),
                                      ('fused_two_launch_graph', True, True, False), ('fused_one_launch_graph', True, True, True)):
        w = dict(bench.WORKLOADS['c2'])
        from rl_games_b200.runner import Runner
        r = Runner()
        p = bench.make_params(w, dev, 'b200_synthetic', True, graph=True)
        p['config']['b200_cuda_graph_multi_gpu'] = graph
        p['config']['b200_fused_allreduce'] = fused
        p['config']['b200_fused_split_allreduce'] = split
        r.load({'params': p})
        agent = r.algo_factory.create(r.algo_name, base_name='mgpu', params=r.params)
        agent.init_tensors()
        agent.obs = agent.env_reset()
        dist.broadcast(agent.model.flat, 0)
        agent._repack()
        ts, _ = bench.timed_epochs(agent, 6, None, world)
        flat = torch.cat([agent.model.flat, agent.model.exp_avg, agent.model.exp_avg_sq, agent.opt_state.float(),
                          agent.model.running_mean_std.running_mean.float(), agent.model.running_mean_std.running_var.float(),
                          agent.model.value_mean_std.running_mean.float()])
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        same = all(torch.equal(gathered[0], g) for g in gathered[1:])
        cnt = torch.tensor([int(agent.model.running_mean_std.count)], device=dev)
        cnts = [torch.empty_like(cnt) for _ in range(world)]
        dist.all_gather(cnts, cnt)
        if ref_flat is None:
            ref_flat = agent.model.flat.clone()
        out[mode] = {'fused_allreduce': agent.fused_allreduce, 'fused_split_allreduce': bool(fused and split), 'max_abs_diff_vs_nccl_eager': float((agent.model.flat - ref_flat).abs().max()),
                     'identical_across_ranks': bool(same), 'obs_count': [int(c) for c in cnts],
                                              'ms_per_epoch': [round(t, 3) for t in ts], 'lr': agent.last_lr,
                                              'finite': bool(torch.isfinite(agent.model.flat).all()),
                                              'graph_captured': (agent._graph_update is not None) or (agent._graph_epoch is not None)}
        agent._graph_update = agent._graph_epoch = None
        del agent
        torch.cuda.synchronize()
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
