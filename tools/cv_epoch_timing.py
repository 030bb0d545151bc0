"""Developer tool: what the tensor-core critic (central_value_config mixed_precision: True) buys on an mjlab-like central-value workload.

Times A2CAgentCV.train_epoch() on the on-GPU synthetic env with the critic on the fp32 CUDA-core kernels and on the tensor cores, the two
agents alternating within one process, and CentralValueNet.train_net() on its own.  Defaults follow configs/mjlab/ppo_go1_velocity.yaml:
4096 envs x horizon 24, minibatch 24576, actor and critic MLP [512, 256, 128], 5 actor and 5 critic mini-epochs, adaptive LR with
schedule_type standard.  The synthetic env has no privileged observation group, so the critic reads the actor's observations through the
state_space fallback; the observation / action sizes are illustrative, not go1's.

    python tools/cv_epoch_timing.py --out DIR [--epochs 8 --rounds 3 --warmup 3 --actor-mp absent true]

Each timed epoch is bracketed by CUDA events; 256 MiB are written between epochs (outside the events) so no epoch starts on the previous
one's L2.  Writes DIR/cv_epoch_timing.json (card name and power limit included) and prints it."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit,clocks.max.sm',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:          # the name from the runtime, the limit unknown
        return {'name': torch.cuda.get_device_name(), 'power_limit': 'unavailable (%s)' % type(e).__name__}


def params(a, critic_mp, actor_mp, train_dir):
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': list(a.units), 'activation': 'elu', 'initializer': {'name': 'default'}}}
    cv = {'minibatch_size': a.cv_minibatch, 'mini_epochs': a.cv_mini_epochs, 'learning_rate': 5e-4, 'clip_value': True, 'normalize_input': True,
          'mixed_precision': critic_mp,
          'network': {'name': 'actor_critic', 'central_value': True,
                      'mlp': {'units': list(a.cv_units), 'activation': 'elu', 'initializer': {'name': 'default'}}}}
    config = {'name': 'cv_timing', 'env_name': 'b200_synthetic', 'reward_shaper': {'scale_value': 1.0}, 'device': 'cuda:0',
              'normalize_input': True, 'normalize_value': True, 'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95,
              'learning_rate': 1e-3, 'lr_schedule': 'adaptive', 'kl_threshold': 0.016, 'schedule_type': 'standard', 'grad_norm': 1.0,
              'entropy_coef': 0.0, 'truncate_grads': True, 'e_clip': 0.2, 'clip_value': False, 'use_smooth_clamp': True,
              'bound_loss_type': 'regularisation', 'bounds_loss_coef': 0.0, 'max_epochs': -1, 'num_actors': a.envs, 'horizon_length': a.horizon,
              'minibatch_size': a.minibatch, 'mini_epochs': a.mini_epochs, 'critic_coef': 1, 'print_stats': False, 'train_dir': train_dir,
              'central_value_config': cv, 'env_config': {'obs_dim': a.obs_dim, 'act_dim': a.act_dim, 'device': 'cuda:0', 'seed': 5}}
    if actor_mp != 'absent':
        config['mixed_precision'] = actor_mp == 'true'
    return {'seed': 5, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network, 'config': config}


def build(a, critic_mp, actor_mp, train_dir):
    from rl_games_b200.runner import Runner
    r = Runner()
    r.load({'params': params(a, critic_mp, actor_mp, train_dir)})
    agent = r.algo_factory.create(r.algo_name, base_name='cv_timing', params=r.params)
    agent.init_tensors()
    agent.obs = agent.env_reset()
    assert agent.central_value_net.gemm_tc == critic_mp
    return agent


def time_epochs(agent, n, flush):
    from rl_games_b200 import ops
    out = []
    for _ in range(n):
        ops.fill_u32(flush, 1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        agent.epoch_num += 1
        agent.train_epoch()
        e.record()
        out.append((s, e))
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in out]


def time_train_net(agent, n, flush):
    """the critic's update phase alone, on the dataset the agent's last epoch left"""
    from rl_games_b200 import ops
    cv, out = agent.central_value_net, []
    for _ in range(n):
        ops.fill_u32(flush, 1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        cv.train_net(agent.old_values_n, agent.returns_n, agent.valid)
        e.record()
        out.append((s, e))
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in out]


def summary(xs):
    return {'median_ms': statistics.median(xs), 'min_ms': min(xs), 'max_ms': max(xs), 'n': len(xs)}


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    p.add_argument('--out', required=True)
    p.add_argument('--envs', type=int, default=4096)
    p.add_argument('--horizon', type=int, default=24)
    p.add_argument('--minibatch', type=int, default=24576)
    p.add_argument('--mini-epochs', type=int, default=5)
    p.add_argument('--cv-minibatch', type=int, default=24576)
    p.add_argument('--cv-mini-epochs', type=int, default=5)
    p.add_argument('--units', type=int, nargs='+', default=[512, 256, 128])
    p.add_argument('--cv-units', type=int, nargs='+', default=[512, 256, 128])
    p.add_argument('--obs-dim', type=int, default=64)
    p.add_argument('--act-dim', type=int, default=12)
    p.add_argument('--epochs', type=int, default=8, help='timed epochs per arm and round')
    p.add_argument('--rounds', type=int, default=3, help='alternations of the two critic arms')
    p.add_argument('--warmup', type=int, default=3)
    p.add_argument('--actor-mp', nargs='+', default=['absent', 'true'], choices=['absent', 'true', 'false'],
                   help="the agent-level mixed_precision key ('absent' = as the mjlab YAMLs ship)")
    a = p.parse_args()
    if not torch.cuda.is_available():
        sys.exit('cv_epoch_timing needs a CUDA device')
    torch.cuda.set_device(0)
    tmp = tempfile.mkdtemp(prefix='b200_cv_timing_')
    flush = torch.empty(64 << 20, dtype=torch.int32, device='cuda:0')          # 256 MiB, overwritten between timed epochs
    res = {'card': card(), 'workload': {k: getattr(a, k) for k in ('envs', 'horizon', 'minibatch', 'mini_epochs', 'cv_minibatch', 'cv_mini_epochs',
                                                                      'units', 'cv_units', 'obs_dim', 'act_dim')},
           'note': 'synthetic on-GPU env; the critic reads the observations (state_space fallback); dimensions illustrative, not go1\'s',
           'l2': 'flushed between timed epochs / train_net calls (256 MiB write outside the event pairs)', 'runs': []}
    try:
        for actor_mp in a.actor_mp:
            agents = {mp: build(a, mp, actor_mp, tmp) for mp in (False, True)}
            actor_path = 'fused tcgen05' if agents[True].use_tc else ('layer-wise tcgen05' if agents[True].gemm_tc else 'fp32')
            for ag in agents.values():
                time_epochs(ag, a.warmup, flush)
            ep = {False: [], True: []}
            for r in range(a.rounds):
                for mp in ((False, True) if r % 2 == 0 else (True, False)):
                    ep[mp] += time_epochs(agents[mp], a.epochs, flush)
            tn = {False: [], True: []}
            for r in range(a.rounds):
                for mp in ((False, True) if r % 2 == 0 else (True, False)):
                    tn[mp] += time_train_net(agents[mp], a.epochs, flush)
            run = {'actor_mixed_precision': actor_mp, 'actor_kernels': actor_path}
            for mp, name in ((False, 'critic_fp32'), (True, 'critic_tc')):
                run[name] = {'epoch': summary(ep[mp]), 'train_net': summary(tn[mp])}
            run['epoch_speedup'] = run['critic_fp32']['epoch']['median_ms'] / run['critic_tc']['epoch']['median_ms']
            run['train_net_speedup'] = run['critic_fp32']['train_net']['median_ms'] / run['critic_tc']['train_net']['median_ms']
            res['runs'].append(run)
            del agents
            torch.cuda.empty_cache()
    finally:
        shutil.rmtree(tmp, True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'cv_epoch_timing.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
