"""What the continuous (agent.A2CAgent) and the discrete (agent_discrete.DiscreteA2CAgent) agents share -- the reference's A2CBase
(common/a2c_common.py): config parsing and validation, multi-GPU and device setup, env creation, the LR scheduler choice, run
directories and the summary writer, the device-resident episode meters, the cross-rank normaliser sync, the outer train() loop, summary
scalars and checkpoints.

A subclass refuses what it does not build before ``super().__init__``, parses its own keys (action space and model, precision) after
it, ends its ``__init__`` with ``self.algo_observer.after_init(self)``, and provides init_tensors / env_reset / train_epoch and two
optimiser hooks for checkpoints: ``_optimizer_lr()`` (the lr the optimizer state dict records) and ``_restore_optimizer(lr, step)``
(hands a checkpoint's optimizer lr -- None if it has none -- and step to the device optimiser state).
"""
import os
from datetime import datetime

import numpy as np
import torch
import torch.distributed as dist

from .common import AdaptiveScheduler, DefaultAlgoObserver, DefaultRewardsShaper, IdentityScheduler, LinearScheduler, create_vec_env, \
    make_summary_writer
from .dist_utils import PackedStatsSync
from .model import CompileTolerantModel, resolve_device

STATS_SYNC_MODES = ('pooled', 'broadcast')


class _MeterView:
    """torch_ext.AverageMeter look-alike over the device-resident meter block (torch_ext.py:326-352)."""

    def __init__(self, agent, slot):
        self._a, self._slot = agent, slot

    @property
    def current_size(self):
        return int(self._a._meter_host()[3])

    def __len__(self):
        return self.current_size

    def get_mean(self):
        return np.asarray([self._a._meter_host()[self._slot]], dtype=np.float32)

    @property
    def mean(self):
        return torch.tensor([self._a._meter_host()[self._slot]], dtype=torch.float32)

    def clear(self):
        self._a.meter.zero_()
        self._a._meter_cache = None


class A2CBase(CompileTolerantModel):
    def __init__(self, base_name, params):
        self.config = config = params['config']
        # a2c_common.py:172-188: PBT runs carry the policy's index in the experiment name
        pbt_str = f'_pbt_{config["pbt_idx"]:02d}' if config.get('population_based_training', False) else ''
        self.experiment_name = config.get('full_experiment_name') or (config['name'] + pbt_str + datetime.now().strftime("_%d-%H-%M-%S"))
        config.setdefault('features', {})
        self.algo_observer = config['features'].get('observer') or DefaultAlgoObserver()
        self.algo_observer.before_init(base_name, config, self.experiment_name)
        self.network_params = params['network']
        self.name = base_name

        # multi-GPU (a2c_common.py:206-220): one process per GPU, actors sharded by rank
        self.multi_gpu = config.get('multi_gpu', False)
        self.multi_gpu_sync_stats = config.get('multi_gpu_sync_stats', True)
        mode = config.get('multi_gpu_sync_stats_mode', 'pooled')
        if mode not in STATS_SYNC_MODES:
            raise ValueError(f"multi_gpu_sync_stats_mode must be one of {STATS_SYNC_MODES}, got '{mode}'")
        self.multi_gpu_sync_stats_mode = mode
        self.local_rank = self.global_rank = 0
        self.world_size = 1
        if self.multi_gpu:
            self.local_rank = int(os.getenv('LOCAL_RANK', '0'))
            self.global_rank = int(os.getenv('RANK', '0'))
            self.world_size = int(os.getenv('WORLD_SIZE', '1'))
            config['device'] = 'cuda:' + str(self.local_rank)
        self.ppo_device = config.get('device', 'cuda:0')
        self._require_cuda()
        self.device_t = resolve_device(self.ppo_device)          # 'cuda' without an index = the current device
        if self.multi_gpu:
            if not dist.is_initialized():
                dist.init_process_group('nccl', rank=self.global_rank, world_size=self.world_size,
                                        device_id=torch.device(config['device']))
            if self.global_rank != 0:
                config['print_stats'] = False

        self.network_path = config.get('network_path', './nn/')
        self.env_config = config.get('env_config', {})
        self.num_actors = config['num_actors']
        self.env_name = config['env_name']
        self.env_info = config.get('env_info')
        if self.env_info is None:
            self.vec_env = create_vec_env(self.env_name, self.num_actors, **self.env_config)
            self.env_info = self.vec_env.get_env_info()
        else:
            self.vec_env = config.get('vec_env', None)
        self.value_size = self.env_info.get('value_size', 1)
        self.num_agents = self.env_info.get('agents', 1)
        if self.num_agents != 1:
            raise NotImplementedError('multi-agent envs are not on the B200 hot path yet')
        self.observation_space = self.env_info['observation_space']
        if type(self.observation_space).__name__ == 'Dict':
            raise NotImplementedError('Dict observation spaces are not on the B200 hot path yet')
        self.obs_shape = self.observation_space.shape
        if len(self.obs_shape) != 1:
            raise NotImplementedError('only flat observations are on the B200 hot path')
        self.autoreset_mode = self.env_info.get('autoreset_mode', 'same_step')
        self.mask_autoreset_rows = self.autoreset_mode == 'next_step'
        self.has_central_value = False
        self.central_value_net = None

        # PPO hyperparameters (a2c_common.py:190-491)
        self.ppo = config.get('ppo', True)
        self.max_epochs = config.get('max_epochs', -1)
        self.max_frames = max(config.get('max_frames', -1), config.get('max_steps', -1))
        self.horizon_length = config['horizon_length']
        self.seq_length = config.get('seq_length', 4)
        self.normalize_advantage = config['normalize_advantage']
        self.normalize_input = config['normalize_input']
        self.normalize_value = config.get('normalize_value', False)
        self.critic_coef = config['critic_coef']
        self.grad_norm = config['grad_norm']
        self.gamma = config['gamma']
        self.tau = config['tau']
        self.e_clip = config['e_clip']
        self.clip_value = config['clip_value']
        self.entropy_coef = config['entropy_coef']
        self.truncate_grads = config.get('truncate_grads', False)
        self.weight_decay = config.get('weight_decay', 0.0)
        self.value_bootstrap = config.get('value_bootstrap', True)
        self.use_smooth_clamp = config.get('use_smooth_clamp', False)
        self.games_to_track = config.get('games_to_track', 100)
        self.print_stats = config.get('print_stats', True)
        self.save_freq = config.get('save_frequency', 0)
        self.save_best_after = config.get('save_best_after', 100)
        rs = config['reward_shaper']
        self.rewards_shaper = rs if not isinstance(rs, dict) else DefaultRewardsShaper(**rs)

        self.batch_size = self.horizon_length * self.num_actors * self.num_agents
        self.batch_size_envs = self.horizon_length * self.num_actors
        if 'minibatch_size' not in config and 'minibatch_size_per_env' not in config:
            raise ValueError("Configuration must include either 'minibatch_size' or 'minibatch_size_per_env'. "
                             "Neither was found in the provided config.")
        self.minibatch_size_per_env = config.get('minibatch_size_per_env', 0)
        self.minibatch_size = config.get('minibatch_size', self.num_actors * self.minibatch_size_per_env)
        if self.minibatch_size <= 0:
            raise ValueError(f"'minibatch_size' must be greater than 0. Calculated value: {self.minibatch_size}.")
        self.num_minibatches = self.batch_size // self.minibatch_size
        if self.batch_size % self.minibatch_size != 0:
            raise ValueError(f"'batch_size' ({self.batch_size}) must be divisible by 'minibatch_size' ({self.minibatch_size}). "
                             "Ensure that 'batch_size' is a multiple of 'minibatch_size'.")
        if self.minibatch_size % self.horizon_length != 0:
            raise NotImplementedError("minibatch_size must be a multiple of horizon_length on the B200 path "
                                      "(minibatches are whole-env slices of the time-major arena)")
        self.envs_per_mb = self.minibatch_size // self.horizon_length
        self.mini_epochs_num = config['mini_epochs']

        self.last_lr = float(config['learning_rate'])
        self.is_adaptive_lr = config['lr_schedule'] == 'adaptive'
        self.linear_lr = config['lr_schedule'] == 'linear'
        if self.is_adaptive_lr:
            self.kl_threshold = config['kl_threshold']
            self.scheduler = AdaptiveScheduler(self.kl_threshold, min_lr=config.get('min_lr', 1e-6),
                                               max_lr=config.get('max_lr', 1e-2), lr_multiplier=config.get('lr_multiplier', 1.5))
        elif self.linear_lr and (self.max_epochs != -1 or self.max_frames != -1):
            use_epochs = self.max_epochs != -1
            self.scheduler = LinearScheduler(self.last_lr, min_lr=config.get('min_lr', 1e-6),
                                             max_steps=self.max_epochs if use_epochs else self.max_frames,
                                             use_epochs=use_epochs, apply_to_entropy=config.get('schedule_entropy', False),
                                             start_entropy_coef=config.get('entropy_coef'))
        else:
            self.scheduler = IdentityScheduler()
        self.stop_fn = config.get('stop_fn', None)
        if self.stop_fn is not None and not callable(self.stop_fn):
            raise ValueError(f"'stop_fn' must be callable, got {type(self.stop_fn).__name__}")

        self.frame = self.epoch_num = self.curr_frames = 0
        self.update_time = self.play_time = 0
        self.mean_rewards = self.last_mean_rewards = -float('inf')
        self.train_dir = config.get('train_dir', 'runs')
        self.experiment_dir = os.path.join(self.train_dir, self.experiment_name)
        self.nn_dir = os.path.join(self.experiment_dir, 'nn')
        self.summaries_dir = os.path.join(self.experiment_dir, 'summaries')
        for d in (self.train_dir, self.experiment_dir, self.nn_dir, self.summaries_dir):
            os.makedirs(d, exist_ok=True)
        self.writer = make_summary_writer(self.summaries_dir) if self.global_rank == 0 else None
        self.is_rnn = False
        self.rnn_states = None
        self._meter_cache = None
        self._tensors_ready = False
        self.obs = None
        self.game_rewards = _MeterView(self, 0)
        self.game_shaped_rewards = _MeterView(self, 1)
        self.game_lengths = _MeterView(self, 2)

    @property
    def device(self):
        return self.ppo_device

    def _require_cuda(self):
        """no CPU fallback: the kernels are the product (the host-logic tests replace this hook together with every op)"""
        if not str(self.ppo_device).startswith('cuda'):
            raise RuntimeError('rl_games_b200 agents run on CUDA only (device=%r): there is no CPU fallback' % self.ppo_device)
        torch.cuda.set_device(resolve_device(self.ppo_device))

    @staticmethod
    def _sync():
        torch.cuda.synchronize()

    def _meter_host(self):
        if self._meter_cache is None:
            self._meter_cache = self.meter.cpu().numpy()
        return self._meter_cache

    def update_epoch(self):
        self.epoch_num += 1
        return self.epoch_num

    def clear_stats(self, clean_rewards=True):
        self.meter.zero_()
        self._meter_cache = None
        if clean_rewards:
            self.mean_rewards = self.last_mean_rewards = -float('inf')
        self.algo_observer.after_clear_stats()

    # =============================================================================== multi-GPU stats sync
    def _stats_modules(self):
        mods = []
        if self.normalize_input:
            mods.append(('obs', self.model.running_mean_std))
        if self.normalize_value:
            mods.append(('value', self.model.value_mean_std))
        return mods

    def sync_running_stats(self):
        """a2c_common.py:782-808: pooled = all-reduce of per-epoch moment DELTAS (merge_rank_stats :61-93), packed into
        one fp64 all-reduce for all normalisers; broadcast = rank 0's stats."""
        if not self.multi_gpu or not self.multi_gpu_sync_stats:
            return
        mods = self._stats_modules()
        if not mods:
            return
        if self.multi_gpu_sync_stats_mode == 'broadcast':
            for _, m in mods:
                for t in (m.count, m.running_mean, m.running_var):
                    dist.broadcast(t, 0)
                m.refresh()
            return
        self._stats_sync_obj().sync(lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM))
        for _, m in mods:
            m.refresh()

    def _stats_sync_obj(self):
        if getattr(self, '_stats_sync', None) is None:
            self._stats_sync = PackedStatsSync([(n, m.count, m.running_mean, m.running_var) for n, m in self._stats_modules()])
        return self._stats_sync

    def _seed_stats_sync_snapshots(self):
        """a2c_common.py:767-780: after a weight load the restored normaliser history is not a delta of this epoch"""
        if not self.multi_gpu or not self.multi_gpu_sync_stats or self.multi_gpu_sync_stats_mode == 'broadcast':
            return
        self._stats_sync_obj().seed()

    # =============================================================================== train loop
    def _on_train_start(self):
        """what a subclass's train() presets before the first epoch (the reference's two loops differ here)"""

    def _broadcast_weights(self):
        """every rank starts from rank 0's weights (replaces broadcast_object_list of the pickled state_dict, a2c_common.py:1670-1680)"""
        dist.broadcast(self.model.flat, 0)

    def train(self):
        """a2c_common.py:1662-1782 (DiscreteA2CBase.train :1361-1470 is the same loop): frame / epoch accounting, summary scalars,
        periodic / best / final checkpoints, score_to_win / max_epochs / max_frames / stop_fn; rank 0 logs, checkpoints and decides
        when every rank stops.  Returns (last_mean_rewards, epoch_num)."""
        self.init_tensors()
        total_time = 0
        self.obs = self.env_reset()
        self._on_train_start()
        if self.multi_gpu:
            self._broadcast_weights()
        while True:
            epoch_num = self.update_epoch()
            # the continuous tuple carries b_losses between c_losses and entropies (its write_stats reads them from last_stats)
            step_time, play_time, update_time, sum_time, *losses, last_lr, lr_mul = self.train_epoch()
            a_losses, c_losses, entropies, kls = losses[0], losses[1], losses[-2], losses[-1]
            total_time += sum_time
            curr_frames = self.curr_frames * self.world_size if self.multi_gpu else self.curr_frames
            self.frame += curr_frames
            frame = self.frame // self.num_agents
            should_exit = False
            if self.global_rank == 0:
                if self.print_stats:
                    st = max(step_time, 1e-9)
                    print(f'fps step: {curr_frames / st:.0f} fps step and policy inference: {curr_frames / play_time:.0f} '
                          f'fps total: {curr_frames / sum_time:.0f} epoch: {epoch_num:.0f}/{self.max_epochs:.0f} frames: {frame:.0f}')
                self.write_stats(total_time, epoch_num, step_time, play_time, update_time, a_losses, c_losses, entropies, kls,
                                 last_lr, lr_mul, frame, sum_time, play_time, curr_frames)
                mean_rewards = None
                if self.game_rewards.current_size > 0:
                    mh = self._meter_host()
                    # float32 array like AverageMeter.get_mean() (torch_ext.py:349-352): checkpoint names embed str() of it
                    mean_rewards = np.asarray([mh[0]], dtype=np.float32)
                    self.mean_rewards = mean_rewards[0]
                    for tag, val in (('rewards', mh[0]), ('shaped_rewards', mh[1])):
                        self.writer.add_scalar(tag + '/step', val, frame)
                        self.writer.add_scalar(tag + '/iter', val, epoch_num)
                        self.writer.add_scalar(tag + '/time', val, total_time)
                    self.writer.add_scalar('episode_lengths/step', mh[2], frame)
                    self.writer.add_scalar('episode_lengths/iter', mh[2], epoch_num)
                    self.writer.add_scalar('episode_lengths/time', mh[2], total_time)
                    checkpoint_name = self.config['name'] + '_ep_' + str(epoch_num) + '_rew_' + str(mean_rewards[0])
                    if self.save_freq > 0 and epoch_num % self.save_freq == 0:
                        self.save(os.path.join(self.nn_dir, 'last_' + checkpoint_name))
                    if mean_rewards[0] > self.last_mean_rewards and epoch_num >= self.save_best_after:
                        print('saving next best rewards: ', mean_rewards)
                        self.last_mean_rewards = mean_rewards[0]
                        self.save(os.path.join(self.nn_dir, self.config['name']))
                        if 'score_to_win' in self.config and self.last_mean_rewards > self.config['score_to_win']:
                            print('Maximum reward achieved. Network won!')
                            self.save(os.path.join(self.nn_dir, checkpoint_name))
                            should_exit = True
                if epoch_num >= self.max_epochs and self.max_epochs != -1:
                    if self.game_rewards.current_size == 0:
                        print('WARNING: Max epochs reached before any env terminated at least once')
                        mean_rewards = -np.inf
                    self.save(os.path.join(self.nn_dir, 'last_' + self.config['name'] + '_ep_' + str(epoch_num)
                                           + '_rew_' + str(mean_rewards).replace('[', '_').replace(']', '_')))
                    print('MAX EPOCHS NUM!')
                    should_exit = True
                if self.frame >= self.max_frames and self.max_frames != -1:
                    if self.game_rewards.current_size == 0:
                        mean_rewards = -np.inf
                    self.save(os.path.join(self.nn_dir, 'last_' + self.config['name'] + '_frame_' + str(self.frame)
                                           + '_rew_' + str(mean_rewards).replace('[', '_').replace(']', '_')))
                    print('MAX FRAMES NUM!')
                    should_exit = True
                if not should_exit and self.stop_fn is not None and self.stop_fn(self):
                    self.save(os.path.join(self.nn_dir, 'last_' + self.config['name'] + '_custom_stop_ep_' + str(epoch_num)))
                    print('Custom stop callback returned True. Stopping training.')
                    should_exit = True
            if self.multi_gpu:
                t = torch.tensor(float(should_exit), device=self.device_t)
                dist.broadcast(t, 0)
                should_exit = bool(t.item())
            if should_exit:
                return self.last_mean_rewards, epoch_num

    def write_stats(self, total_time, epoch_num, step_time, play_time, update_time, a_losses, c_losses, entropies, kls,
                    last_lr, lr_mul, frame, scaled_time, scaled_play_time, curr_frames):
        """a2c_common.py:527-547: the same summary scalars, tag for tag; the loss lists are averaged like torch_ext.mean_list"""
        w = self.writer
        mean = lambda xs: float(torch.stack(list(xs)).mean())     # noqa: E731
        w.add_scalar('performance/step_inference_rl_update_fps', curr_frames / scaled_time, frame)
        w.add_scalar('performance/step_inference_fps', curr_frames / scaled_play_time, frame)
        w.add_scalar('performance/step_fps', curr_frames / max(step_time, 1e-9), frame)
        w.add_scalar('performance/rl_update_time', update_time, frame)
        w.add_scalar('performance/step_inference_time', play_time, frame)
        w.add_scalar('performance/step_time', step_time, frame)
        w.add_scalar('losses/a_loss', mean(a_losses), frame)
        w.add_scalar('losses/c_loss', mean(c_losses), frame)
        w.add_scalar('losses/entropy', mean(entropies), frame)
        w.add_scalar('info/last_lr', last_lr * lr_mul, frame)
        w.add_scalar('info/lr_mul', lr_mul, frame)
        w.add_scalar('info/e_clip', self.e_clip * lr_mul, frame)
        w.add_scalar('info/kl', mean(kls), frame)
        w.add_scalar('info/epochs', epoch_num, frame)
        self.algo_observer.after_print_stats(frame, epoch_num, total_time)

    # =============================================================================== checkpoints (a2c_common.py:825-921)
    def get_weights(self):
        return {'model': self.model.state_dict()}

    def get_stats_weights(self, model_stats=False):
        state = {}
        if model_stats:
            if self.normalize_input:
                state['running_mean_std'] = self.model.running_mean_std.state_dict('')
            if self.normalize_value:
                state['reward_mean_std'] = self.model.value_mean_std.state_dict('')
        return state

    def set_stats_weights(self, weights):
        if self.normalize_input and 'running_mean_std' in weights:
            self.model.running_mean_std.load_state_dict(weights['running_mean_std'])
        if self.normalize_value and 'reward_mean_std' in weights:
            self.model.value_mean_std.load_state_dict(weights['reward_mean_std'])

    def set_weights(self, weights):
        self.model.load_state_dict(weights['model'])
        self.set_stats_weights(weights)
        self._seed_stats_sync_snapshots()

    def get_full_state_weights(self):
        self.init_tensors()
        state = self.get_weights()
        state['epoch'] = self.epoch_num
        state['frame'] = self.frame
        state['optimizer'] = self.model.optimizer_state_dict(self._optimizer_lr(), float(self.opt_state.cpu()[1]), self.weight_decay)
        state['last_mean_rewards'] = self.last_mean_rewards
        if self.vec_env is not None and hasattr(self.vec_env, 'get_env_state'):
            state['env_state'] = self.vec_env.get_env_state()
        if self.config.get('capability_manifest') is not None:
            state['capability_manifest'] = self.config['capability_manifest']
        return state

    def set_full_state_weights(self, weights, set_epoch=True):
        self.init_tensors()
        self.set_weights(weights)
        if set_epoch:
            self.epoch_num = weights['epoch']
            self.frame = weights['frame']
        # a2c_common.py:852-866 restores the OPTIMIZER (its param-group lr included) but not self.last_lr
        lr, step = self.model.load_optimizer_state_dict(weights['optimizer'])
        self._restore_optimizer(lr, step)
        self.last_mean_rewards = weights.get('last_mean_rewards', -float('inf'))
        if self.vec_env is not None and hasattr(self.vec_env, 'set_env_state'):
            self.vec_env.set_env_state(weights.get('env_state', None))
        if 'capability_manifest' in weights and self.config.get('capability_manifest') is None:
            self.config['capability_manifest'] = weights['capability_manifest']
        self._seed_stats_sync_snapshots()

    def save(self, fn):
        """torch_ext.save_checkpoint (torch_ext.py:90-92): `<fn>.pth` via torch.save"""
        torch.save(self.get_full_state_weights(), fn + '.pth')

    def restore(self, fn, set_epoch=True):
        """torch_ext.load_checkpoint (torch_ext.py:94-112): strips `_orig_mod.` prefixes"""
        checkpoint = torch.load(fn, map_location=self.device_t, weights_only=False)
        if 'model' in checkpoint:
            checkpoint['model'] = {k.replace('_orig_mod.', ''): v for k, v in checkpoint['model'].items()}
        self.set_full_state_weights(checkpoint, set_epoch=set_epoch)
