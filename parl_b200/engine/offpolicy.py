"""DDPG / TD3 / SAC on one B200 with exploration, replay and updates on the device — the replacement of the per-step
loop of benchmark/torch/{td3,sac,ddpg}/train.py (agent.sample -> env.step -> rpm.append -> rpm.sample_batch ->
agent.learn, one env step at a time).

Exploration is ONE launch of rl_explore_mlp per call: K lock-step steps of B MuJoCo-shaped synthetic envs, the actor
read in place from the model's parameters (FlatAdam views, so every launch explores with the current weights), the
transitions written straight into the rows of a ``utils.ReplayMemory``.  Each update draws a batch with
rl_replay_sample_uniform (replay size and draw index live in device memory) and hands it to the unchanged
``DDPG`` / ``TD3`` / ``SAC`` class: networks on torch autograd through the user's ``parl.Model``, the critic's TD
target / loss / gradient in rl_twin_q_td_loss_fwd_bwd and Adam in rl_adam_step.

The update is replayed as CUDA graphs (both optimisers keep their step count and learning rate on the device): a critic
graph (sampler, draw-index increment, critic update) and, for TD3, an actor + Polyak graph replayed every policy_freq
calls (the host keeps ``TD3.total_it`` in step); DDPG and SAC replay critic, actor and Polyak graphs.  Each part runs
eagerly the first time it is needed (on the capture stream, so that its lazy initialisation happens outside a capture),
is captured the second time and replayed from then on.  One replayed update is bit-identical to the eager class update
on the same batch (tests/test_gpu_offpolicy.py).
"""
import math

import torch

from .. import kernels
from ..algorithms import DDPG, TD3, SAC
from ..utils.replay_memory import ReplayMemory
from .nets import TD3MujocoModel, SACMujocoModel, DDPGMujocoModel

# train.py constants of the reference (benchmark/torch/{td3,sac,ddpg}/train.py)
_DEFAULTS = {
    'td3': dict(batch_size=256, actor_lr=3e-4, critic_lr=3e-4),
    'sac': dict(batch_size=256, actor_lr=3e-4, critic_lr=3e-4),
    'ddpg': dict(batch_size=100, actor_lr=1e-3, critic_lr=1e-3),
}
_MODELS = {'td3': TD3MujocoModel, 'sac': SACMujocoModel, 'ddpg': DDPGMujocoModel}


class OffPolicyEngine(object):
    def __init__(self, kind='td3', num_envs=256, memory_size=int(1e6), batch_size=None, warmup_size=int(1e4),
                 steps_per_iter=1, updates_per_iter=1, expl_noise=0.1, seed=0, obs_dim=17, act_dim=6, gamma=0.99,
                 tau=0.005, actor_lr=None, critic_lr=None, alpha=0.2, policy_noise=0.2, noise_clip=0.5,
                 policy_freq=2, p_done=0.01, max_episode_steps=1000, env_offset=0, model=None, device=None):
        if kind not in _DEFAULTS:
            raise ValueError("OffPolicyEngine: kind must be 'td3', 'sac' or 'ddpg', got %r" % (kind, ))
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = dev = torch.device(device)
        d = _DEFAULTS[kind]
        self.kind = kind
        self.B, self.D, self.AD = int(num_envs), int(obs_dim), int(act_dim)
        self.batch_size = int(batch_size if batch_size is not None else d['batch_size'])
        self.warmup_size, self.steps_per_iter, self.updates_per_iter = (int(warmup_size), int(steps_per_iter),
                                                                        int(updates_per_iter))
        self.expl_noise, self.seed, self.env_offset = float(expl_noise), int(seed), int(env_offset)
        self.p_done, self.max_episode_steps = float(p_done), int(max_episode_steps)
        actor_lr = float(actor_lr if actor_lr is not None else d['actor_lr'])
        critic_lr = float(critic_lr if critic_lr is not None else d['critic_lr'])
        self.model = (model if model is not None else _MODELS[kind](obs_dim, act_dim)).to(dev)
        if kind == 'td3':
            self.alg = TD3(self.model, gamma=float(gamma), tau=float(tau), actor_lr=actor_lr, critic_lr=critic_lr,
                           policy_noise=policy_noise, noise_clip=noise_clip, policy_freq=policy_freq)
        elif kind == 'sac':
            self.alg = SAC(self.model, gamma=float(gamma), tau=float(tau), alpha=float(alpha), actor_lr=actor_lr,
                           critic_lr=critic_lr)
        else:
            self.alg = DDPG(self.model, gamma=float(gamma), tau=float(tau), actor_lr=actor_lr, critic_lr=critic_lr)
        # the plan takes the parameter pointers once: build it after the optimisers re-homed the parameters
        layers, act, self.head = self.model.native_actor_layers()
        self.plan = kernels.MlpPlan(layers, act)
        self.mode = kernels.EXPLORE_SAC if kind == 'sac' else kernels.EXPLORE_NOISE
        self.rpm = ReplayMemory(memory_size, obs_dim, act_dim, device=dev)
        if self.B > self.rpm.max_size:
            raise ValueError('OffPolicyEngine: num_envs %d exceeds memory_size %d' % (self.B, self.rpm.max_size))
        self.stats = kernels.EpisodeStats(self.B, dev)
        self.obs_cur = torch.zeros((self.B, self.D), dtype=torch.float32, device=dev)
        self.size_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.draw_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        f32 = torch.float32
        n = self.batch_size
        self._batch = (torch.empty((n, self.D), dtype=f32, device=dev), torch.empty((n, self.AD), dtype=f32, device=dev),
                       torch.empty(n, dtype=f32, device=dev), torch.empty((n, self.D), dtype=f32, device=dev),
                       torch.empty(n, dtype=f32, device=dev))
        self.env_steps = 0
        self.sample_steps = 0
        self.learn_steps = 0
        self.alg.actor_optimizer.enable_device_state()
        self.alg.critic_optimizer.enable_device_state()
        self._stream = torch.cuda.Stream(device=dev)
        self._warm, self._graphs, self._outs = set(), {}, {}
        self.reset()

    def reset(self):
        """First observation of every env (the env's reset draw at step 0) and zeroed episode counters."""
        kernels.env_mujoco_synth_step(self.obs_cur, None, None, self.stats, self.seed, 0, env_offset=self.env_offset,
                                      reset=True)
        self.env_steps = 0

    # ------------------------------------------------------------------ actor side
    def _explore(self, mode, K):
        per_launch = max(self.rpm.max_size // self.B, 1)        # a launch never overwrites its own rows
        while K > 0:
            k = min(K, per_launch)
            self.plan.explore(self.rpm, mode, k, self.obs_cur, self.stats, self.seed, self.env_steps, head=self.head,
                              expl_noise=self.expl_noise, env_offset=self.env_offset, p_done=self.p_done,
                              max_episode_steps=self.max_episode_steps)
            self.rpm.commit(k * self.B)
            self.env_steps += k
            self.sample_steps += k * self.B
            K -= k
        self.size_dev.fill_(self.rpm.size())

    def warmup(self):
        """Uniform random actions until the replay holds warmup_size transitions (train.py: WARMUP_SIZE)."""
        self._explore(kernels.EXPLORE_WARMUP, max(1, int(math.ceil(self.warmup_size / float(self.B)))))

    def explore(self):
        """steps_per_iter lock-step steps of every env with the current policy and its exploration rule."""
        self._explore(self.mode, self.steps_per_iter)

    # ------------------------------------------------------------------ learner side
    def _critic_part(self):
        obs, action, reward, next_obs, terminal = kernels.replay_sample_uniform(
            self.rpm, self.batch_size, self.size_dev, self.draw_dev, self.seed, out=self._batch)
        self.draw_dev.add_(1)
        return self.alg._critic_learn(obs, action, reward, next_obs, terminal)

    def _actor_part(self):
        return self.alg._actor_learn(self._batch[0])

    def _polyak_part(self):
        self.alg.sync_target()

    def _run(self, name, fn, opt):
        """First call: eager on the capture stream; second: capture, then replay; later: replay."""
        cur = torch.cuda.current_stream(self.device)
        if name not in self._warm:
            self._stream.wait_stream(cur)
            with torch.cuda.stream(self._stream):
                out = fn()
            cur.wait_stream(self._stream)
            self._warm.add(name)
            return out
        if name not in self._graphs:
            count = opt.step_count if opt is not None else 0
            launches = kernels.launch_count()
            self._stream.wait_stream(cur)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self._stream):
                self._outs[name] = fn()
            if opt is not None:
                opt.step_count = count                      # capture is not execution
            n = kernels.launch_count() - launches
            kernels.add_graph_launches(-n)
            self._graphs[name] = (g, n)
        g, n = self._graphs[name]
        g.replay()
        kernels.add_graph_launches(n)
        if opt is not None:
            opt.step_count += 1
        return self._outs[name]

    def _update(self):
        alg = self.alg
        critic_loss = self._run('critic', self._critic_part, alg.critic_optimizer)
        actor_loss = None
        if self.kind == 'td3':
            alg.total_it += 1                               # TD3.learn's counter: actor + Polyak every policy_freq
            if alg.total_it % alg.policy_freq == 0:
                actor_loss = self._run('actor', self._actor_part, alg.actor_optimizer)
        else:
            actor_loss = self._run('actor', self._actor_part, alg.actor_optimizer)
            self._run('polyak', self._polyak_part, None)
        return critic_loss, actor_loss

    def learn(self):
        """updates_per_iter updates, each on a fresh uniform batch of the replay; returns the device losses
        (critic, actor) of the last one (actor None on a TD3 call without an actor update)."""
        out = None
        for _ in range(self.updates_per_iter):
            out = self._update()
            self.learn_steps += 1
        return out

    def step(self):
        self.explore()
        return self.learn()

    def get_metrics(self):
        tot = self.stats.totals.tolist()
        n = max(tot[0], 1.0)
        return dict(sample_steps=self.sample_steps, episodes=int(tot[0]), mean_episode_rewards=tot[1] / n,
                    mean_episode_steps=tot[2] / n, replay_size=self.rpm.size(), learn_steps=self.learn_steps)
