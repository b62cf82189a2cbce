"""Policy/value networks of the target examples as ``parl.Model`` subclasses (a13, SURVEY.md §8a).

AtariActorCritic  = the 84x84 actor-critic of benchmark/torch/a2c/atari_model.py:23-96 (conv 8x8/4,
                    4x4/2, 3x3/1, fc 512, policy/value heads, xavier-normal init) — used for the C3
                    IMPALA config because examples/IMPALA/atari_model.py is sized for 42x42 inputs.
MujocoModel       = benchmark/torch/ppo/mujoco_model.py:27-53 (two 64-unit tanh MLPs, state-independent
                    log-std parameter).
CartPoleModel     = benchmark/torch/QuickStart/cartpole_model.py:21-38 (softmax policy) and an
                    actor-critic variant for A2C on CartPole (C2).
Observations arrive as uint8 [N,4,84,84] views of the device rollout buffer and are scaled by 1/255
inside the model, as the reference models do (``obs / 255.0``).
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from ..core import Model


class AtariActorCritic(Model):
    def __init__(self, act_dim, compute_dtype=torch.bfloat16):
        super(AtariActorCritic, self).__init__()
        self.conv1 = nn.Conv2d(4, 32, kernel_size=8, stride=4, padding=1)
        self.conv2 = nn.Conv2d(32, 64, kernel_size=4, stride=2, padding=2)
        self.conv3 = nn.Conv2d(64, 64, kernel_size=3, stride=1, padding=0)
        self.fc = nn.Linear(64 * 9 * 9, 512)
        self.fc_pi = nn.Linear(512, act_dim)
        self.fc_v = nn.Linear(512, 1)
        self.compute_dtype = compute_dtype
        for m in self.modules():                       # atari_model.py:89-96
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                nn.init.xavier_normal_(m.weight)
                nn.init.constant_(m.bias, 0)

    def _trunk(self, x):
        """Accepts (a) bf16 [N,21,21,64]: conv1's space-to-depth input from rl_obs_stack_gather(s2d=True),
        already scaled by 1/255, or the same layout in uint8 (unscaled bytes, scaled here); (b) bf16 [N,84,84,4] NHWC, already scaled; (c) uint8/float [N,4,84,84] as in
        the reference (scaled here by 1/255).  Activations stay NHWC (channels_last); the flatten before
        ``fc`` is taken in (H,W,C) order with the weight columns permuted accordingly, which is the same
        function as the reference's (C,H,W) nn.Flatten + nn.Linear."""
        dt = self.compute_dtype if x.is_cuda else torch.float32
        with torch.autocast(device_type=x.device.type, dtype=dt, enabled=dt != torch.float32):
            if x.dtype == torch.uint8 and x.dim() == 4 and x.shape[-1] == 64:
                x = (x.float() * (1.0 / 255.0)).to(torch.bfloat16)     # the rounding the u8in conv kernels apply
            if x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[-1] == 64:
                # 8x8/4/pad-1 conv == 2x2/1 conv over 4x4 pixel blocks: W1[o,c,4a+dy,4b+dx] -> W1'[o,(dy,dx,c),a,b]
                w1 = self.conv1.weight.view(32, 4, 2, 4, 2, 4).permute(0, 3, 5, 1, 2, 4).reshape(32, 64, 2, 2)
                x = F.relu(F.conv2d(x.permute(0, 3, 1, 2), w1, self.conv1.bias))
            else:
                if x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[-1] == 4:
                    x = x.permute(0, 3, 1, 2)              # zero-copy NCHW view with channels_last strides
                else:
                    x = (x.to(dt) / 255.0).contiguous(memory_format=torch.channels_last)
                x = F.relu(self.conv1(x))
            x = F.relu(self.conv2(x))
            x = F.relu(self.conv3(x))
            n = x.shape[0]
            feat = x.permute(0, 2, 3, 1).reshape(n, -1)     # (H,W,C) order: a view for channels_last activations
            wfc = self.fc.weight.view(512, 64, 9, 9).permute(0, 2, 3, 1).reshape(512, 64 * 9 * 9)
            return F.relu(F.linear(feat, wfc, self.fc.bias))

    def policy(self, x):
        h = self._trunk(x)
        return F.linear(h.float(), self.fc_pi.weight, self.fc_pi.bias)

    def value(self, x):
        h = self._trunk(x)
        return F.linear(h.float(), self.fc_v.weight, self.fc_v.bias).squeeze(1)

    def policy_and_value(self, x):
        h = self._trunk(x).float()
        logits = F.linear(h, self.fc_pi.weight, self.fc_pi.bias)
        values = F.linear(h, self.fc_v.weight, self.fc_v.bias).squeeze(1)
        return logits, values


def _dim(space_or_int):
    """The reference models take gym spaces (``MujocoModel(obs_space, act_space)``); plain ints work too."""
    if hasattr(space_or_int, 'shape'):
        shp = tuple(space_or_int.shape)
        n = 1
        for d in shp:
            n *= int(d)
        return n
    return int(space_or_int)


def _orthogonal(layer, std=2 ** 0.5, bias_const=0.0):
    nn.init.orthogonal_(layer.weight, std)
    nn.init.constant_(layer.bias, bias_const)
    return layer


class MujocoModel(Model):
    """benchmark/torch/ppo/mujoco_model.py:27-53: shared 64-64 tanh trunk, value head, policy-mean head,
    state-independent log-std parameter; orthogonal init (std sqrt2 / 1.0 / 0.01)."""

    def __init__(self, obs_space=17, act_space=6):
        super(MujocoModel, self).__init__()
        obs_dim, act_dim = _dim(obs_space), _dim(act_space)
        self.fc1 = _orthogonal(nn.Linear(obs_dim, 64))
        self.fc2 = _orthogonal(nn.Linear(64, 64))
        self.fc_value = _orthogonal(nn.Linear(64, 1), std=1.0)
        self.fc_policy = _orthogonal(nn.Linear(64, act_dim), std=0.01)
        self.fc_pi_std = nn.Parameter(torch.zeros(1, act_dim))

    def _trunk(self, obs):
        return torch.tanh(self.fc2(torch.tanh(self.fc1(obs))))

    def value(self, obs):
        return self.fc_value(self._trunk(obs))

    def policy(self, obs):
        mean = self.fc_policy(self._trunk(obs))
        return mean, torch.exp(self.fc_pi_std.expand_as(mean))

    def native_layers(self):
        """Row segments per linear layer for rl_mlp_fwd/bwd: outputs = [mean (act_dim) | value (1)]."""
        from ..kernels import ACT_TANH
        return [[(self.fc1.weight, self.fc1.bias)], [(self.fc2.weight, self.fc2.bias)],
                [(self.fc_policy.weight, self.fc_policy.bias), (self.fc_value.weight, self.fc_value.bias)]], ACT_TANH


class CartPoleActorCritic(Model):
    """Actor-critic MLP for A2C on CartPole (BASELINE configs[1]); the reference ships no CartPole A2C model, the
    layout follows its Atari actor-critic (shared trunk, policy + value heads, benchmark/torch/a2c/atari_model.py)."""

    def __init__(self, obs_dim=4, act_dim=2, hidden=64):
        super(CartPoleActorCritic, self).__init__()
        self.fc1, self.fc2 = nn.Linear(obs_dim, hidden), nn.Linear(hidden, hidden)
        self.fc_pi, self.fc_v = nn.Linear(hidden, act_dim), nn.Linear(hidden, 1)

    def _trunk(self, x):
        return torch.tanh(self.fc2(torch.tanh(self.fc1(x))))

    def policy(self, x):
        return self.fc_pi(self._trunk(x))

    def value(self, x):
        return self.fc_v(self._trunk(x)).squeeze(1)

    def policy_and_value(self, x):
        h = self._trunk(x)
        return self.fc_pi(h), self.fc_v(h).squeeze(1)

    def native_layers(self):
        from ..kernels import ACT_TANH
        return [[(self.fc1.weight, self.fc1.bias)], [(self.fc2.weight, self.fc2.bias)],
                [(self.fc_pi.weight, self.fc_pi.bias), (self.fc_v.weight, self.fc_v.bias)]], ACT_TANH


class CartPolePolicy(Model):
    """benchmark/torch/QuickStart/cartpole_model.py:21-38: forward returns action probabilities."""

    def __init__(self, obs_dim=4, act_dim=2):
        super(CartPolePolicy, self).__init__()
        self.fc1 = nn.Linear(obs_dim, act_dim * 10)
        self.fc2 = nn.Linear(act_dim * 10, act_dim)

    def forward(self, x):
        return F.softmax(self.fc2(torch.tanh(self.fc1(x))), dim=-1)

    def native_layers(self):
        """Logits (the softmax is applied by the consumer)."""
        from ..kernels import ACT_TANH
        return [[(self.fc1.weight, self.fc1.bias)], [(self.fc2.weight, self.fc2.bias)]], ACT_TANH


class CartPoleQModel(Model):
    """examples/DQN/cartpole_model.py:21-41: 128-128 ReLU MLP -> Q values."""

    def __init__(self, obs_dim=4, act_dim=2, hidden=128):
        super(CartPoleQModel, self).__init__()
        self.fc1, self.fc2, self.fc3 = nn.Linear(obs_dim, hidden), nn.Linear(hidden, hidden), nn.Linear(hidden, act_dim)

    def forward(self, obs):
        return self.fc3(F.relu(self.fc2(F.relu(self.fc1(obs)))))

    def native_layers(self):
        from ..kernels import ACT_RELU
        return [[(self.fc1.weight, self.fc1.bias)], [(self.fc2.weight, self.fc2.bias)],
                [(self.fc3.weight, self.fc3.bias)]], ACT_RELU


class AtariQModel(Model):
    """benchmark/torch/dqn/model.py:19-95: conv 5x5/p2 -> pool -> conv 5x5/p2 -> pool -> conv 4x4/p1 -> pool ->
    conv 3x3/p1 -> flatten 6400 -> linear (or the dueling pair of 512-unit streams), kaiming-normal fan-out init,
    ``obs / 255`` inside the model."""

    def __init__(self, act_dim, dueling=False):
        super(AtariQModel, self).__init__()
        self.conv1 = nn.Conv2d(4, 32, kernel_size=5, stride=1, padding=2)
        self.conv2 = nn.Conv2d(32, 32, kernel_size=5, stride=1, padding=2)
        self.conv3 = nn.Conv2d(32, 64, kernel_size=4, stride=1, padding=1)
        self.conv4 = nn.Conv2d(64, 64, kernel_size=3, stride=1, padding=1)
        self.dueling = dueling
        if dueling:
            self.linear_1_adv, self.linear_2_adv = nn.Linear(6400, 512), nn.Linear(512, act_dim)
            self.linear_1_val, self.linear_2_val = nn.Linear(6400, 512), nn.Linear(512, 1)
        else:
            self.linear_1 = nn.Linear(6400, act_dim)
        for m in self.modules():
            if isinstance(m, (nn.Linear, nn.Conv2d)):
                nn.init.kaiming_normal_(m.weight, mode='fan_out', nonlinearity='relu')
                nn.init.zeros_(m.bias)

    def forward(self, obs):
        x = obs.float() / 255.0
        x = F.max_pool2d(F.relu(self.conv1(x)), 2, 2)
        x = F.max_pool2d(F.relu(self.conv2(x)), 2, 2)
        x = F.max_pool2d(F.relu(self.conv3(x)), 2, 2)
        x = F.relu(self.conv4(x)).flatten(1)
        if self.dueling:
            a = self.linear_2_adv(F.relu(self.linear_1_adv(x)))
            v = self.linear_2_val(F.relu(self.linear_1_val(x)))
            return a + (v - a.mean(dim=1, keepdim=True))
        return self.linear_1(x)


# ---- continuous-control actor / critic pairs (benchmark/torch/{td3,sac,ddpg}/mujoco_model.py), torch default init ----
class _TwinCritic(Model):
    """Two 256-256 ReLU Q networks on cat(obs, action) (td3 / sac mujoco_model.py Critic)."""

    def __init__(self, obs_dim, act_dim):
        super(_TwinCritic, self).__init__()
        self.l1, self.l2, self.l3 = nn.Linear(obs_dim + act_dim, 256), nn.Linear(256, 256), nn.Linear(256, 1)
        self.l4, self.l5, self.l6 = nn.Linear(obs_dim + act_dim, 256), nn.Linear(256, 256), nn.Linear(256, 1)

    def forward(self, obs, action):
        sa = torch.cat([obs, action], 1)
        q1 = self.l3(F.relu(self.l2(F.relu(self.l1(sa)))))
        q2 = self.l6(F.relu(self.l5(F.relu(self.l4(sa)))))
        return q1, q2

    def Q1(self, obs, action):
        sa = torch.cat([obs, action], 1)
        return self.l3(F.relu(self.l2(F.relu(self.l1(sa)))))


class _TanhActor(Model):
    """ReLU MLP with a tanh head (td3 / ddpg mujoco_model.py Actor)."""

    def __init__(self, obs_dim, act_dim, h1, h2):
        super(_TanhActor, self).__init__()
        self.l1, self.l2, self.l3 = nn.Linear(obs_dim, h1), nn.Linear(h1, h2), nn.Linear(h2, act_dim)

    def forward(self, obs):
        return torch.tanh(self.l3(F.relu(self.l2(F.relu(self.l1(obs))))))


class _GaussianActor(Model):
    """sac/mujoco_model.py Actor: 256-256 ReLU trunk, mean and log-std heads, log-std clamped to [-20, 2]."""

    def __init__(self, obs_dim, act_dim):
        super(_GaussianActor, self).__init__()
        self.l1, self.l2 = nn.Linear(obs_dim, 256), nn.Linear(256, 256)
        self.mean_linear, self.std_linear = nn.Linear(256, act_dim), nn.Linear(256, act_dim)

    def forward(self, obs):
        x = F.relu(self.l2(F.relu(self.l1(obs))))
        return self.mean_linear(x), torch.clamp(self.std_linear(x), min=-20.0, max=2.0)


class _DDPGCritic(Model):
    """ddpg/mujoco_model.py Critic: obs -> 400 (ReLU), cat action -> 300 (ReLU) -> 1."""

    def __init__(self, obs_dim, act_dim):
        super(_DDPGCritic, self).__init__()
        self.l1, self.l2, self.l3 = nn.Linear(obs_dim, 400), nn.Linear(400 + act_dim, 300), nn.Linear(300, 1)

    def forward(self, obs, action):
        q = F.relu(self.l1(obs))
        return self.l3(F.relu(self.l2(torch.cat([q, action], 1))))


class _ActorCriticModel(Model):
    def policy(self, obs):
        return self.actor_model(obs)

    def value(self, obs, action):
        return self.critic_model(obs, action)

    def get_actor_params(self):
        return self.actor_model.parameters()

    def get_critic_params(self):
        return self.critic_model.parameters()


class TD3MujocoModel(_ActorCriticModel):
    """benchmark/torch/td3/mujoco_model.py: actor 17 -> 256 -> 256 -> act (tanh), twin 256-256 critics."""

    def __init__(self, obs_space=17, act_space=6):
        super(TD3MujocoModel, self).__init__()
        obs_dim, act_dim = _dim(obs_space), _dim(act_space)
        self.actor_model = _TanhActor(obs_dim, act_dim, 256, 256)
        self.critic_model = _TwinCritic(obs_dim, act_dim)

    def Q1(self, obs, action):
        return self.critic_model.Q1(obs, action)

    def native_actor_layers(self):
        """Row segments per linear layer of the actor for rl_explore_mlp (ReLU hidden layers, tanh head)."""
        from ..kernels import ACT_RELU, HEAD_TANH
        a = self.actor_model
        return [[(a.l1.weight, a.l1.bias)], [(a.l2.weight, a.l2.bias)], [(a.l3.weight, a.l3.bias)]], ACT_RELU, HEAD_TANH


class SACMujocoModel(_ActorCriticModel):
    """benchmark/torch/sac/mujoco_model.py: actor 17 -> 256 -> 256 -> {mean, log-std}, twin 256-256 critics."""

    def __init__(self, obs_space=17, act_space=6):
        super(SACMujocoModel, self).__init__()
        obs_dim, act_dim = _dim(obs_space), _dim(act_space)
        self.actor_model = _GaussianActor(obs_dim, act_dim)
        self.critic_model = _TwinCritic(obs_dim, act_dim)

    def Q1(self, obs, action):
        return self.critic_model.Q1(obs, action)

    def native_actor_layers(self):
        """Head outputs = [mean (act_dim) | log-std (act_dim)] (the kernel applies the clamp)."""
        from ..kernels import ACT_RELU, HEAD_MEAN_LOGSTD
        a = self.actor_model
        return [[(a.l1.weight, a.l1.bias)], [(a.l2.weight, a.l2.bias)],
                [(a.mean_linear.weight, a.mean_linear.bias), (a.std_linear.weight, a.std_linear.bias)]], \
            ACT_RELU, HEAD_MEAN_LOGSTD


class DDPGMujocoModel(_ActorCriticModel):
    """benchmark/torch/ddpg/mujoco_model.py: actor 17 -> 400 -> 300 -> act (tanh), critic 400 / 300."""

    def __init__(self, obs_space=17, act_space=6):
        super(DDPGMujocoModel, self).__init__()
        obs_dim, act_dim = _dim(obs_space), _dim(act_space)
        self.actor_model = _TanhActor(obs_dim, act_dim, 400, 300)
        self.critic_model = _DDPGCritic(obs_dim, act_dim)

    def Q1(self, obs, action):
        return self.critic_model(obs, action)

    def native_actor_layers(self):
        from ..kernels import ACT_RELU, HEAD_TANH
        a = self.actor_model
        return [[(a.l1.weight, a.l1.bias)], [(a.l2.weight, a.l2.bias)], [(a.l3.weight, a.l3.bias)]], ACT_RELU, HEAD_TANH
