"""CPU restatement of rl_explore_mlp and rl_replay_sample_uniform (TEST INFRASTRUCTURE, see oracle/__init__.py).

Exploration (benchmark/torch/{td3,sac,ddpg}/train.py + mujoco_agent.py):
  mode 0 warm-up      a = 2u - 1, u = 24-bit uniform of word d % 4 of philox(env, step, d // 4, STREAM_ACTION)
                      (np.random.uniform(-1, 1) before WARMUP_SIZE)                              exact in float32
  mode 1 noise        a = clip(tanh(out) + sigma * z, -1, 1)   (td3 / ddpg mujoco_agent.sample)
  mode 2 SAC          a = tanh(mean + exp(clip(log_std, -20, 2)) * z)   (SAC.sample)
  z = Box-Muller of the STREAM_GAUSS words of (env, step, d // 4), restated in float64 here; the actor forward is
  float64 too, so the device's fp32 actions are compared within a tolerance.
Env: ``envs.MujocoSynthVec`` (reward / done at (env, step), next observation at step + 1); terminal = done and not
the time-limit step (train.py: ``terminal = float(done) if steps < env._max_episode_steps else 0``).
Ring: step t of env b goes to row (pos + t*B + b) % capacity.
Uniform sampler: row i of draw d = (x * size) >> 32, x = word 0 of philox(i, d, 0, STREAM_REPLAY).
"""
import numpy as np

from . import philox as ph
from .envs import MujocoSynthVec


def ring_rows(pos, t, B, capacity):
    """Replay rows written by lock-step t of envs 0..B-1."""
    return (int(pos) + int(t) * B + np.arange(B, dtype=np.int64)) % int(capacity)


def terminal_flags(done, ep_len_before, max_episode_steps):
    """terminal = done unless this step is the time-limit step (the episode length reaches max_episode_steps)."""
    done = np.asarray(done, bool)
    if not max_episode_steps:
        return done.astype(np.int32)
    at_limit = np.asarray(ep_len_before) + 1 >= int(max_episode_steps)
    return (done & ~at_limit).astype(np.int32)


def actor_forward64(layers, obs, head):
    """layers: [(W [out,in], b [out]), ...] float arrays (ReLU between layers); head 0 -> tanh(out),
    head 1 -> (mean, log_std clamped to [-20, 2]).  float64."""
    x = np.asarray(obs, np.float64)
    for i, (w, b) in enumerate(layers):
        x = x @ np.asarray(w, np.float64).T + np.asarray(b, np.float64)
        if i + 1 < len(layers):
            x = np.maximum(x, 0.0)
    if head == 0:
        return np.tanh(x)
    ad = x.shape[1] // 2
    return x[:, :ad], np.clip(x[:, ad:], -20.0, 2.0)


def uniform_actions(seed, env_ids, step, AD):
    k0, k1 = ph.split_seed(seed)
    nblk = (AD + 3) // 4
    w = ph.philox4x32(np.asarray(env_ids, np.uint32)[:, None], np.uint32(step), np.arange(nblk, dtype=np.uint32)[None],
                      ph.STREAM_ACTION, k0, k1)
    u = np.stack([ph.u01_24(v) for v in w], axis=-1).reshape(len(env_ids), nblk * 4)[:, :AD]
    return (np.float32(2.0) * u - np.float32(1.0)).astype(np.float32)


def gauss64(seed, env_ids, step, AD, stream=ph.STREAM_GAUSS):
    k0, k1 = ph.split_seed(seed)
    nblk = (AD + 3) // 4
    w = ph.philox4x32(np.asarray(env_ids, np.uint32)[:, None], np.uint32(step), np.arange(nblk, dtype=np.uint32)[None],
                      stream, k0, k1)

    def u(v):
        return ((v >> np.uint32(8)).astype(np.float64) + 0.5) * 2.0 ** -24

    out = []
    for a, b in ((w[0], w[1]), (w[2], w[3])):
        r, th = np.sqrt(-2.0 * np.log(u(a))), 2.0 * np.pi * u(b)
        out += [r * np.cos(th), r * np.sin(th)]
    return np.stack(out, axis=-1).reshape(len(env_ids), nblk * 4)[:, :AD]


def policy_actions(mode, head_out, z, sigma):
    if mode == 1:
        return np.clip(head_out + sigma * z, -1.0, 1.0)
    mean, log_std = head_out
    return np.tanh(mean + np.exp(log_std) * z)


def explore(layers, head, mode, K, B, AD, seed, step0, obs0, ep_ret0, ep_len0, capacity, pos, sigma=0.1, p_done=0.01,
            max_episode_steps=0, env_offset=0, obs_rows=None):
    """K lock-step steps of B envs.  Returns dict(rows [K,B], obs, next_obs [K,B,D] f32, reward [K,B] f32,
    terminal [K,B] i32, done [K,B] bool, action [K,B,AD] (float32 in mode 0, float64 otherwise), obs_cur, ep_ret,
    ep_len, completed).  The policy is evaluated on ``obs_rows`` [K,B,D] when given (the device's observations, whose
    Box-Muller libm rounding differs from numpy's in the last bits) and on the oracle's own observations otherwise."""
    env = MujocoSynthVec(B, seed, obs_dim=np.asarray(obs0).shape[1], p_done=p_done,
                         max_episode_steps=max_episode_steps, env_offset=env_offset)
    env.step_count = int(step0)
    env.ep_ret = np.asarray(ep_ret0, np.float32).copy()
    env.ep_len = np.asarray(ep_len0, np.int32).copy()
    obs = np.asarray(obs0, np.float32)
    out = dict(rows=[], obs=[], next_obs=[], reward=[], terminal=[], done=[], action=[])
    for t in range(K):
        step = int(step0) + t
        ids = env.ids
        if mode == 0:
            a = uniform_actions(seed, ids, step, AD)
        else:
            x = obs if obs_rows is None else obs_rows[t]
            a = policy_actions(mode, actor_forward64(layers, x, head), gauss64(seed, ids, step, AD), sigma)
        len_before = env.ep_len.copy()
        nobs, rew, done = env.step()
        out['rows'].append(ring_rows(pos, t, B, capacity))
        out['obs'].append(obs)
        out['next_obs'].append(nobs)
        out['reward'].append(rew)
        out['done'].append(done)
        out['terminal'].append(terminal_flags(done, len_before, max_episode_steps))
        out['action'].append(a)
        obs = nobs
    res = {k: np.stack(v) for k, v in out.items()}
    res.update(obs_cur=obs, ep_ret=env.ep_ret, ep_len=env.ep_len, completed=env.completed)
    return res


def sample_rows(n, draw, size, seed):
    """Uniform replay rows of draw ``draw`` over ``size`` rows (exact integer map)."""
    k0, k1 = ph.split_seed(seed)
    x = ph.philox4x32(np.arange(n, dtype=np.uint32), np.uint32(draw), 0, ph.STREAM_REPLAY, k0, k1)[0]
    return ((x.astype(np.uint64) * np.uint64(max(int(size), 1))) >> np.uint64(32)).astype(np.int64)
