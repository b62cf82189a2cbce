"""Functional torch-tensor front end of the C ABI (include/parl_b200.h).

Every function takes/returns CUDA tensors, enqueues exactly the named kernel on
the current stream and never synchronises.  No CPU fallback: CPU tensors raise.
"""
import torch

from . import _lib
from ._lib import ptr, stream, check, require_cuda

TIME_MAJOR = 0
ENV_MAJOR = 1

_workspaces = {}
_graph_launches = 0


def launch_count():
    """C-ABI kernel launches issued so far (eager calls + launches replayed from captured CUDA graphs)."""
    return _lib.launches + _graph_launches


def reset_launch_count():
    global _graph_launches
    _lib.launches = 0
    _graph_launches = 0


def add_graph_launches(n):
    global _graph_launches
    _graph_launches += int(n)


def set_shiftconv_form(form):
    """0 (default): one MMA group per filter tap; 1: column-tap-fused TMA-window conv tiles (measured slower; kept as
    an experiment and cross-check)."""
    _lib.check_config(_lib.load().rl_debug_set_shiftconv_form(int(form)), 'debug_set_shiftconv_form')


def set_gemm_cluster(enable):
    """1 (default): 2 x 2 cluster + TMA multicast form of rl_gemm_bf16_tn where the output has >= 2 x 2 wide tiles."""
    _lib.check_config(_lib.load().rl_debug_set_gemm_cluster(1 if enable else 0), 'debug_set_gemm_cluster')


def set_pdl(enable):
    """1: programmatic dependent launch of the per-env-step chain kernels; 0 (default): plain stream order."""
    _lib.check_config(_lib.load().rl_debug_set_pdl(1 if enable else 0), 'debug_set_pdl')


def set_sm_limit(max_ctas):
    """Cap the CTAs of the persistent network kernels launched from now on (0 = one per SM)."""
    check(_lib.load().rl_set_sm_limit(int(max_ctas)), 'set_sm_limit')
    _lib.launches -= 1


def loss_workspace(device, n_cols):
    """Zero-initialised scratch for the loss kernels (partials + ticket), cached per device."""
    need = _lib.load().rl_loss_workspace_bytes(int(n_cols))
    key = (device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def vtrace_from_importance_weights(behaviour_actions_log_probs, target_actions_log_probs, discounts, rewards, values,
                                   bootstrap_value, clip_rho_threshold=1.0, clip_pg_rho_threshold=1.0):
    """parl/algorithms/paddle/impala/vtrace.py:36-139 on [T,B] float32 CUDA tensors -> (vs, pg_advantages)."""
    args = [behaviour_actions_log_probs, target_actions_log_probs, discounts, rewards, values, bootstrap_value]
    require_cuda(*args)
    T, B = rewards.shape
    vs = torch.empty_like(values)
    pg = torch.empty_like(values)
    cr = -1.0 if clip_rho_threshold is None else float(clip_rho_threshold)
    cp = -1.0 if clip_pg_rho_threshold is None else float(clip_pg_rho_threshold)
    check(_lib.load().rl_vtrace_from_importance_weights(*[ptr(a) for a in args], T, B, cr, cp, ptr(vs), ptr(pg),
                                                        stream()), 'vtrace_from_importance_weights')
    return vs, pg


def vtrace_loss_fwd_bwd(target_logits, behaviour_logits, actions, rewards, dones, values, T, B, gamma,
                        vf_loss_coeff, entropy_coeff, clip_rho_threshold=1.0, clip_pg_rho_threshold=1.0,
                        layout=TIME_MAJOR, want_returns=False, out=None):
    """Fused IMPALA loss + gradient (rl_vtrace_loss_fwd_bwd).

    target_logits / behaviour_logits: [T*B, A] (or [T,B,A]) float32 in `layout` order,
    actions int32/int64, rewards f32, dones bool/uint8, values f32 — all T*B long.
    Returns dict(losses[5] device tensor = total, pi, vf, entropy, kl; d_logits; d_values; vs; pg_advantages).
    """
    require_cuda(target_logits, behaviour_logits, actions, rewards, dones, values)
    A = target_logits.shape[-1]
    assert target_logits.numel() == T * B * A and behaviour_logits.numel() == T * B * A
    assert target_logits.dtype == torch.float32 and behaviour_logits.dtype == torch.float32
    assert actions.dtype in (torch.int32, torch.int64) and actions.numel() == T * B
    if dones.dtype == torch.bool:
        dones = dones.view(torch.uint8)
    assert dones.dtype == torch.uint8 and rewards.dtype == torch.float32 and values.dtype == torch.float32
    dev = target_logits.device
    if out is None:
        out = {}
    losses = out.get('losses')
    if losses is None:
        losses = torch.empty(8, dtype=torch.float32, device=dev)
    d_logits = out.get('d_logits')
    if d_logits is None:
        d_logits = torch.empty_like(target_logits)
    d_values = out.get('d_values')
    if d_values is None:
        d_values = torch.empty_like(values)
    vs = pg = None
    if want_returns:
        vs = torch.empty((T - 1, B), dtype=torch.float32, device=dev)
        pg = torch.empty((T - 1, B), dtype=torch.float32, device=dev)
    ws = loss_workspace(dev, B)
    cr = -1.0 if clip_rho_threshold is None else float(clip_rho_threshold)
    cp = -1.0 if clip_pg_rho_threshold is None else float(clip_pg_rho_threshold)
    check(_lib.load().rl_vtrace_loss_fwd_bwd(
        ptr(target_logits), ptr(behaviour_logits), ptr(actions), 1 if actions.dtype == torch.int64 else 0,
        ptr(rewards), ptr(dones), ptr(values), T, B, A, layout, float(gamma), cr, cp, float(vf_loss_coeff),
        float(entropy_coeff), ptr(losses), ptr(d_logits), ptr(d_values), ptr(vs), ptr(pg), ptr(ws), ws.numel(),
        stream()), 'vtrace_loss_fwd_bwd')
    return dict(losses=losses, d_logits=d_logits, d_values=d_values, vs=vs, pg_advantages=pg)


def _chk(name, t, dtype=None, numel=None, optional=False):
    """dtype / element-count validation of one wrapper argument (the C ABI takes raw pointers)."""
    if t is None:
        if optional:
            return
        raise RuntimeError('parl_b200: %s is required' % name)
    if dtype is not None:
        dts = dtype if isinstance(dtype, (tuple, list)) else (dtype, )
        if t.dtype not in dts:
            raise RuntimeError('parl_b200: %s must be %s, got %s' % (name, ' or '.join(str(d) for d in dts), t.dtype))
    if numel is not None and t.numel() != numel:
        raise RuntimeError('parl_b200: %s must have %d elements, got %d' % (name, numel, t.numel()))


def _as_u8(t):
    """done / terminal flags as uint8 (bool is reinterpreted, float is converted)."""
    if t.dtype == torch.bool:
        return t.view(torch.uint8)
    if t.dtype == torch.uint8:
        return t
    return (t != 0).to(torch.uint8)


# --------------------------------------------------------------------------- envs / sampling
class EpisodeStats(object):
    """Device-side episode bookkeeping shared by the env steppers."""

    def __init__(self, B, device, ring_cap=4096):
        self.ep_ret = torch.zeros(B, dtype=torch.float32, device=device)
        self.ep_len = torch.zeros(B, dtype=torch.int32, device=device)
        self.totals = torch.zeros(4, dtype=torch.float32, device=device)
        self.ring_cap = ring_cap
        self.ring_ret = torch.zeros(max(ring_cap, 1), dtype=torch.float32, device=device)
        self.ring_len = torch.zeros(max(ring_cap, 1), dtype=torch.int32, device=device)
        self.ring_head = torch.zeros(1, dtype=torch.int32, device=device)

    def args(self):
        return [ptr(self.ep_ret), ptr(self.ep_len), ptr(self.totals), ptr(self.ring_ret), ptr(self.ring_len),
                ptr(self.ring_head), self.ring_cap]


def env_atari_synth_step(frame_out, reward_out, done_out, age_in, age_out, stats, seed, step, p_done=0.1,
                         env_offset=0, logits=None, actions_out=None, reset=False, step_dev=None):
    B, HW = frame_out.shape[0], frame_out[0].numel()
    A = logits.shape[-1] if logits is not None else 0
    check(_lib.load().rl_env_atari_synth_step(
        ptr(frame_out), ptr(reward_out), ptr(done_out), ptr(age_in), ptr(age_out), ptr(logits), A, ptr(actions_out),
        *stats.args(), B, HW, int(seed), int(step), ptr(step_dev), int(env_offset), float(p_done),
        1 if reset else 0, stream()), 'env_atari_synth_step')


def env_atari_synth_step_gather(planes, t, reward_out, done_out, age_in, age_out, stats, seed, obs_next, p_done=0.1,
                                env_offset=0, logits=None, actions_out=None, step_dev=None, step=0):
    """Env step of row t (new frame -> planes[t+4]) fused with the uint8 space-to-depth gather of obs(t+1) into
    ``obs_next`` [B,21,21,64] (rl_env_atari_synth_step_gather); 84x84 frames."""
    require_cuda(planes, obs_next)
    P, B = planes.shape[0], planes.shape[1]
    assert planes[0, 0].numel() == 84 * 84 and planes.dtype == torch.uint8 and 0 <= t and t + 4 < P
    assert obs_next.dtype == torch.uint8 and obs_next.numel() == B * 21 * 21 * 64 and obs_next.is_contiguous()
    A = logits.shape[-1] if logits is not None else 0
    check(_lib.load().rl_env_atari_synth_step_gather(
        ptr(planes), int(t), ptr(reward_out), ptr(done_out), ptr(age_in), ptr(age_out), ptr(logits), A, ptr(actions_out),
        *stats.args(), B, int(seed), int(step), ptr(step_dev), int(env_offset), float(p_done), ptr(obs_next), stream()),
        'env_atari_synth_step_gather')


def obs_stack_gather(planes, ages, t_begin, t_count, out, layout=TIME_MAJOR, scale=1.0, s2d=False):
    """planes [P,B,HW] u8, ages [T+1,B] u8 -> out [t_count*B, 4, HW] (uint8 / float32, NCHW) or
    [t_count*B, HW, 4] (bfloat16, NHWC, value*scale)."""
    if ages is None:        # already stacked observations [n,4,84,84] -> space-to-depth (host-contract path)
        assert s2d and planes.dim() == 4 and planes.shape[1] == 4
        B, HW, t_begin, t_count = planes.shape[0], planes[0, 0].numel(), 0, 1
    else:
        P, B, HW = planes.shape[0], planes.shape[1], planes[0, 0].numel()
    dt = {torch.uint8: 0, torch.float32: 1, torch.bfloat16: 2}[out.dtype]
    if s2d:
        # bfloat16: value * scale; uint8: bytes untouched (the conv1 kernels scale while widening, u8in variants)
        assert out.dtype in (torch.bfloat16, torch.uint8) and out.numel() == t_count * B * 21 * 21 * 64
        dt = 3 if out.dtype == torch.bfloat16 else 4
    else:
        assert out.numel() == t_count * B * 4 * HW
    check(_lib.load().rl_obs_stack_gather(ptr(planes), ptr(ages), B, HW, int(t_begin), int(t_count), layout, dt,
                                          float(scale), ptr(out), stream()), 'obs_stack_gather')
    return out


def env_mujoco_synth_step(obs_out, reward_out, done_out, stats, seed, step, p_done=0.01, max_episode_steps=0,
                          env_offset=0, reset=False):
    B, D = obs_out.shape
    check(_lib.load().rl_env_mujoco_synth_step(
        ptr(obs_out), ptr(reward_out), ptr(done_out), *stats.args(), B, D, int(max_episode_steps), int(seed),
        int(step), int(env_offset), float(p_done), 1 if reset else 0, stream()), 'env_mujoco_synth_step')


def env_cartpole_step(state, obs_out, reward_out, done_out, actions, stats, seed, step, max_episode_steps=200,
                      env_offset=0, reset=False):
    B = state.shape[0]
    check(_lib.load().rl_env_cartpole_step(
        ptr(state), ptr(obs_out), ptr(reward_out), ptr(done_out), ptr(actions), *stats.args(), B,
        int(max_episode_steps), int(seed), int(step), int(env_offset), 1 if reset else 0, stream()),
        'env_cartpole_step')


def sample_categorical(logits, seed, step, env_offset=0, want_logp=False):
    require_cuda(logits)
    _chk('logits', logits, torch.float32)
    N, A = logits.shape
    actions = torch.empty(N, dtype=torch.int32, device=logits.device)
    logp = torch.empty(N, dtype=torch.float32, device=logits.device) if want_logp else None
    check(_lib.load().rl_sample_categorical(ptr(logits), N, A, int(seed), int(step), int(env_offset), ptr(actions),
                                            ptr(logp), stream()), 'sample_categorical')
    return (actions, logp) if want_logp else actions


def sample_gaussian(mean, logstd, seed, step, env_offset=0):
    require_cuda(mean, logstd)
    N, D = mean.shape
    _chk('mean', mean, torch.float32)
    _chk('logstd', logstd, torch.float32, D)
    action = torch.empty_like(mean)
    logp = torch.empty(N, dtype=torch.float32, device=mean.device)
    check(_lib.load().rl_sample_gaussian(ptr(mean), ptr(logstd), N, D, int(seed), int(step), int(env_offset),
                                         ptr(action), ptr(logp), stream()), 'sample_gaussian')
    return action, logp


# --------------------------------------------------------------------------- flat losses / scans
def _flat_ws(device, n_rows, extra=0):
    need = _lib.load().rl_flat_workspace_bytes(int(n_rows), int(extra))
    key = ('flat', device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _act_flag(actions):
    assert actions.dtype in (torch.int32, torch.int64)
    return 1 if actions.dtype == torch.int64 else 0


def a2c_loss_fwd_bwd(logits, values, actions, advantages, target_values, vf_loss_coeff, entropy_coeff):
    """parl/algorithms/torch/a2c.py:40-60 -> dict(losses[4]={total,pi,vf,entropy}, d_logits, d_values)."""
    require_cuda(logits, values, actions, advantages, target_values)
    N, A = logits.shape
    _chk('logits', logits, torch.float32)
    _chk('values', values, torch.float32, N)
    _chk('actions', actions, (torch.int32, torch.int64), N)
    _chk('advantages', advantages, torch.float32, N)
    _chk('target_values', target_values, torch.float32, N)
    dev = logits.device
    losses = torch.empty(4, dtype=torch.float32, device=dev)
    d_logits, d_values = torch.empty_like(logits), torch.empty_like(values)
    ws = _flat_ws(dev, N)
    check(_lib.load().rl_a2c_loss_fwd_bwd(ptr(logits), ptr(values), ptr(actions), _act_flag(actions), ptr(advantages),
                                          ptr(target_values), N, A, float(vf_loss_coeff), float(entropy_coeff),
                                          ptr(losses), ptr(d_logits), ptr(d_values), ptr(ws), ws.numel(), stream()),
          'a2c_loss_fwd_bwd')
    return dict(losses=losses, d_logits=d_logits, d_values=d_values)


def gae_scan_segments(rewards, values, dones, bootstrap_value, gamma, lam):
    """calc_gae per episode segment (rl_utils.py:34-51, a2c/actor.py:82-102) on [T,B] -> (adv, target_values)."""
    require_cuda(rewards, values, dones, bootstrap_value)
    dones = _as_u8(dones)
    T, B = rewards.shape
    _chk('rewards', rewards, torch.float32)
    _chk('values', values, torch.float32, T * B)
    _chk('dones', dones, torch.uint8, T * B)
    _chk('bootstrap_value', bootstrap_value, torch.float32, B)
    adv, tv = torch.empty_like(rewards), torch.empty_like(rewards)
    check(_lib.load().rl_gae_scan_segments(ptr(rewards), ptr(values), ptr(dones), ptr(bootstrap_value), T, B,
                                           float(gamma), float(lam), ptr(adv), ptr(tv), stream()), 'gae_scan_segments')
    return adv, tv


def gae_scan(rewards, values, dones, last_value, last_done, gamma=0.99, gae_lambda=0.95, out=None):
    """RolloutStorage.compute_returns (benchmark/torch/ppo/storage.py:45-64) -> (advantages, returns)."""
    require_cuda(rewards, values, dones, last_value, last_done)
    T, B = rewards.shape
    # the kernel reads the done flags as float32 (RolloutStorage keeps them as float, storage.py:31)
    if dones.dtype != torch.float32:
        dones = dones.float()
    if last_done.dtype != torch.float32:
        last_done = last_done.float()
    _chk('rewards', rewards, torch.float32)
    _chk('values', values, torch.float32, T * B)
    _chk('dones', dones, torch.float32, T * B)
    _chk('last_value', last_value, torch.float32, B)
    _chk('last_done', last_done, torch.float32, B)
    adv, ret = out if out is not None else (torch.empty_like(rewards), torch.empty_like(rewards))
    _chk('advantages', adv, torch.float32, T * B)
    _chk('returns', ret, torch.float32, T * B)
    check(_lib.load().rl_gae_scan(ptr(rewards), ptr(values), ptr(dones), ptr(last_value), ptr(last_done), T, B,
                                  float(gamma), float(gae_lambda), ptr(adv), ptr(ret), stream()), 'gae_scan')
    return adv, ret


def adv_stats(adv):
    require_cuda(adv)
    _chk('adv', adv, torch.float32)
    stats = torch.empty(2, dtype=torch.float32, device=adv.device)
    check(_lib.load().rl_adv_stats(ptr(adv), adv.numel(), ptr(stats), stream()), 'adv_stats')
    return stats


def ppo_loss_fwd_bwd(values, batch_action, batch_value, batch_return, batch_logprob, batch_adv, logits=None,
                     mean=None, logstd=None, clip_param=0.1, value_loss_coef=0.5, entropy_coef=0.01,
                     use_clipped_value_loss=True, norm_adv=True, stats=None):
    """parl/algorithms/torch/ppo.py:102-138 -> dict(losses[4]={value,action,entropy,total}, d_values, d_logits|d_mean,d_logstd)."""
    require_cuda(values, batch_action, batch_value, batch_return, batch_logprob, batch_adv, logits, mean, logstd)
    dev = values.device
    N = values.numel()
    for nm, t in (('values', values), ('batch_value', batch_value), ('batch_return', batch_return),
                  ('batch_logprob', batch_logprob), ('batch_adv', batch_adv)):
        _chk(nm, t, torch.float32, N)
    if logits is not None:
        _chk('logits', logits, torch.float32, N * logits.shape[-1])
        _chk('batch_action', batch_action, (torch.int32, torch.int64), N)
    else:
        _chk('mean', mean, torch.float32, N * mean.shape[-1])
        _chk('logstd', logstd, torch.float32, mean.shape[-1])
        _chk('batch_action', batch_action, torch.float32, mean.numel())
    _chk('stats', stats, torch.float32, 2, optional=True)
    if norm_adv and stats is None:
        stats = adv_stats(batch_adv)
    if not norm_adv:
        stats = None
    losses = torch.empty(4, dtype=torch.float32, device=dev)
    d_values = torch.empty_like(values)
    if logits is not None:
        AD = logits.shape[-1]
        d_main, d_ls, flag = torch.empty_like(logits), None, _act_flag(batch_action)
    else:
        AD = mean.shape[-1]
        assert batch_action.dtype == torch.float32
        d_main, d_ls, flag = torch.empty_like(mean), torch.empty_like(logstd), 0
    ws = _flat_ws(dev, N, AD)
    check(_lib.load().rl_ppo_loss_fwd_bwd(
        ptr(logits), ptr(mean), ptr(logstd), ptr(batch_action), flag, ptr(values), ptr(batch_value), ptr(batch_return),
        ptr(batch_logprob), ptr(batch_adv), ptr(stats), N, AD, float(clip_param), float(value_loss_coef),
        float(entropy_coef), 1 if use_clipped_value_loss else 0, ptr(losses), ptr(d_main), ptr(d_ls), ptr(d_values),
        ptr(ws), ws.numel(), stream()), 'ppo_loss_fwd_bwd')
    out = dict(losses=losses, d_values=d_values)
    if logits is not None:
        out['d_logits'] = d_main
    else:
        out['d_mean'], out['d_logstd'] = d_main, d_ls
    return out


def td_loss_fwd_bwd(q, q_target_next, action, reward, terminal, gamma, q_online_next=None, weights=None,
                    want_td_abs=False):
    """dqn.py:64-69 / ddqn.py:64-72 / per_alg.py:48-69 -> dict(losses[1], d_q, td_abs)."""
    require_cuda(q, q_target_next, action, reward, terminal, q_online_next, weights)
    M, A = q.shape
    dev = q.device
    _chk('q', q, torch.float32)
    _chk('q_target_next', q_target_next, torch.float32, M * A)
    _chk('q_online_next', q_online_next, torch.float32, M * A, optional=True)
    _chk('action', action, (torch.int32, torch.int64), M)
    _chk('reward', reward, torch.float32, M)
    _chk('terminal', terminal, torch.float32, M)
    _chk('weights', weights, torch.float32, M, optional=True)
    losses = torch.empty(1, dtype=torch.float32, device=dev)
    d_q = torch.empty_like(q)
    td = torch.empty(M, dtype=torch.float32, device=dev) if want_td_abs else None
    ws = _flat_ws(dev, M)
    check(_lib.load().rl_td_loss_fwd_bwd(ptr(q), ptr(q_target_next), ptr(q_online_next), ptr(action), _act_flag(action),
                                         ptr(reward), ptr(terminal), ptr(weights), M, A, float(gamma), ptr(losses),
                                         ptr(d_q), ptr(td), ptr(ws), ws.numel(), stream()), 'td_loss_fwd_bwd')
    return dict(losses=losses, d_q=d_q, td_abs=td)


def twin_q_td_loss_fwd_bwd(q1, q1_target_next, reward, terminal, gamma, q2=None, q2_target_next=None,
                           next_log_prob=None, alpha=0.0, want_target=False):
    """Continuous-control critic TD (ddpg.py:63-73 / td3.py:78-94 / sac.py:90-99) ->
    dict(losses[3] = total, mse1, mse2; d_q1; d_q2 or None; target or None).  All inputs are [N] (or [N,1]) float32."""
    require_cuda(q1, q1_target_next, reward, terminal, q2, q2_target_next, next_log_prob)
    N = q1.numel()
    dev = q1.device
    _chk('q1', q1, torch.float32)
    _chk('q2', q2, torch.float32, N, optional=True)
    _chk('q1_target_next', q1_target_next, torch.float32, N)
    _chk('q2_target_next', q2_target_next, torch.float32, N, optional=True)
    _chk('next_log_prob', next_log_prob, torch.float32, N, optional=True)
    _chk('reward', reward, torch.float32, N)
    _chk('terminal', terminal, torch.float32, N)
    for t in (q1, q2, q1_target_next, q2_target_next, next_log_prob, reward, terminal):
        assert t is None or t.is_contiguous(), 'twin_q_td_loss: tensors must be contiguous'
    losses = torch.zeros(3, dtype=torch.float32, device=dev)
    d_q1 = torch.empty_like(q1)
    d_q2 = torch.empty_like(q2) if q2 is not None else None
    target = torch.empty(N, dtype=torch.float32, device=dev) if want_target else None
    ws = _flat_ws(dev, N)
    check(_lib.load().rl_twin_q_td_loss_fwd_bwd(ptr(q1), ptr(q2), ptr(q1_target_next), ptr(q2_target_next),
                                                ptr(next_log_prob), ptr(reward), ptr(terminal), N, float(gamma),
                                                float(alpha), ptr(losses), ptr(d_q1), ptr(d_q2), ptr(target), ptr(ws),
                                                ws.numel(), stream()), 'twin_q_td_loss_fwd_bwd')
    return dict(losses=losses, d_q1=d_q1, d_q2=d_q2, target=target)


def pg_loss_fwd_bwd(prob, action, reward):
    """policy_gradient.py:54-75 -> dict(losses[1], d_prob)."""
    require_cuda(prob, action, reward)
    N, A = prob.shape
    _chk('prob', prob, torch.float32)
    _chk('action', action, (torch.int32, torch.int64), N)
    _chk('reward', reward, torch.float32, N)
    losses = torch.empty(1, dtype=torch.float32, device=prob.device)
    d_prob = torch.empty_like(prob)
    ws = _flat_ws(prob.device, N)
    check(_lib.load().rl_pg_loss_fwd_bwd(ptr(prob), ptr(action), _act_flag(action), ptr(reward), N, A, ptr(losses),
                                         ptr(d_prob), ptr(ws), ws.numel(), stream()), 'pg_loss_fwd_bwd')
    return dict(losses=losses, d_prob=d_prob)


# --------------------------------------------------------------------------- replay
class DeviceSumTree(object):
    """fp64 sum-tree in HBM with the reference's heap indexing (proportional_per.py:18-70)."""

    def __init__(self, capacity, device):
        self.capacity = int(capacity)
        self.tree = torch.zeros(2 * self.capacity - 1, dtype=torch.float64, device=device)
        self.state = torch.tensor([10.0, 1.0], dtype=torch.float64, device=device)   # _min, _max_priority

    def store(self, write_pos, n, alpha, eps, delta=None):
        _chk('delta', delta, torch.float32, int(n), optional=True)
        check(_lib.load().rl_per_store(ptr(self.tree), ptr(self.state), self.capacity, int(write_pos), int(n),
                                       ptr(delta), float(alpha), float(eps), stream()), 'per_store')

    def update(self, tree_idx, priorities, alpha, eps):
        _chk('tree_idx', tree_idx, torch.int32)
        _chk('priorities', priorities, torch.float32, tree_idx.numel())
        check(_lib.load().rl_per_update(ptr(self.tree), ptr(self.state), self.capacity, ptr(tree_idx), ptr(priorities),
                                        tree_idx.numel(), float(alpha), float(eps), stream()), 'per_update')

    def sample(self, seg_num, beta, size, u=None, seed=0, draw=0):
        dev = self.tree.device
        _chk('u', u, torch.float32, int(seg_num), optional=True)
        tidx = torch.empty(seg_num, dtype=torch.int32, device=dev)
        eidx = torch.empty(seg_num, dtype=torch.int32, device=dev)
        w = torch.empty(seg_num, dtype=torch.float32, device=dev)
        check(_lib.load().rl_per_sample(ptr(self.tree), ptr(self.state), self.capacity, int(seg_num), ptr(u), int(seed),
                                        int(draw), float(beta), float(size), ptr(tidx), ptr(eidx), ptr(w), stream()),
              'per_sample')
        return tidx, eidx, w


def replay_gather_frames(frames, is_over, idx, curr_size, context_len, lanes=1, n_out=None, out=None):
    """benchmark/torch/dqn/replay_memory.py:59-85 for a batch of start indices -> [n, n_out (default ctx+1), HW]
    uint8; ``lanes`` interleaved per-env streams (row = position*lanes + lane), see include/parl_b200.h."""
    require_cuda(frames, is_over, idx)
    HW = frames[0].numel()
    n = idx.numel()
    _chk('frames', frames, torch.uint8)
    _chk('idx', idx, torch.int32)
    n_out = context_len + 1 if n_out is None else int(n_out)
    if out is None:
        out = torch.empty((n, n_out, HW), dtype=torch.uint8, device=frames.device)
    _chk('out', out, torch.uint8, n * n_out * HW)
    is_over = _as_u8(is_over)
    _chk('is_over', is_over, torch.uint8, frames.numel() // HW)
    check(_lib.load().rl_replay_gather_frames(ptr(frames), ptr(is_over), ptr(idx), n, int(curr_size), int(context_len),
                                              HW, int(lanes), n_out, ptr(out), stream()), 'replay_gather_frames')
    return out


def gather_rows(src, idx):
    """out[i] = src[idx[i]] for a 2-D (or N-D, row-contiguous) tensor with 4-byte-multiple rows."""
    require_cuda(src, idx)
    assert idx.dtype == torch.int32
    row_bytes = src[0].numel() * src.element_size()
    out = torch.empty((idx.numel(), ) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    check(_lib.load().rl_gather_rows(ptr(src), ptr(idx), idx.numel(), row_bytes, ptr(out), stream()), 'gather_rows')
    return out


def gather_cast(src_flat, idx, out):
    """out[i] = cast(src_flat[idx[i]]) (idx < 0 -> 0), out bfloat16 or float32 (rl_gather_cast): the one-launch refresh
    of the network kernels' operand copies from the flat float32 master buffer."""
    require_cuda(src_flat, idx, out)
    _chk('src', src_flat, torch.float32)
    _chk('idx', idx, torch.int32)
    assert out.dtype in (torch.bfloat16, torch.float32) and out.numel() == idx.numel() and out.is_contiguous()
    check(_lib.load().rl_gather_cast(ptr(src_flat), ptr(idx), idx.numel(), ptr(out), 1 if out.dtype == torch.bfloat16 else 0,
                                     stream()), 'gather_cast')
    return out


# --------------------------------------------------------------------------- optimizer
def grad_global_norm(grad_flat, out_norm):
    _chk('grad', grad_flat, torch.float32)
    _chk('norm', out_norm, torch.float32, 1)
    ws = _flat_ws(grad_flat.device, 1)
    check(_lib.load().rl_grad_global_norm(ptr(grad_flat), grad_flat.numel(), ptr(out_norm), ptr(ws), ws.numel(),
                                          stream()), 'grad_global_norm')
    return out_norm


def adam_step(param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step, grad_div=1.0, grad_norm=None,
              max_norm=0.0, clip_mode=0, zero_grad=True, lr_device=None, step_device=None):
    n = param.numel()
    for nm, t in (('param', param), ('grad', grad), ('exp_avg', exp_avg), ('exp_avg_sq', exp_avg_sq)):
        _chk(nm, t, torch.float32, n)
    _chk('grad_norm', grad_norm, torch.float32, 1, optional=True)
    _chk('lr_device', lr_device, torch.float32, 1, optional=True)
    _chk('step_device', step_device, torch.int32, 1, optional=True)
    check(_lib.load().rl_adam_step(ptr(param), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), param.numel(), ptr(lr_device),
                                   float(lr), float(beta1), float(beta2), float(eps), int(step), float(grad_div),
                                   ptr(grad_norm), float(max_norm), int(clip_mode), 1 if zero_grad else 0,
                                   ptr(step_device), stream()),
          'adam_step')


# --------------------------------------------------------------------------- tensor-core contractions
def gemm_bf16_tn(a, b, bias=None, relu=False, out_dtype=torch.bfloat16, out=None):
    """C = act(a @ b.T + bias) on tcgen05 (rl_gemm_bf16_tn): a [M,K] bf16, b [N,K] bf16 (nn.Linear weight layout)."""
    require_cuda(a, b, bias)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.shape[1] == b.shape[1]
    M, K = a.shape
    N = b.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    assert out.dtype in (torch.bfloat16, torch.float32)
    if M <= 2048 and K >= 1024:
        # few output tiles, long reduction (the actor's fc layer at small per-GPU batch): split-K with a per-stream
        # workspace (two streams never share partials)
        ws = _raw_ws(a.device, 8 << 20, 'gemm_splitk_%d' % torch.cuda.current_stream(a.device).cuda_stream)
        check(_lib.load().rl_gemm_bf16_tn_splitk(ptr(a), ptr(b), ptr(bias), ptr(out), M, N, K, a.stride(0), b.stride(0),
                                                 out.stride(0), 1 if relu else 0,
                                                 1 if out.dtype == torch.float32 else 0, ptr(ws), ws.numel(), stream()),
              'gemm_bf16_tn_splitk')
        return out
    check(_lib.load().rl_gemm_bf16_tn(ptr(a), ptr(b), ptr(bias), ptr(out), M, N, K, a.stride(0), b.stride(0),
                                      out.stride(0), 1 if relu else 0, 1 if out.dtype == torch.float32 else 0,
                                      stream()), 'gemm_bf16_tn')
    return out


def gemm_bf16_tn_heads(a, b, bias, h_out, w2, b2, out2, relu=True):
    """h_out = act(a @ b.T + bias) (bf16) and out2 = h_out @ w2.T + b2 (float32, <= 32 head rows) in one call
    (rl_gemm_bf16_tn_heads): at small batch the split-K reduce and the heads are a single kernel."""
    require_cuda(a, b, bias, h_out, w2, b2, out2)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and w2.dtype == torch.bfloat16
    assert h_out.dtype == torch.bfloat16 and out2.dtype == torch.float32 and bias.dtype == torch.float32
    M, K = a.shape
    N, N2 = b.shape[0], w2.shape[0]
    assert h_out.shape == (M, N) and out2.shape == (M, N2) and w2.shape[1] == N and w2.is_contiguous()
    ws = _raw_ws(a.device, 8 << 20, 'gemm_splitk_%d' % torch.cuda.current_stream(a.device).cuda_stream) \
        if (M <= 2048 and K >= 1024) else None
    check(_lib.load().rl_gemm_bf16_tn_heads(ptr(a), ptr(b), ptr(bias), ptr(h_out), M, N, K, a.stride(0), b.stride(0),
                                            h_out.stride(0), 1 if relu else 0, ptr(w2), ptr(b2), N2, ptr(out2),
                                            out2.stride(0), ptr(ws), ws.numel() if ws is not None else 0, stream()),
          'gemm_bf16_tn_heads')
    return out2


def conv2d_nhwc_bf16_fwd(x, weight_krsc, bias, KH, KW, stride, pad, relu=True, out=None):
    """NHWC bf16 conv forward on tcgen05 (rl_conv2d_nhwc_bf16_fwd): x [N,H,W,Cin], weight [Cout, KH*KW*Cin] (r,s,c)."""
    require_cuda(x, weight_krsc, bias)
    assert x.dtype == torch.bfloat16 and weight_krsc.dtype == torch.bfloat16 and bias.dtype == torch.float32
    N, H, W, Cin = x.shape
    Cout = weight_krsc.shape[0]
    Ho, Wo = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = torch.empty((N, Ho, Wo, Cout), dtype=torch.bfloat16, device=x.device)
    check(_lib.load().rl_conv2d_nhwc_bf16_fwd(ptr(x), ptr(weight_krsc), ptr(bias), ptr(out), N, H, W, Cin, Cout, KH, KW,
                                              stride, pad, 1 if relu else 0, stream()), 'conv2d_nhwc_bf16_fwd')
    return out


def conv2d_s1_nhwc_bf16_fwd(x, weight_krsc, bias, KH, KW, relu=True, out=None, out_mode=0, in_scale=1.0 / 255.0):
    """Stride-1 NHWC bf16 conv forward in TMA-window form (rl_conv2d_s1_nhwc_bf16_fwd); a uint8 ``x`` (conv1 on the
    space-to-depth observation) goes to rl_conv2d_s1_u8in_bf16_fwd, operand = bf16(byte * in_scale)."""
    require_cuda(x, weight_krsc, bias)
    assert x.dtype in (torch.bfloat16, torch.uint8) and weight_krsc.dtype == torch.bfloat16 and bias.dtype == torch.float32
    N, H, W, Cin = x.shape
    Cout = weight_krsc.shape[0]
    if out is None:
        assert out_mode == 0
        out = torch.empty((N, H - KH + 1, W - KW + 1, Cout), dtype=torch.bfloat16, device=x.device)
    if x.dtype == torch.uint8:
        assert Cin == 64
        check(_lib.load().rl_conv2d_s1_u8in_bf16_fwd(ptr(x), float(in_scale), ptr(weight_krsc), ptr(bias), ptr(out), N, H, W,
                                                     Cout, KH, KW, 1 if relu else 0, int(out_mode), stream()),
              'conv2d_s1_u8in_bf16_fwd')
        return out
    check(_lib.load().rl_conv2d_s1_nhwc_bf16_fwd(ptr(x), ptr(weight_krsc), ptr(bias), ptr(out), N, H, W, Cin, Cout, KH,
                                                 KW, 1 if relu else 0, int(out_mode), stream()), 'conv2d_s1_nhwc_bf16_fwd')
    return out


def conv2d_s1_nhwc_bf16_dgrad(dout_grid, weight_t_krsc, KH, KW, out, act_mask=None, out_mode=0):
    """Data gradient of the TMA-window conv (rl_conv2d_s1_nhwc_bf16_dgrad).  dout_grid [N,H,W,Cout] on the
    input grid, weight_t_krsc [Cin, KH*KW*Cout]; out [N,OGH,OGW,Cin] (mode 0) or [N,21,21,32] (mode 2)."""
    require_cuda(dout_grid, weight_t_krsc, out, act_mask)
    N, H, W, Cout = dout_grid.shape
    Cin = weight_t_krsc.shape[0]
    OGH, OGW = (out.shape[1], out.shape[2]) if out_mode == 0 else (0, 0)
    check(_lib.load().rl_conv2d_s1_nhwc_bf16_dgrad(ptr(dout_grid), ptr(weight_t_krsc), ptr(act_mask), ptr(out), N, H, W,
                                                   Cout, Cin, KH, KW, int(out_mode), OGH, OGW, stream()),
          'conv2d_s1_nhwc_bf16_dgrad')
    return out


def _raw_ws(device, nbytes, key):
    k = (key, device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(k)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        _workspaces[k] = ws
    return ws


def conv2d_s1_nhwc_bf16_wgrad(dout_grid, x, KH, KW, dw_krsc=None, accumulate=False, db=None, in_scale=1.0 / 255.0):
    """Weight gradient of the TMA-window conv (rl_conv2d_s1_nhwc_bf16_wgrad) -> dw [Cout, KH*KW*Cin] float32;
    db (optional [Cout] float32) receives the bias gradient from the same pass.  A uint8 ``x`` goes to
    rl_conv2d_s1_u8in_bf16_wgrad (operand = bf16(byte * in_scale))."""
    require_cuda(dout_grid, x, dw_krsc, db)
    N, H, W, Cout = dout_grid.shape
    Cin = x.shape[-1]
    assert x.shape[:3] == dout_grid.shape[:3] and x.dtype in (torch.bfloat16, torch.uint8)
    if dw_krsc is None:
        dw_krsc = torch.empty((Cout, KH * KW * Cin), dtype=torch.float32, device=x.device)
    ws = _raw_ws(x.device, _lib.load().rl_conv_wgrad_workspace_bytes(KH, KW, Cin), 'wgrad')
    if x.dtype == torch.uint8:
        assert Cin == 64
        check(_lib.load().rl_conv2d_s1_u8in_bf16_wgrad(ptr(dout_grid), ptr(x), float(in_scale), ptr(dw_krsc), ptr(db), N, H,
                                                       W, Cout, KH, KW, 1 if accumulate else 0, ptr(ws), ws.numel(),
                                                       stream()), 'conv2d_s1_u8in_bf16_wgrad')
        return dw_krsc
    check(_lib.load().rl_conv2d_s1_nhwc_bf16_wgrad(ptr(dout_grid), ptr(x), ptr(dw_krsc), ptr(db), N, H, W, Cin, Cout, KH, KW,
                                                   1 if accumulate else 0, ptr(ws), ws.numel(), stream()),
          'conv2d_s1_nhwc_bf16_wgrad')
    return dw_krsc


def colsum_bf16(x, out=None):
    """Column sums of a [rows, C] bf16 matrix -> float32 [C] (rl_colsum_bf16)."""
    require_cuda(x, out)
    C = x.shape[-1]
    rows = x.numel() // C
    if out is None:
        out = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = _raw_ws(x.device, 1184 * C * 4, 'colsum')
    check(_lib.load().rl_colsum_bf16(ptr(x), rows, C, ptr(out), ptr(ws), ws.numel(), stream()), 'colsum_bf16')
    return out


def gemm_bf16_tn_masked(a, b, mask, out):
    """out = (a @ b.T) * (mask > 0) on tcgen05 (rl_gemm_bf16_tn_masked); row strides of a / b / out / mask may
    exceed their widths (sub-matrix views)."""
    require_cuda(a, b)
    M, K = a.shape
    N = b.shape[0]
    assert out.shape == (M, N) and mask.shape == (M, N) and a.stride(1) == 1 and out.stride(1) == 1 and mask.stride(1) == 1
    check(_lib.load().rl_gemm_bf16_tn_masked(ptr(a), ptr(b), ptr(out), ptr(mask), M, N, K, a.stride(0), b.stride(0),
                                             out.stride(0), mask.stride(0), 1 if out.dtype == torch.float32 else 0,
                                             stream()), 'gemm_bf16_tn_masked')
    return out


def bias_act_bf16(x, bias, relu=True):
    require_cuda(x, bias)
    assert x.dtype == torch.bfloat16 and bias.dtype == torch.float32
    N = x.shape[-1]
    check(_lib.load().rl_bias_act_bf16(ptr(x), ptr(bias), x.numel() // N, N, 1 if relu else 0, stream()), 'bias_act_bf16')
    return x


def mask_scatter_grid_bf16(src, act, dst, n, PH, PW, GH, GW, C):
    require_cuda(src, act, dst)
    check(_lib.load().rl_mask_scatter_grid_bf16(ptr(src), ptr(act), ptr(dst), int(n), PH, PW, GH, GW, C, stream()),
          'mask_scatter_grid_bf16')
    return dst


# --------------------------------------------------------------------------- fused fp32 MLP (K6, MLP model family)
ACT_RELU, ACT_TANH, ACT_NONE = 0, 1, 2
HEAD_TANH, HEAD_MEAN_LOGSTD = 0, 1                       # rl_explore_mlp actor heads
EXPLORE_WARMUP, EXPLORE_NOISE, EXPLORE_SAC = 0, 1, 2     # rl_explore_mlp exploration rules


class MlpPlan(object):
    """Shape + parameter-pointer tables of one MLP for rl_mlp_fwd / rl_mlp_bwd.

    ``layers`` is a list (one entry per linear layer) of lists of (weight, bias) tensors — the row segments of that
    layer in torch nn.Linear layout; the last layer's segments are the heads (outputs concatenated).  Pointers are
    taken once: parameters re-homed into a FlatAdam buffer keep their addresses, so build the plan AFTER the
    optimiser.  ``grads`` may be given as matching (dweight, dbias) tensors (default: the parameters' .grad)."""

    def __init__(self, layers, act):
        import ctypes
        self.act = int(act)
        segs = []
        dims = [layers[0][0][0].shape[1]]
        for li, seg_list in enumerate(layers):
            rows = 0
            for (w, b) in seg_list:
                require_cuda(w, b)
                assert w.dtype == torch.float32 and w.dim() == 2 and w.shape[1] == dims[li], 'layer %d weight' % li
                assert b is None or (b.dtype == torch.float32 and b.numel() == w.shape[0])
                segs.append((li, w, b))
                rows += w.shape[0]
            dims.append(rows)
        self.dims_list = dims
        self.n_layers = len(layers)
        self.segs = segs
        self.device = segs[0][1].device
        n = len(segs)
        IntA, PtrA = ctypes.c_int * n, ctypes.c_void_p * n
        self.c_dims = (ctypes.c_int * len(dims))(*dims)
        self.c_layer = IntA(*[s[0] for s in segs])
        self.c_rows = IntA(*[s[1].shape[0] for s in segs])
        self.c_w = PtrA(*[s[1].data_ptr() for s in segs])
        self.c_b = PtrA(*[(s[2].data_ptr() if s[2] is not None else None) for s in segs])
        self._PtrA = PtrA
        self._grad_tabs = None
        self.ws = torch.empty(int(_lib.load().rl_mlp_workspace_bytes(self.n_layers, self.c_dims)), dtype=torch.uint8,
                              device=self.device)

    @property
    def out_dim(self):
        return self.dims_list[-1]

    def forward(self, x, out=None, out2=None, split=0):
        """x [n, in] -> out [n, out_dim]; with ``split`` the output columns are delivered as two dense tensors
        (out [n, split], out2 [n, out_dim - split]) — e.g. the policy head and the value head."""
        require_cuda(x, out, out2)
        assert x.dtype == torch.float32 and x.dim() == 2 and x.shape[1] == self.dims_list[0]
        n = x.shape[0]
        first = split if split else self.out_dim
        if out is None:
            out = torch.empty((n, first), dtype=torch.float32, device=x.device)
        _chk('out', out, torch.float32, n * first)
        if split:
            if out2 is None:
                out2 = torch.empty((n, self.out_dim - split), dtype=torch.float32, device=x.device)
            _chk('out2', out2, torch.float32, n * (self.out_dim - split))
        check(_lib.load().rl_mlp_fwd(ptr(x), n, self.n_layers, self.c_dims, len(self.segs), self.c_layer, self.c_rows,
                                     self.c_w, self.c_b, self.act, ptr(out), ptr(out2) if split else None, int(split),
                                     stream()), 'mlp_fwd')
        return (out, out2) if split else out

    def backward(self, x, d_out, grads=None, accumulate=False, d_out2=None, split=0):
        """Parameter gradients of sum(out * d_out) into ``grads`` [(dw, db), ...] (default: each parameter's .grad)."""
        require_cuda(x, d_out, d_out2)
        n = x.shape[0]
        _chk('x', x, torch.float32, n * self.dims_list[0])
        _chk('d_out', d_out, torch.float32, n * (split if split else self.out_dim))
        if split:
            _chk('d_out2', d_out2, torch.float32, n * (self.out_dim - split))
        if grads is None:
            if self._grad_tabs is None:
                gw = [s[1].grad for s in self.segs]
                gb = [(s[2].grad if s[2] is not None else None) for s in self.segs]
                assert all(g is not None for g in gw), 'parameters have no .grad buffers (build a FlatAdam first)'
                self._grad_tabs = (self._PtrA(*[g.data_ptr() for g in gw]),
                                   self._PtrA(*[(g.data_ptr() if g is not None else None) for g in gb]), gw, gb)
            c_dw, c_db = self._grad_tabs[0], self._grad_tabs[1]
        else:
            c_dw = self._PtrA(*[g[0].data_ptr() for g in grads])
            c_db = self._PtrA(*[(g[1].data_ptr() if g[1] is not None else None) for g in grads])
        check(_lib.load().rl_mlp_bwd(ptr(x), n, self.n_layers, self.c_dims, len(self.segs), self.c_layer, self.c_rows,
                                     self.c_w, self.c_b, self.act, ptr(d_out), ptr(d_out2) if split else None,
                                     int(split), c_dw, c_db, 1 if accumulate else 0, ptr(self.ws), self.ws.numel(),
                                     stream()), 'mlp_bwd')

    def rollout(self, env_kind, policy_kind, T, obs_cur, stats, seed, step0, obs_out, act_out, rew_out, done_out,
                logp_out=None, val_out=None, logits_out=None, logstd=None, has_value=True, env_offset=0, p_done=0.01,
                max_episode_steps=0, vecnorm=None):
        """rl_rollout_mlp: T lock-step steps of all envs in ONE launch (policy forward + sampling + env step)."""
        require_cuda(obs_cur, obs_out, act_out, rew_out, done_out, logp_out, val_out, logits_out, logstd)
        B, D = obs_cur.shape
        AD = self.out_dim - (1 if has_value else 0)
        _chk('obs_cur', obs_cur, torch.float32, B * self.dims_list[0])
        _chk('obs_out', obs_out, torch.float32, T * B * D)
        _chk('act_out', act_out, torch.int32 if policy_kind == 0 else torch.float32, T * B * (1 if policy_kind == 0 else AD))
        _chk('rew_out', rew_out, torch.float32, T * B)
        _chk('done_out', done_out, torch.uint8, T * B)
        _chk('logp_out', logp_out, torch.float32, T * B, optional=True)
        _chk('val_out', val_out, torch.float32, (T + 1) * B, optional=True)
        _chk('logits_out', logits_out, torch.float32, T * B * AD, optional=True)
        _chk('logstd', logstd, torch.float32, AD, optional=policy_kind == 0)
        check(_lib.load().rl_rollout_mlp(self.n_layers, self.c_dims, len(self.segs), self.c_layer, self.c_rows, self.c_w,
                                         self.c_b, self.act, int(env_kind), int(policy_kind), int(T), B, AD,
                                         1 if has_value else 0, ptr(logstd), ptr(obs_cur), *stats.args(), int(seed),
                                         int(step0), int(env_offset), float(p_done), int(max_episode_steps),
                                         ptr(obs_out), ptr(act_out), ptr(logp_out), ptr(val_out), ptr(logits_out),
                                         ptr(rew_out), ptr(done_out),
                                         vecnorm.c_state if vecnorm is not None else None,
                                         vecnorm.c_cfg if vecnorm is not None else None,
                                         vecnorm.flags if vecnorm is not None else 0, stream()), 'rollout_mlp')

    def explore(self, memory, mode, K, obs_cur, stats, seed, step0, head=HEAD_TANH, expl_noise=0.1, env_offset=0,
                p_done=0.01, max_episode_steps=1000):
        """rl_explore_mlp: K lock-step steps of B = obs_cur.shape[0] envs in ONE launch (actor forward + exploration
        rule + env step), transitions written into ``memory`` (a utils.ReplayMemory) at rows
        (memory._curr_pos + t*B + b) % memory.max_size.  The caller advances the memory with ``memory.commit(K*B)``."""
        if self.act != ACT_RELU:
            raise RuntimeError('parl_b200: explore needs ReLU hidden layers (act %d)' % self.act)
        if head not in (HEAD_TANH, HEAD_MEAN_LOGSTD):
            raise RuntimeError('parl_b200: explore head must be HEAD_TANH or HEAD_MEAN_LOGSTD, got %r' % (head, ))
        if int(mode) not in (EXPLORE_WARMUP, EXPLORE_NOISE, EXPLORE_SAC):
            raise RuntimeError('parl_b200: explore mode must be 0, 1 or 2, got %r' % (mode, ))
        if int(mode) == EXPLORE_NOISE and head != HEAD_TANH:
            raise RuntimeError('parl_b200: explore mode 1 needs the tanh head')
        if int(mode) == EXPLORE_SAC and head != HEAD_MEAN_LOGSTD:
            raise RuntimeError('parl_b200: explore mode 2 needs the mean|log-std head')
        AD = self.out_dim if head == HEAD_TANH else self.out_dim // 2
        D = self.dims_list[0]
        m = memory
        require_cuda(obs_cur, m.obs, m.action, m.reward, m.terminal, m.next_obs)
        if obs_cur.dim() != 2 or obs_cur.shape[1] != D:
            raise RuntimeError('parl_b200: obs_cur must be [B, %d], got %s' % (D, tuple(obs_cur.shape)))
        B, cap = obs_cur.shape[0], m.max_size
        _chk('obs_cur', obs_cur, torch.float32, B * D)
        _chk('memory.obs', m.obs, torch.float32, cap * D)
        _chk('memory.next_obs', m.next_obs, torch.float32, cap * D)
        _chk('memory.action', m.action, torch.float32, cap * AD)
        _chk('memory.reward', m.reward, torch.float32, cap)
        _chk('memory.terminal', m.terminal, torch.int32, cap)
        _chk('stats.ep_len', stats.ep_len, torch.int32, B)
        if int(K) < 1 or int(K) * B > cap:
            raise RuntimeError('parl_b200: explore K*B = %d transitions must be in 1..%d (the replay capacity)'
                               % (int(K) * B, cap))
        check(_lib.load().rl_explore_mlp(self.n_layers, self.c_dims, len(self.segs), self.c_layer, self.c_rows, self.c_w,
                                         self.c_b, int(head), int(mode), int(K), B, AD, float(expl_noise), ptr(obs_cur),
                                         *stats.args(), int(seed), int(step0), int(env_offset), float(p_done),
                                         int(max_episode_steps), ptr(m.obs), ptr(m.action), ptr(m.reward),
                                         ptr(m.terminal), ptr(m.next_obs), cap, int(m._curr_pos), stream()),
              'explore_mlp')


def replay_sample_uniform(memory, n, size_dev, draw_dev, seed, out=None, want_idx=False):
    """rl_replay_sample_uniform: n uniform rows of the first min(size_dev[0], memory.max_size) rows of ``memory`` (a
    utils.ReplayMemory with float actions) -> (obs, action, reward [n], next_obs, terminal [n]) float32 device tensors
    (``out``: the same tuple preallocated), plus the int32 rows with ``want_idx``.  size_dev / draw_dev: int32 [1]
    device tensors."""
    m = memory
    require_cuda(m.obs, m.action, m.reward, m.terminal, m.next_obs, size_dev, draw_dev)
    cap, D = m.obs.shape
    AD = m.action.shape[1]
    _chk('memory.obs', m.obs, torch.float32, cap * D)
    _chk('memory.next_obs', m.next_obs, torch.float32, cap * D)
    _chk('memory.action', m.action, torch.float32, cap * AD)
    _chk('memory.reward', m.reward, torch.float32, cap)
    _chk('memory.terminal', m.terminal, torch.int32, cap)
    _chk('size_dev', size_dev, torch.int32, 1)
    _chk('draw_dev', draw_dev, torch.int32, 1)
    n = int(n)
    if n < 1:
        raise RuntimeError('parl_b200: replay_sample_uniform needs n >= 1, got %d' % n)
    dev = m.obs.device
    if out is None:
        f32 = torch.float32
        out = (torch.empty((n, D), dtype=f32, device=dev), torch.empty((n, AD), dtype=f32, device=dev),
               torch.empty(n, dtype=f32, device=dev), torch.empty((n, D), dtype=f32, device=dev),
               torch.empty(n, dtype=f32, device=dev))
    obs, act, rew, nobs, term = out
    require_cuda(obs, act, rew, nobs, term)
    for nm, t, k in (('obs', obs, n * D), ('action', act, n * AD), ('reward', rew, n), ('next_obs', nobs, n * D),
                     ('terminal', term, n)):
        _chk(nm, t, torch.float32, k)
    idx = torch.empty(n, dtype=torch.int32, device=dev) if want_idx else None
    check(_lib.load().rl_replay_sample_uniform(ptr(m.obs), ptr(m.action), ptr(m.reward), ptr(m.terminal),
                                               ptr(m.next_obs), D, AD, ptr(size_dev), ptr(draw_dev), cap, n, int(seed),
                                               ptr(obs), ptr(act), ptr(rew), ptr(term), ptr(nobs), ptr(idx), stream()),
          'replay_sample_uniform')
    return (obs, act, rew, nobs, term, idx) if want_idx else (obs, act, rew, nobs, term)


ENV_MUJOCO_SYNTH, ENV_CARTPOLE = 0, 1
POLICY_CATEGORICAL, POLICY_GAUSSIAN = 0, 1


class VecNormalize(object):
    """Device VecNormalizeEnv state for B envs of obs dim D (rl_vecnormalize_step / the fused rollout):
    per-env running observation statistics and return statistics in float64 (parl/env/mujoco_wrappers.py:95-168)."""

    def __init__(self, B, D, device, ob=True, ret=True, clipob=10.0, cliprew=10.0, gamma=0.99, epsilon=1e-8):
        import ctypes
        f64 = torch.float64
        self.B, self.D = int(B), int(D)
        self.ob_mean = torch.zeros((B, D), dtype=f64, device=device)
        self.ob_var = torch.ones((B, D), dtype=f64, device=device)
        self.ob_count = torch.full((B, ), 1e-4, dtype=f64, device=device)
        self.ret = torch.zeros(B, dtype=f64, device=device)
        self.ret_mean = torch.zeros(B, dtype=f64, device=device)
        self.ret_var = torch.ones(B, dtype=f64, device=device)
        self.ret_count = torch.full((B, ), 1e-4, dtype=f64, device=device)
        self.ob, self.norm_ret, self.training = bool(ob), bool(ret), True
        self.clipob, self.cliprew, self.gamma, self.epsilon = float(clipob), float(cliprew), float(gamma), float(epsilon)
        self._state = [self.ob_mean, self.ob_var, self.ob_count, self.ret, self.ret_mean, self.ret_var, self.ret_count]
        self.c_state = (ctypes.c_void_p * 7)(*[t.data_ptr() for t in self._state])
        self.c_cfg = (ctypes.c_double * 4)(self.clipob, self.cliprew, self.gamma, self.epsilon)

    @property
    def flags(self):
        return (1 if self.training else 0) | (2 if self.ob else 0) | (4 if self.norm_ret else 0)

    def train(self):
        self.training = True

    def eval(self):
        self.training = False

    def _call(self, obs_in, obs_out, reward, done, term_obs, reward_step):
        require_cuda(obs_in, obs_out, reward, done, term_obs)
        _chk('obs', obs_in, torch.float32, self.B * self.D)
        _chk('obs_out', obs_out, torch.float32, self.B * self.D)
        _chk('reward', reward, torch.float32, self.B, optional=not reward_step)
        _chk('done', done, torch.uint8, self.B, optional=not reward_step)
        _chk('terminal_obs', term_obs, torch.float32, self.B * self.D, optional=True)
        check(_lib.load().rl_vecnormalize_step(ptr(obs_in), ptr(term_obs), ptr(obs_out), ptr(reward), ptr(done),
                                               *[ptr(t) for t in self._state], self.B, self.D,
                                               1 if self.training else 0, 1 if self.ob else 0,
                                               1 if self.norm_ret else 0, 1 if reward_step else 0, self.clipob,
                                               self.cliprew, self.gamma, self.epsilon, stream()), 'vecnormalize_step')
        return obs_out

    def reset(self, obs, out=None):
        """VecNormalizeEnv.reset(): filter the first observations ([B, D] float32; in place unless ``out``)."""
        self.ret.zero_()
        return self._call(obs, obs if out is None else out, None, None, None, False)

    def step(self, obs, reward, done, terminal_obs=None, out=None):
        """VecNormalizeEnv.step() (+ reset where done): reward is normalised IN PLACE, returns filtered obs."""
        return self._call(obs, obs if out is None else out, reward, _as_u8(done), terminal_obs, True)
