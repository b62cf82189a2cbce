"""GPU: off-policy continuous control — rl_explore_mlp and rl_replay_sample_uniform against oracle/offpolicy.py, and
OffPolicyEngine (DDPG / TD3 / SAC with exploration, replay and updates on the device).

Exact where the arithmetic is exact: rewards, terminal flags, done counts, episode totals, warm-up actions and replay
rows are bit-exact against the oracle.  Observations come from the shared Box-Muller helper (libm log / cos on the
device), so they are bit-exact against the stand-alone env stepper rl_env_mujoco_synth_step and within the float
tolerance of tests/test_gpu_envs.py against numpy.  Policy actions are within 1e-5 of the float64 restatement."""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import offpolicy as ooff

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
D, AD = 17, 6


def _actor(kind, seed=0):
    from parl_b200.engine import nets
    from parl_b200 import kernels as K
    torch.manual_seed(seed)
    model = {'td3': nets.TD3MujocoModel, 'sac': nets.SACMujocoModel, 'ddpg': nets.DDPGMujocoModel}[kind](D, AD).to(DEV)
    layers, act, head = model.native_actor_layers()
    plan = K.MlpPlan(layers, act)
    params = [(torch.cat([w for w, _ in segs]).detach().double().cpu().numpy(),
               torch.cat([b for _, b in segs]).detach().double().cpu().numpy())
              for segs in layers]
    return model, plan, head, params


def _fresh(B, cap, seed, pos=0):
    from parl_b200 import kernels as K
    from parl_b200.utils import ReplayMemory
    rm = ReplayMemory(cap, D, AD, device=DEV)
    rm._curr_pos = pos
    st = K.EpisodeStats(B, DEV, ring_cap=0)
    obs = torch.zeros(B, D, device=DEV)
    K.env_mujoco_synth_step(obs, None, None, st, seed, 0, reset=True)
    return rm, st, obs


def _rows(rm, rows):
    r = torch.as_tensor(rows.reshape(-1), device=DEV)
    return (rm.obs[r].cpu().numpy(), rm.action[r].cpu().numpy(), rm.reward[r, 0].cpu().numpy(),
            rm.terminal[r, 0].cpu().numpy(), rm.next_obs[r].cpu().numpy())


def _check_explore(plan, head, params, B, K, mode):
    """One launch of K steps on a ring that wraps inside the launch, against the oracle."""
    seed, sigma, p_done, max_steps = 11, 0.1, 0.2, 4
    cap = K * B + 13                                    # not a multiple of B
    pos = cap - (K * B) // 2 - 1                        # the ring wraps inside the launch
    rm, st, obs = _fresh(B, cap, seed, pos)
    obs0 = obs.cpu().numpy()
    plan.explore(rm, mode, K, obs, st, seed, 0, head=head, expl_noise=sigma, p_done=p_done, max_episode_steps=max_steps)
    torch.cuda.synchronize()
    rows = np.stack([ooff.ring_rows(pos, t, B, cap) for t in range(K)])
    o, a, r, term, no = _rows(rm, rows)
    ref = ooff.explore(params, head, mode, K, B, AD, seed, 0, obs0, np.zeros(B), np.zeros(B, np.int32), cap, pos,
                       sigma=sigma, p_done=p_done, max_episode_steps=max_steps, obs_rows=o.reshape(K, B, D))
    assert np.array_equal(r, ref['reward'].reshape(-1))
    assert np.array_equal(term, ref['terminal'].reshape(-1))
    np.testing.assert_allclose(o, ref['obs'].reshape(-1, D), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(no, ref['next_obs'].reshape(-1, D), rtol=1e-4, atol=1e-5)
    assert np.array_equal(o.reshape(K, B, D)[1:], no.reshape(K, B, D)[:-1])      # next_obs(t) is obs(t+1)
    assert np.array_equal(obs.cpu().numpy(), no.reshape(K, B, D)[-1])
    if mode == 0:
        assert np.array_equal(a, ref['action'].reshape(-1, AD))
    else:
        np.testing.assert_allclose(a, ref['action'].reshape(-1, AD), rtol=0, atol=1e-5)
    assert np.array_equal(st.ep_ret.cpu().numpy(), ref['ep_ret'])
    assert np.array_equal(st.ep_len.cpu().numpy(), ref['ep_len'])
    tot = st.totals.cpu().numpy()
    comp = ref['completed']
    assert tot[0] == len(comp)
    assert tot[1] == sum(c[0] for c in comp) and tot[2] == sum(c[1] for c in comp)


@pytest.mark.parametrize('kind', ['td3', 'sac', 'ddpg'])
@pytest.mark.parametrize('B', [1, 63, 64, 1000])
@pytest.mark.parametrize('K', [1, 7])
@pytest.mark.parametrize('warm', [True, False])
def test_explore_matches_oracle(kind, B, K, warm):
    from parl_b200 import kernels as Kn
    mode = Kn.EXPLORE_WARMUP if warm else (Kn.EXPLORE_SAC if kind == 'sac' else Kn.EXPLORE_NOISE)
    _, plan, head, params = _actor(kind)
    _check_explore(plan, head, params, B, K, mode)


@pytest.mark.parametrize('hidden,B', [((256, 256), 2500),     # 79 tiles: 2-CTA clusters, several 4x4 blocks per thread
                                      ((256, 256), 4096),
                                      ((400, 300), 2500),     # DDPG shape: 8-CTA clusters, two waves
                                      ((64, ), 100),          # 1 hidden layer
                                      ((512, ), 40),          # the widest supported layer
                                      ((128, 96, 64), 300)])  # 3 hidden layers
def test_explore_layouts_match_oracle(hidden, B):
    """Cluster sizes, block loops and hidden-layer counts the reference actors at small B do not reach."""
    import torch.nn as nn
    from parl_b200 import kernels as Kn
    torch.manual_seed(5)
    dims = (D, ) + tuple(hidden) + (AD, )
    lins = [nn.Linear(dims[i], dims[i + 1]).to(DEV) for i in range(len(dims) - 1)]
    layers = [[(m.weight, m.bias)] for m in lins]
    plan = Kn.MlpPlan(layers, Kn.ACT_RELU)
    params = [(m.weight.detach().double().cpu().numpy(), m.bias.detach().double().cpu().numpy()) for m in lins]
    _check_explore(plan, Kn.HEAD_TANH, params, B, 2, Kn.EXPLORE_NOISE)


def test_observations_bit_exact_vs_env_stepper():
    from parl_b200 import kernels as Kn
    B, K, seed = 100, 6, 5
    _, plan, head, _ = _actor('td3')
    rm, st, obs = _fresh(B, K * B, seed)
    obs_ref = obs.clone()
    plan.explore(rm, Kn.EXPLORE_NOISE, K, obs, st, seed, 0, head=head, p_done=0.1, max_episode_steps=3)
    st2 = Kn.EpisodeStats(B, DEV, ring_cap=0)
    rew, done = torch.zeros(B, device=DEV), torch.zeros(B, dtype=torch.uint8, device=DEV)
    for t in range(K):
        assert torch.equal(rm.obs[t * B:(t + 1) * B], obs_ref)
        Kn.env_mujoco_synth_step(obs_ref, rew, done, st2, seed, t, p_done=0.1, max_episode_steps=3)
        assert torch.equal(rm.next_obs[t * B:(t + 1) * B], obs_ref)
        assert torch.equal(rm.reward[t * B:(t + 1) * B, 0], rew)
    assert torch.equal(obs, obs_ref)
    assert torch.equal(st.totals, st2.totals) and torch.equal(st.ep_len, st2.ep_len)


def test_k_steps_in_one_launch_equal_k_launches():
    from parl_b200 import kernels as Kn
    for kind in ('td3', 'sac', 'ddpg'):
        B, K, seed = 77, 5, 3
        mode = Kn.EXPLORE_SAC if kind == 'sac' else Kn.EXPLORE_NOISE
        _, plan, head, _ = _actor(kind)
        rm1, st1, obs1 = _fresh(B, K * B + 3, seed, pos=7)
        rm2, st2, obs2 = _fresh(B, K * B + 3, seed, pos=7)
        plan.explore(rm1, mode, K, obs1, st1, seed, 0, head=head, max_episode_steps=2)
        for t in range(K):
            plan.explore(rm2, mode, 1, obs2, st2, seed, t, head=head, max_episode_steps=2)
            rm2.commit(B)
        for f in ('obs', 'action', 'reward', 'terminal', 'next_obs'):
            assert torch.equal(getattr(rm1, f), getattr(rm2, f)), (kind, f)
        assert torch.equal(obs1, obs2)
        for f in ('ep_ret', 'ep_len', 'totals'):
            assert torch.equal(getattr(st1, f), getattr(st2, f)), (kind, f)


def test_time_limit_and_terminal():
    from parl_b200 import kernels as Kn
    B, K, seed = 40, 12, 9
    _, plan, head, _ = _actor('td3')
    rm, st, obs = _fresh(B, K * B, seed)
    plan.explore(rm, Kn.EXPLORE_NOISE, K, obs, st, seed, 0, head=head, p_done=0.0, max_episode_steps=5)
    assert int(rm.terminal.sum()) == 0                                  # only time limits end episodes
    assert st.totals[0].item() == 2 * B and st.totals[2].item() == 10 * B
    assert torch.equal(st.ep_len, torch.full((B, ), 2, dtype=torch.int32, device=DEV))
    rm, st, obs = _fresh(B, K * B, seed)
    plan.explore(rm, Kn.EXPLORE_NOISE, K, obs, st, seed, 0, head=head, p_done=1.0, max_episode_steps=5)
    assert bool((rm.terminal == 1).all()) and st.totals[0].item() == K * B     # every step ends a real episode
    rm, st, obs = _fresh(B, K * B, seed)
    plan.explore(rm, Kn.EXPLORE_NOISE, K, obs, st, seed, 0, head=head, p_done=1.0, max_episode_steps=1)
    assert int(rm.terminal.sum()) == 0                                  # ... except on the time-limit step


def test_wrappers_reject_malformed_input():
    from parl_b200 import kernels as Kn
    from parl_b200.engine import nets
    B = 8
    _, plan, head, _ = _actor('td3')
    rm, st, obs = _fresh(B, 64, 1)
    with pytest.raises(RuntimeError, match='replay capacity'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 9, obs, st, 1, 0, head=head)            # 9 * 8 > 64
    with pytest.raises(RuntimeError, match='obs_cur'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 1, obs.double(), st, 1, 0, head=head)
    with pytest.raises(RuntimeError, match='obs_cur'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 1, obs[:, :5].contiguous(), st, 1, 0, head=head)
    with pytest.raises(RuntimeError, match='CUDA'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 1, obs.cpu(), st, 1, 0, head=head)
    with pytest.raises(RuntimeError, match='contiguous'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 1, obs.t().contiguous().t(), st, 1, 0, head=head)
    with pytest.raises(RuntimeError, match='mode 1 needs the tanh head'):
        plan.explore(rm, Kn.EXPLORE_NOISE, 1, obs, st, 1, 0, head=Kn.HEAD_MEAN_LOGSTD)
    wide = nets._TanhActor(D, AD, 600, 64).to(DEV)
    wplan = Kn.MlpPlan([[(wide.l1.weight, wide.l1.bias)], [(wide.l2.weight, wide.l2.bias)],
                        [(wide.l3.weight, wide.l3.bias)]], Kn.ACT_RELU)
    with pytest.raises(RuntimeError, match='width 600'):
        wplan.explore(rm, Kn.EXPLORE_NOISE, 1, obs, st, 1, 0)
    size = torch.ones(1, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match='size_dev'):
        Kn.replay_sample_uniform(rm, 4, size.long(), size, 0)
    with pytest.raises(RuntimeError, match='draw_dev'):
        Kn.replay_sample_uniform(rm, 4, size, torch.ones(2, dtype=torch.int32, device=DEV), 0)
    with pytest.raises(RuntimeError, match='reward'):
        Kn.replay_sample_uniform(rm, 4, size, size, 0, out=(torch.empty(4, D, device=DEV),
                                                             torch.empty(4, AD, device=DEV),
                                                             torch.empty(5, device=DEV), torch.empty(4, D, device=DEV),
                                                             torch.empty(4, device=DEV)))


def test_replay_sampler_rows_and_gather():
    from parl_b200 import kernels as Kn
    B, K, seed, cap = 50, 8, 4, 1000
    _, plan, head, _ = _actor('sac')
    rm, st, obs = _fresh(B, cap, seed)
    plan.explore(rm, Kn.EXPLORE_SAC, K, obs, st, seed, 0, head=head)
    rm.commit(K * B)
    size = torch.tensor([rm.size()], dtype=torch.int32, device=DEV)
    for d in (0, 1, 12345):
        draw = torch.tensor([d], dtype=torch.int32, device=DEV)
        o, a, r, no, t, idx = Kn.replay_sample_uniform(rm, 333, size, draw, 77, want_idx=True)
        want = ooff.sample_rows(333, d, rm.size(), 77)
        assert np.array_equal(idx.cpu().numpy(), want)
        il = idx.long()
        assert torch.equal(o, rm.obs[il]) and torch.equal(a, rm.action[il]) and torch.equal(no, rm.next_obs[il])
        assert torch.equal(r, rm.reward[il, 0]) and torch.equal(t, rm.terminal[il, 0].float())


def test_replay_sampler_never_reads_past_the_ring():
    from parl_b200 import kernels as Kn
    B, cap = 32, 320
    _, plan, head, _ = _actor('td3')
    rm, st, obs = _fresh(B, cap, 6)
    plan.explore(rm, Kn.EXPLORE_WARMUP, cap // B, obs, st, 6, 0, head=head)
    rm.commit(cap)
    size = torch.tensor([cap + 100000], dtype=torch.int32, device=DEV)      # a size the ring does not have
    draw = torch.tensor([3], dtype=torch.int32, device=DEV)
    o, a, r, no, t, idx = Kn.replay_sample_uniform(rm, 1000, size, draw, 8, want_idx=True)
    assert np.array_equal(idx.cpu().numpy(), ooff.sample_rows(1000, 3, cap, 8))
    assert torch.equal(o, rm.obs[idx.long()])


def test_replay_sampler_in_captured_graph():
    from parl_b200 import kernels as Kn
    B, cap = 64, 4096
    _, plan, head, _ = _actor('td3')
    rm, st, obs = _fresh(B, cap, 2)
    plan.explore(rm, Kn.EXPLORE_WARMUP, cap // B, obs, st, 2, 0, head=head)
    rm.commit(cap)
    size = torch.tensor([100], dtype=torch.int32, device=DEV)
    draw = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = Kn.replay_sample_uniform(rm, 256, size, draw, 5, want_idx=True)     # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = Kn.replay_sample_uniform(rm, 256, size, draw, 5, want_idx=True)
        draw.add_(1)
    draw.zero_()
    seen = []
    for sz in (100, 100, 3000, 4096):
        size.fill_(sz)
        g.replay()
        torch.cuda.synchronize()
        idx = out[5].cpu().numpy()
        assert idx.min() >= 0 and idx.max() < sz
        assert np.array_equal(idx, ooff.sample_rows(256, len(seen), sz, 5))
        seen.append(idx)
    assert not np.array_equal(seen[0], seen[1])                            # fresh rows on every replay
    assert seen[3].max() >= 3000                                           # the row range follows the device size


def _engine(kind, seed=0, **kw):
    from parl_b200.engine.offpolicy import OffPolicyEngine
    args = dict(num_envs=64, memory_size=5000, warmup_size=1000, batch_size=64, seed=seed)
    args.update(kw)
    torch.manual_seed(seed)
    return OffPolicyEngine(kind, **args)


def test_engine_replay_accounting_and_save_load():
    e = _engine('td3', memory_size=1000, warmup_size=300, steps_per_iter=4)
    assert e.rpm.size() == 0
    e.warmup()                                    # ceil(300 / 64) = 5 lock-steps = 320 rows
    assert e.rpm.size() == 320 and e.rpm._curr_pos == 320 and e.env_steps == 5
    for _ in range(3):
        e.explore()                               # 3 x 256 rows: wraps at 1000
    assert e.rpm.size() == 1000 and e.rpm._curr_pos == (320 + 768) % 1000 and e.env_steps == 17
    assert int(e.size_dev.item()) == 1000
    e.learn()
    assert int(e.draw_dev.item()) == 1
    from parl_b200.utils import ReplayMemory
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, 'rpm.npz')
        e.rpm.save(p)
        rm2 = ReplayMemory(1000, D, AD, device=DEV)
        rm2.load(p)
    assert rm2.size() == e.rpm.size() and rm2._curr_pos == e.rpm._curr_pos
    for f in ('obs', 'action', 'reward', 'terminal', 'next_obs'):
        assert torch.equal(getattr(rm2, f), getattr(e.rpm, f)), f
    obs, act, rew, nobs, term = e.rpm.sample_batch(32)
    assert obs.shape == (32, D) and act.shape == (32, AD) and np.isfinite(act).all()


@pytest.mark.parametrize('kind', ['td3', 'sac', 'ddpg'])
def test_engine_same_seed_same_weights(kind):
    outs = []
    for _ in range(2):
        e = _engine(kind, seed=3)
        e.warmup()
        for _ in range(20):
            e.step()
        torch.cuda.synchronize()
        outs.append([p.detach().clone() for p in list(e.model.parameters()) + list(e.alg.target_model.parameters())])
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize('kind', ['td3', 'sac', 'ddpg'])
def test_engine_losses_finite_200_iterations(kind):
    e = _engine(kind, seed=1)
    e.warmup()
    before = [p.detach().clone() for p in e.model.get_actor_params()]
    for _ in range(200):
        out = e.step()
    torch.cuda.synchronize()
    critic_loss, actor_loss = out
    assert torch.isfinite(critic_loss).all()
    assert actor_loss is None or torch.isfinite(actor_loss).all()
    for p in e.model.parameters():
        assert torch.isfinite(p).all()
    assert any(not torch.equal(a, b) for a, b in zip(before, e.model.get_actor_params()))
    m = e.get_metrics()
    assert m['learn_steps'] == 200 and m['replay_size'] == min(5000, 1024 + 200 * 64)


@pytest.mark.parametrize('kind', ['td3', 'sac', 'ddpg'])
def test_graphed_update_equals_eager_class_update(kind):
    """The replayed CUDA graphs of the update are the class's eager update: same weights and target weights, bit for
    bit, on the same batches (TD3 without target-policy noise over policy_freq calls, SAC on a fixed epsilon)."""
    e = _engine(kind, seed=2, **({'policy_noise': 0.0} if kind == 'td3' else {}))
    if kind == 'sac':
        eps = torch.randn(e.batch_size, AD, device=DEV)
        e.alg.noise_fn = lambda mean: eps
    e.warmup()
    calls = e.alg.policy_freq if kind == 'td3' else 1
    for _ in range(3 * calls):                     # eager, capture + replay, replay for every part
        e.learn()
    assert set(e._graphs) == ({'critic', 'actor'} if kind == 'td3' else {'critic', 'actor', 'polyak'})
    alg = e.alg
    opts = (alg.actor_optimizer, alg.critic_optimizer)
    state = [t for o in opts for t in (o.flat, o.exp_avg, o.exp_avg_sq, o.step_dev)]
    state += [p.data for p in alg.target_model.parameters()]
    torch.cuda.synchronize()
    snap = [t.clone() for t in state]
    counts = [o.step_count for o in opts]
    total_it = getattr(alg, 'total_it', None)
    batches = []
    for _ in range(calls):
        e.learn()
        batches.append(tuple(b.clone() for b in e._batch))
    graphed = [p.detach().clone() for p in list(e.model.parameters()) + list(alg.target_model.parameters())]
    for t, v in zip(state, snap):
        t.copy_(v)
    for o, c in zip(opts, counts):
        o.step_count = c
    if total_it is not None:
        alg.total_it = total_it
    for b in batches:
        alg.learn(*b)
    torch.cuda.synchronize()
    eager = list(e.model.parameters()) + list(alg.target_model.parameters())
    assert len(graphed) == len(eager)
    for g, p in zip(graphed, eager):
        assert torch.equal(g, p)
