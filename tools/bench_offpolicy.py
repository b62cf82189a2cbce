"""Off-policy continuous control on one GPU: one JSON line per kind (td3, sac, ddpg) at the reference actor / critic
shapes (benchmark/torch/{td3,sac,ddpg}/mujoco_model.py, obs 17, action 6).

  explore_us_per_step[B]   rl_explore_mlp time per lock-step of B envs (CUDA events around launches of K steps,
                           after warm-up launches), and the achieved fp32 GFLOP/s on the actor's 2 * sum(in * out)
                           FLOPs per env-step
  update_ms_eager /       one DDPG / TD3 / SAC update on a batch of the reference size (sampler included): the
  update_ms_graph          class's eager learn() against the engine's replayed CUDA graphs
  engine_env_steps_per_s,  OffPolicyEngine.step() at the stated config (num_envs, steps_per_iter, updates_per_iter),
  engine_updates_per_s     host clock around iterations that end in a device synchronise
The GPU name and power limit are read in the same run.  The working set of the explore kernel (the actor, < 1 MB) is
L2-resident by design; the replay (1 M rows, 180 MB) is not.

    python tools/bench_offpolicy.py [--iters 200] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from parl_b200 import kernels as K                       # noqa: E402
from parl_b200.engine.offpolicy import OffPolicyEngine   # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or None
    except Exception:
        power = None
    return name, power


def actor_flops(model):
    layers, _, _ = model.native_actor_layers()
    return 2 * sum(w.shape[0] * w.shape[1] for segs in layers for w, _ in segs)


def time_explore(e, B, steps=32, reps=20):
    """us per lock-step of B envs (policy mode) on a fresh replay of the engine's kind."""
    from parl_b200.utils import ReplayMemory
    dev = e.device
    rm = ReplayMemory(steps * B, e.D, e.AD, device=dev)
    st = K.EpisodeStats(B, dev)
    obs = torch.zeros(B, e.D, device=dev)
    K.env_mujoco_synth_step(obs, None, None, st, 0, 0, reset=True)
    for _ in range(3):
        e.plan.explore(rm, e.mode, steps, obs, st, 0, 0, head=e.head)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for r in range(reps):
        e.plan.explore(rm, e.mode, steps, obs, st, 0, r * steps, head=e.head)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / (reps * steps)


def _timed(fn, n):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / n


def time_update(e, n=100):
    """(eager, graph) ms per update at the reference batch, sampler included: the class's own learn() on a freshly
    drawn device batch, against the engine's replayed graphs."""
    def eager():
        batch = K.replay_sample_uniform(e.rpm, e.batch_size, e.size_dev, e.draw_dev, e.seed, out=e._batch)
        e.draw_dev.add_(1)
        e.alg.learn(*batch)
    return _timed(eager, n), _timed(e.learn, n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--num-envs', type=int, default=256)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_offpolicy: no CUDA device (the measurement needs the GPU)')
    name, power = gpu_info()
    lines = []
    for kind in ('td3', 'sac', 'ddpg'):
        torch.manual_seed(0)
        e = OffPolicyEngine(kind, num_envs=args.num_envs, seed=0)
        flops = actor_flops(e.model)
        res = dict(kind=kind, gpu=name, power_limit=power, actor_mflop_per_env_step=flops / 1e6)
        for B in (256, 1024, 4096):
            us = time_explore(e, B)
            res['explore_us_per_step_B%d' % B] = round(us, 2)
            res['explore_gflops_B%d' % B] = round(flops * B / (us * 1e-6) / 1e9, 1)
        e.warmup()
        eager_ms, graph_ms = time_update(e)
        res['update_ms_eager'], res['update_ms_graph'] = round(eager_ms, 3), round(graph_ms, 3)
        for _ in range(10):
            e.step()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(args.iters):
            e.step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t
        res.update(engine_config=dict(num_envs=e.B, steps_per_iter=e.steps_per_iter, updates_per_iter=e.updates_per_iter,
                                      batch_size=e.batch_size, iters=args.iters),
                   engine_env_steps_per_s=round(args.iters * e.steps_per_iter * e.B / dt, 1),
                   engine_updates_per_s=round(args.iters * e.updates_per_iter / dt, 1))
        line = json.dumps(res)
        print(line, flush=True)
        lines.append(line)
        del e
    if args.out:
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
