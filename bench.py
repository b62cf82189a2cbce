#!/usr/bin/env python
"""bench.py — IMPALA env-steps/s on synthetic Atari-shaped envs (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" = one full actor-learner iteration of the hot path: T=50 lock-step env steps of the whole
actor pool (policy forward + fused sample/env-step kernel per time step, trajectories written straight
into the (T,B) HBM rollout buffer) followed by one IMPALA learner update on the 50 x B batch (network
forward, fused V-trace+loss kernel, backward, gradient all-reduce over NCCL when N>1, clip + Adam).
Workload: configs[2] of BASELINE.json — 4096 actors in total, sharded B/N per GPU (strong scaling).
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'env_steps_per_sec_impala_4096_actors'
UNIT = 'env-steps/s'
TOTAL_ENVS = 4096
T_STEPS = 50
ACT_DIM = 18
K1_NCU_TRAFFIC_BYTES = 32.19e6        # dram read + write of one K1 (v8) launch at B=4096 (ncu --set full, profiles/r02_k1_v8_ncu.txt)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--envs', type=int, default=TOTAL_ENVS, help='total env instances over all GPUs')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--cpu-seconds', type=float, default=16.0, help='timed CPU-baseline sample of our arm')
    ap.add_argument('--ref-seconds', type=float, default=90.0, help='--impl reference: timed steady state in total')
    ap.add_argument('--ref-warmup-seconds', type=float, default=20.0)
    ap.add_argument('--ref-deepmind-seconds', type=float, default=20.0,
                    help='--impl reference: extra run of the full wrap_deepmind pipeline flavour (0 = skip)')
    ap.add_argument('--no-pipeline', action='store_true', help='strictly sequential rollout -> learn')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (rank 0) to DIR/<name>.npy, float32, at most 64 MB')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs dumps the timed path of --impl ours')
    return args


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.rows, self._stop, self._th = gpu_index, [], False, None

    def _run(self):
        while not self._stop:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop = True
        if self._th:
            self._th.join(timeout=6)
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace('.', '').isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.rows))


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU actor-learner path (examples/IMPALA/train.py + actor.py; oracle port —
    the Python reference itself cannot travel to the GPU box) on all host cores, learner on one B200 through torch
    eager as BASELINE.md section 3 asks.  ONE long-lived actor pool for the whole arm; a "step" is a wall-clock
    window over which sample_total_steps / elapsed is read exactly as the reference logs it (train.py:93,227,243).
    Under torchrun only rank 0 measures; the other ranks exit 0 without work."""
    if rank != 0:
        return
    from oracle.actor_learner import CpuImpalaCluster
    t_arm = time.time()
    total = args.ref_seconds                                   # timed steady state (>= 60 s by default)
    per = max(1.0, total / max(args.steps, 1))
    warm_per = max(per, args.ref_warmup_seconds / max(args.warmup, 1))
    cl = CpuImpalaCluster(flavour='lean', seed=0)
    try:
        for _ in range(max(args.warmup, 1)):
            cl.window(warm_per)
        wins = [cl.window(per) for _ in range(args.steps)]
        info = cl.info()
    finally:
        cl.close()
    steps_done = sum(w['sample_steps'] for w in wins)
    elapsed = sum(w['elapsed_s'] for w in wins)
    v = steps_done / elapsed
    ls = sum(w['learn_steps'] for w in wins)
    lms = (sum((w['learn_ms_per_batch'] or 0.0) * w['learn_steps'] for w in wins) / ls) if ls else None
    # Appendix-C flavour (i): mock Pong through the whole wrap_deepmind chain, a shorter second run
    dm = None
    if args.ref_deepmind_seconds > 0:
        cl2 = CpuImpalaCluster(flavour='deepmind', seed=1)
        try:
            cl2.window(min(20.0, max(8.0, args.ref_deepmind_seconds * 0.5)))
            w2 = cl2.window(args.ref_deepmind_seconds)
            dm = dict(value=w2['env_steps_per_s'], unit=UNIT, seconds=w2['elapsed_s'],
                      what='mock PongNoFrameskip-v4 (210x160x3) -> wrap_deepmind(dim=84) chain (SURVEY.md Appendix C '
                           'flavour i)', learner_ms_per_batch=w2['learn_ms_per_batch'])
        finally:
            cl2.close()
    sample = ('%d actor processes (1 core each) x %d envs x T=%d, lean 84x84 synthetic env + FrameStack4 (SURVEY.md '
              'Appendix C flavour ii, the most favourable for the CPU side), torch-CPU fp32 84x84 actor-critic per '
              'actor, pickle-over-pipe sample dicts, learner torch eager fp32 on %s (train batch %d); %d windows of '
              '%.1f s after %.0f s warm-up' % (info['actors'], info['env_num'], T_STEPS, info['learner_device'],
                                                info['train_batch_size'], args.steps, per,
                                                warm_per * max(args.warmup, 1)))
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=per * 1e3, higher_is_better=True, scaling='strong', vs_baseline=None, dtype='f32',
                data='synthetic', impl='reference',
                config=dict(workload='IMPALA synthetic Atari-shaped 84x84x4->18, CPU actor pool (oracle port of '
                                     'examples/IMPALA on the host cores; one host cannot hold 4096 xparl jobs, so '
                                     'actors = cores - 2, reported as is)',
                            total_envs=info['actors'] * info['env_num'], T=T_STEPS,
                            train_batch_size=info['train_batch_size'], host_cores=info['cores'],
                            learner_device=info['learner_device']),
                cpu_baseline=dict(value=v, unit=UNIT, cores=info['cores'], kind='port', sample=sample,
                                  learner_ms_per_batch=lms, learner_device=info['learner_device'],
                                  deepmind_pipeline=dm),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                arm_wall_s=time.time() - t_arm)
    print(json.dumps(line))
    sys.stdout.flush()


def cpu_baseline_subprocess(args):
    """cpu_baseline leg of our arm: the reference arm as a child process (its actor pool must be forked from a
    process that has not initialised CUDA), bounded to about half a minute."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '4', '--warmup', '2',
           '--ref-seconds', str(args.cpu_seconds), '--ref-warmup-seconds', '8', '--ref-deepmind-seconds', '0']
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=args.cpu_seconds + 120, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith('{'):
                return json.loads(ln)['cpu_baseline']
        sys.stderr.write('cpu_baseline: no line from the child (rc %d)\n%s\n' % (r.returncode, r.stderr[-2000:]))
    except Exception as e:
        sys.stderr.write('cpu_baseline failed: %r\n' % (e, ))
    return None


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    assert args.warmup >= 3, 'timing rules: at least 3 warm-up steps'
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    assert args.envs % world == 0
    B = args.envs // world

    from parl_b200 import kernels
    from parl_b200.engine.impala import ImpalaEngine
    torch.manual_seed(0)                      # identical initial weights on every rank
    eng = ImpalaEngine(num_envs=B, sample_batch_steps=T_STEPS, act_dim=ACT_DIM, seed=1234, device=dev,
                       env_offset=rank * B, pipeline=not args.no_pipeline)
    if world > 1:
        # IMPALA's loss is a SUM over the global batch (impala.py:67-79) -> all-reduce SUM of the flat gradient
        eng.alg.grad_sync = lambda g: dist.all_reduce(g, op=dist.ReduceOp.SUM)

    def step():
        return eng.step(0.001, -0.01)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    kernels.reset_launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        losses = step()
    ev1.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        # before the untimed K1 steps below overwrite the engine's buffers and weights
        dump_outputs(eng, losses, args.dump_outputs)
    if world > 1:
        dist.barrier()
    elapsed_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    elapsed = elapsed_ms.item() * 1e-3
    launches = kernels.launch_count()
    # K1 bracketed by events INSIDE a step: three extra, untimed steps (no event records inside the timed region)
    k1_events = []
    eng.k1_events = k1_events
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    eng.k1_events = None
    total_steps = args.steps * T_STEPS * args.envs
    value = total_steps / elapsed

    # roofline of the HBM-bound kernel the north star names (K1).  Inside a pipelined step its event-bracketed
    # duration includes time-sharing with the actor stream's kernels, so the launch duration used for the roofline is
    # measured right here, live, on the step's own rollout buffers with nothing else in flight (CUDA events on the
    # launching stream); the overlapped in-step figure is reported next to it.
    k1_ms = [a.elapsed_time(b) for a, b in k1_events]
    k1_in_step_us = (sum(k1_ms) / len(k1_ms)) * 1e3 if k1_ms else None
    torch.cuda.synchronize()
    if eng.train_net is not None:
        lg, vl = eng.train_net.logits, eng.train_net.values.view(-1)
    else:
        lg, vl = eng.tgt_logits.view(T_STEPS * B, ACT_DIM), eng.values.view(-1)
    k1_args = (eng.actions.view(-1), eng.rewards.view(-1), eng.dones.view(-1), vl, T_STEPS, B, 0.99, 0.5, -0.01)
    # (a) one event pair per launch, L2 flushed before every launch (a 256 MB fill > the 126 MB L2)
    iso = []
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for i in range(12):
        flush.fill_(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        kernels.vtrace_loss_fwd_bwd(lg, eng.beh_logits.view(T_STEPS * B, ACT_DIM), *k1_args, out=eng.loss_out)
        b.record()
        iso.append((a, b))
    torch.cuda.synchronize()
    iso_ms = sorted(x.elapsed_time(y) for x, y in iso[2:])
    k1_flushed_s = (sum(iso_ms) / len(iso_ms)) * 1e-3
    del flush
    # (b) the launch duration the roofline uses: 64 back-to-back launches over rotating copies of the logits
    # (inputs + outputs of consecutive launches never overlap; the rotation spans > 3x the L2), ONE event pair,
    # so neither the event record latency nor an L2-resident operand is in the figure
    nrot = max(4, int(3 * 126e6 / max(1, (T_STEPS * B * ACT_DIM * 4 * 3))) + 1)
    rot = [(lg.clone(), eng.beh_logits.view(T_STEPS * B, ACT_DIM).clone(),
            dict(losses=torch.zeros(8, device=dev), d_logits=torch.empty((T_STEPS * B, ACT_DIM), device=dev),
                 d_values=torch.empty(T_STEPS * B, device=dev))) for _ in range(nrot)]
    for i in range(nrot):
        kernels.vtrace_loss_fwd_bwd(rot[i][0], rot[i][1], *k1_args, out=rot[i][2])
    torch.cuda.synchronize()
    nl = 64

    def k1_loop():
        for i in range(nl):
            r = rot[i % nrot]
            kernels.vtrace_loss_fwd_bwd(r[0], r[1], *k1_args, out=r[2])

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k1_timing = 'cuda graph of %d launches' % nl
    try:
        # the 64 launches as ONE CUDA graph: a K1 call costs ~10 us of Python + ctypes on the host, more than the
        # kernel itself, so an eager loop would time the host's launch rate instead of the GPU
        k1_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(k1_graph):
            k1_loop()
        k1_graph.replay()
        torch.cuda.synchronize()
        reps = []
        for _ in range(5):
            a.record()
            k1_graph.replay()
            b.record()
            torch.cuda.synchronize()
            reps.append(a.elapsed_time(b) * 1e-3 / nl)
        k1_s = sorted(reps)[len(reps) // 2]
        del k1_graph
    except Exception as exc:                              # noqa: BLE001 - fall back to the eager loop
        sys.stderr.write('bench: K1 graph timing failed (%r); eager loop\n' % (exc, ))
        torch.cuda.synchronize()
        k1_timing = 'eager loop of %d launches' % nl
        a.record()
        k1_loop()
        b.record()
        torch.cuda.synchronize()
        k1_s = a.elapsed_time(b) * 1e-3 / nl
    del rot
    alg_bytes = (T_STEPS - 1) * B * (12 * ACT_DIM + 17) + 4 * B
    peak, peak_src = measured_peaks()
    roof = None
    if k1_s:
        ach = alg_bytes / k1_s / 1e9
        # traffic: dram__bytes_read.sum + dram__bytes_write.sum of one launch at B=4096 from the committed
        # `ncu --set full` capture of this kernel version (profiles/r02_k1_v8_ncu.txt); the gradient tile (15.3 MB) is
        # mostly still in the 126 MB L2 when the launch ends, so the write half shows up only partly
        traffic = K1_NCU_TRAFFIC_BYTES if B == 4096 else None
        roof = dict(bound='hbm', kernel='vtrace_loss_v8_kernel (rl_vtrace_loss_fwd_bwd)', achieved=ach, peak=peak,
                    unit='GB/s', frac=ach / peak, traffic=traffic, peak_source=peak_src,
                    algorithmic_bytes_per_launch=alg_bytes, us_per_launch=k1_s * 1e6,
                    us_per_launch_l2_flushed_single_event_pair=k1_flushed_s * 1e6,
                    frac_l2_flushed_single_event_pair=alg_bytes / k1_flushed_s / 1e9 / peak,
                    us_per_launch_in_pipelined_step=k1_in_step_us,
                    l2='%d rotating operand sets (> 3x L2), %s, one event pair per replay, median of 5' % (nrot, k1_timing))

    # the kernel with the largest share of the step (profiles/r01_bench_launches_final.txt: 15 %): conv1 forward in
    # TMA-window form, timed here live at the learner's batch on the step's own buffers (11.6 GB in, 7.5 GB out: far
    # beyond L2, nothing to flush), CUDA events on the launching stream, nothing else in flight
    dom = None
    try:
        dom = measure_dominant_kernel(eng, kernels, torch, B, peak, peak_src)
    except Exception as e:                       # never lose the bench line over the extra measurement
        sys.stderr.write('dominant-kernel roofline skipped: %r\n' % (e, ))

    # tensor-pipe view of the whole step: policy/value network FLOPs (actor forward + learner forward/backward
    # = 4 x 25.8 MFLOP per env-step, SURVEY.md 8d) over the step time, against the measured sustained bf16 peak
    net_roof = None
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        tpeak, tsrc = float(pk['bf16_tflops_sustained']), 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)'
    except Exception:
        tpeak, tsrc = 1400.0, 'fallback (B200_PROFILING.md sustained)'
    flops_per_step = 4 * 25.8e6 * T_STEPS * B
    ach_tf = flops_per_step * args.steps / elapsed / 1e12
    net_roof = dict(bound='tensor', what='policy/value network (tcgen05 conv/GEMM kernels), per GPU', achieved=ach_tf,
                    peak=tpeak, unit='TFLOP/s', frac=ach_tf / tpeak, peak_source=tsrc)

    # HBM view of the whole step: with the convolutions at 2x2/3x3 filters on 32..128 channels the network kernels are
    # bound by ACTIVATION traffic, not by the tensor pipe.  Algorithmic bytes per env-step of the dataflow as designed
    # (bf16 activations, every tensor read/written once per kernel that needs it; DESIGN.md section 4 table):
    #   rollout 264 KB (gather 84.7, conv1 82.0, conv2 52.4, conv3 25.9, fc+heads 12.4, env frame 7.1)
    #   learner 538 KB (forward 172.7, mask/scatter + fc products 61.1, dgrad 132.9, wgrad 170.9)
    # with the observation plane kept uint8 (the default) the gather writes, and conv1 forward (actor + learner) and
    # conv1's weight gradient read, 28.2 KB less each: 208 KB + 481 KB
    u8_obs = eng.obs_step.dtype == torch.uint8
    per_env_step = (264.5e3 + 537.6e3) - (4 * 28224 if u8_obs else 0)
    step_bytes = per_env_step * T_STEPS * B
    ach_hbm = step_bytes * args.steps / elapsed / 1e9
    step_roof = dict(bound='hbm', what='whole step: activation traffic of the network kernels, per GPU',
                     achieved=ach_hbm, peak=peak, unit='GB/s', frac=ach_hbm / peak, peak_source=peak_src,
                     algorithmic_bytes_per_env_step=per_env_step) if eng.train_net is not None else None

    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(eng, args, world, dev)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess(args)
    if rank == 0:
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=elapsed * 1e3 / args.steps, higher_is_better=True, scaling='strong', vs_baseline=None,
                    dtype='bf16 network (fp32 accumulate, fp32 master weights) / f32 scans+losses', data='synthetic',
                    config=dict(workload='IMPALA synthetic Atari-shaped (84x84x4 -> 18 discrete), %d actors total, '
                                         'T=50, V-trace; configs[2] of BASELINE.json' % args.envs,
                                envs_per_gpu=B, T=T_STEPS, learner_batch=T_STEPS * args.envs,
                                model='84x84 actor-critic (benchmark/torch/a2c/atari_model.py), 2.74 M params',
                                parallelism='dp%d' % world,
                                actor_learner='pipelined (rollout k+1 || learn k, policy lag 1)' if eng.pipeline
                                else 'sequential',
                                network='hand-written tcgen05 kernels (actor fwd; learner fwd+dgrad+wgrad)' if
                                eng.train_net is not None else 'torch',
                                l2_policy='per-step working set (frame ring %.1f GB + observation plane %.1f GB + '
                                          'activations %.1f GB per GPU) >> 126 MB L2; K1 timed alone with L2 flushed' %
                                          ((T_STEPS + 4) * B * 7056 / 1e9, T_STEPS * B * 28224 * eng.obs_step.element_size() / 1e9,
                                           T_STEPS * B * 120e3 / 1e9)),
                    gpu_launches=launches, clocks=clocks, roofline=dom if dom is not None else roof, roofline_k1=roof,
                    roofline_network=net_roof, roofline_step=step_roof,
                    e2e=e2e,
                    cpu_baseline=cpu,
                    learner_losses=[float(x) for x in losses[:5].tolist()])
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_ENV_COLUMNS = 2048                   # env columns kept of each (T, B, ...) buffer: 36 MB in all at 4096 envs
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(eng, losses, out_dir):
    """What the last timed step computed, as float32 .npy files: the losses step() returned, the weights after its
    update, the rollout the update trained on with the learner's logits and values for it, and (pipelined engines)
    the rollout produced alongside it.  The (T, B, ...) buffers keep a fixed, seeded sample of env columns, so
    that two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    B = eng.B
    cols = torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_ENV_COLUMNS), replace=False)))

    def sample(t):
        return t[:, cols.to(t.device)].float().cpu().numpy()

    def rollout(st, prefix):
        return {prefix + 'actions': sample(st['actions']), prefix + 'behaviour_logits': sample(st['beh_logits']),
                prefix + 'rewards': sample(st['rewards']), prefix + 'dones': sample(st['dones'])}

    out = dict(losses=losses.float().cpu().numpy(),
               params=torch.cat([p.detach().reshape(-1) for p in eng.model.parameters()]).float().cpu().numpy(),
               learner_logits=sample(eng.tgt_logits), learner_values=sample(eng.values))
    out.update(rollout(eng._sets[eng._cur_set], ''))
    if eng.pipeline:
        out.update(rollout(eng._sets[1 - eng._cur_set], 'next_'))
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, 'dump of %d bytes exceeds %d' % (total, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


# dram__bytes_read.sum + dram__bytes_write.sum per sample of conv1 forward from the committed ncu captures:
# bf16 input (profiles/r01_learner_kernels_final.txt: 2.948 GB + 1.282 GB at 51 200 samples); uint8 input
# (profiles/r02_conv1_u8_ncu.txt: 1.445 GB + 1.270 GB)
CONV1_NCU_TRAFFIC_PER_SAMPLE = {False: (2.947656e9 + 1.281806e9) / 51200.0, True: (1.445169e9 + 1.269890e9) / 51200.0}


def measure_dominant_kernel(eng, kernels, torch, B, peak, peak_src):
    """Roofline entry of the step's dominant kernel, shiftconv_fwd_kernel<32,1,2,0> (conv1 forward): algorithmic bytes
    per launch = samples x (4*84*84 B of uint8 observation read + 20*20*32*2 B of outputs written)."""
    net = eng.train_net
    if net is None:
        return None
    n = T_STEPS * B
    x0 = eng.x0.view(n, 21, 21, 64) if eng.share_obs else net.x0
    spans = []
    for _ in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        kernels.conv2d_s1_nhwc_bf16_fwd(x0, net.w1, net.b1, 2, 2, relu=True, out=net.a1, out_mode=1)
        b.record()
        spans.append((a, b))
    torch.cuda.synchronize()
    ms = sorted(x.elapsed_time(y) for x, y in spans[1:])
    sec = sum(ms) / len(ms) * 1e-3
    # algorithmic bytes per sample as SURVEY.md 8(d) counts them: the stacked uint8 observation (4 x 84 x 84 = 28 224 B)
    # read + the bf16 feature map written (20 x 20 x 32 x 2 = 25 600 B).  As built the kernel reads the uint8
    # space-to-depth plane (21 x 21 x 64 = 28 224 B per sample, widened to bf16 in shared memory) and writes conv2's
    # zero-padded 2x2-block input (12 x 12 x 128 x 2 = 36 864 B, of which 25 600 B are written, the border stays zero).
    u8 = x0.dtype == torch.uint8
    in_bytes = 21 * 21 * 64 * (1 if u8 else 2)
    alg_bytes = n * (4 * 84 * 84 + 20 * 20 * 32 * 2)
    ach = alg_bytes / sec / 1e9
    # traffic: dram__bytes_read.sum + dram__bytes_write.sum of this kernel in the committed `ncu --set full` capture
    # (CONV1_NCU_TRAFFIC: bytes per sample), scaled to this launch's samples
    traffic = CONV1_NCU_TRAFFIC_PER_SAMPLE[u8] * n if CONV1_NCU_TRAFFIC_PER_SAMPLE[u8] else None
    name = 'shiftconv_fwd_kernel<32,1,2,0,%s> (%s, conv1 forward at the learner batch)' % (
        'true' if u8 else 'false', 'rl_conv2d_s1_u8in_bf16_fwd' if u8 else 'rl_conv2d_s1_nhwc_bf16_fwd')
    return dict(bound='hbm', kernel=name,
                achieved=ach, peak=peak, unit='GB/s', frac=ach / peak, traffic=traffic, peak_source=peak_src,
                algorithmic_bytes_per_launch=alg_bytes, us_per_launch=sec * 1e6, samples_per_launch=n,
                bytes_moved_per_launch_as_built=n * (in_bytes + 20 * 20 * 32 * 2),
                frac_of_peak_as_built=n * (in_bytes + 20 * 20 * 32 * 2) / sec / 1e9 / peak,
                l2='operands (%.1f GB + 7.5 GB at 204 800 samples) far beyond the 126 MB L2' % (204800 * in_bytes / 1e9))


def numa_pin(gpu_index):
    """Bind this process to the CPUs nearest to its GPU before the pinned staging buffers are allocated
    (first-touch places them on the local NUMA node).  Best effort: returns a description or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return 'cpus %d' % len(os.sched_getaffinity(0))
    except Exception as e:
        return 'unpinned (%s)' % type(e).__name__


def copy_bandwidth(torch, dev, nbytes=1 << 30):
    """Measured pinned H2D / D2H copy bandwidth (GB/s) — the ceiling of the host-contract path."""
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {}
    for name, (dst, src) in (('h2d', (d, h)), ('d2h', (h, d))):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            dst.copy_(src, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        out[name] = 3 * nbytes / (a.elapsed_time(b) * 1e-3) / 1e9
    return out


def copy_bandwidth_bidir(torch, dev, nbytes=1 << 30):
    """Pinned H2D and D2H copies running AT THE SAME TIME on two streams (what the host-contract path does: the actor
    downloads sample k+1 while the learner uploads sample k), GB/s per direction.  Called by every rank at once, so
    that GPUs behind a shared PCIe switch / one host memory system see each other's traffic."""
    h_up = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h_dn = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d_up = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_dn = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_up.copy_(h_up, non_blocking=True)
    h_dn.copy_(d_dn, non_blocking=True)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    reps = 3
    with torch.cuda.stream(s_up):
        ev[0].record()
        for _ in range(reps):
            d_up.copy_(h_up, non_blocking=True)
        ev[1].record()
    with torch.cuda.stream(s_dn):
        ev[2].record()
        for _ in range(reps):
            h_dn.copy_(d_dn, non_blocking=True)
        ev[3].record()
    torch.cuda.synchronize()
    return dict(h2d=reps * nbytes / (ev[0].elapsed_time(ev[1]) * 1e-3) / 1e9,
                d2h=reps * nbytes / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e9)


def run_e2e(eng, args, world, dev):
    """The same metric END TO END through the reference-facing surface with HOST buffers, exactly the Learner loop of
    examples/IMPALA/train.py:165-194: a ``@parl.remote_class(wait=False)`` Actor (the device actor pool) whose
    ``sample()`` returns the numpy sample dict (uint8 stacked obs, env-major; D2H into pinned memory inside the
    timed region), ``actor.set_weights(agent.get_weights())`` with numpy weight dicts, and ``agent.learn(numpy...)``
    (H2D inside the timed region).  The next sample is produced while the learner trains on the current one, as
    the reference's sampling threads do."""
    import torch
    import torch.distributed as dist
    import parl_b200 as parl
    from parl_b200.engine.impala_host import DeviceImpalaActor, AtariAgent
    rank = int(os.environ.get('RANK', 0))
    B = args.envs // world
    pin = numa_pin(dev.index)
    parl.connect('localhost:8010')
    Actor = parl.remote_class(wait=False)(DeviceImpalaActor)
    cfg = dict(env_num=B, sample_batch_steps=T_STEPS, act_dim=ACT_DIM, seed=1234, env_offset=rank * B)
    torch.manual_seed(0)
    agent = AtariAgent(cfg, device=dev)
    if world > 1:
        agent.alg.grad_sync = lambda g: dist.all_reduce(g, op=dist.ReduceOp.SUM)
    actor = Actor(cfg, device=dev)
    steps = args.steps
    actor.set_weights(agent.get_weights()).get()
    fut = actor.sample()

    phase = dict(wait_sample=0.0, set_weights=0.0, learn=0.0)     # host wall-clock per phase (timed steps only)

    def one_step(fut):
        t0 = time.time()
        batch = fut.get()
        t1 = time.time()
        actor.set_weights(agent.get_weights())            # queued on the actor's worker: applies before its next sample
        nxt = actor.sample()
        t2 = time.time()
        losses = agent.learn(batch['obs'], batch['actions'], batch['behaviour_logits'], batch['rewards'],
                             batch['dones'], 0.001, -0.01)  # returns Python floats: a D2H read of the step's result
        t3 = time.time()
        phase['wait_sample'] += t1 - t0
        phase['set_weights'] += t2 - t1
        phase['learn'] += t3 - t2
        return nxt, losses, batch

    for _ in range(3):                                    # warm-up (graph capture, allocator, both host buffer sets)
        fut, losses, batch = one_step(fut)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    for k in phase:
        phase[k] = 0.0
    t0 = time.time()
    for _ in range(steps):
        fut, losses, batch = one_step(fut)
    torch.cuda.synchronize()
    el = torch.tensor([time.time() - t0], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    fut.get()
    last_sample_ms = float(actor.last_sample_s) * 1e3     # host wall clock of the actor's last sample() call
    nbytes = sum(v.nbytes for v in batch.values())
    wbytes = sum(v.nbytes for v in agent.get_weights().values())
    bw = copy_bandwidth(torch, dev) if rank == 0 else None
    actor.destroy()
    value = steps * T_STEPS * args.envs / el.item()
    ceiling = ceiling_bidir = bidir = None
    if bw:
        # one direction at a time, this GPU alone: the slower one bounds a step if the link were full duplex at that rate
        ceiling = T_STEPS * B * world / (nbytes / (min(bw['h2d'], bw['d2h']) * 1e9))
    # what the path actually sees: both directions at once, on every rank at the same time.  Every rank takes part in
    # the collectives whatever happens to its own measurement (zeros mark a failed one).
    if world > 1:
        dist.barrier()
    try:
        b2 = copy_bandwidth_bidir(torch, dev)
    except Exception as exc:                              # noqa: BLE001 - the ceiling is a report, not the metric
        sys.stderr.write('bench: bidirectional copy bandwidth not measured (%r)\n' % (exc, ))
        b2 = dict(h2d=0.0, d2h=0.0)
    t = torch.tensor([b2['h2d'], b2['d2h'], 1.0 if b2['h2d'] > 0 else 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    agg = t.tolist()
    if agg[2] == world:
        bidir = dict(h2d_per_gpu=agg[0] / world, d2h_per_gpu=agg[1] / world, h2d_all_gpus=agg[0], d2h_all_gpus=agg[1])
        ceiling_bidir = T_STEPS * B * world / (nbytes / (min(agg[:2]) / world * 1e9))
    return dict(value=value, unit=UNIT, h2d_bytes_per_step=nbytes + wbytes, d2h_bytes_per_step=nbytes + wbytes + 40,
                steps=steps, ms_per_step=el.item() * 1e3 / steps,
                path='@parl.remote_class(wait=False) Actor.sample() -> numpy dict (uint8 stacked obs, env-major, pinned) '
                     '-> AtariAgent.learn(numpy) ; actor.set_weights(agent.get_weights()) numpy weight dicts '
                     '(examples/IMPALA/train.py:165-194)',
                host_buffers=pin, copy_bandwidth_gbs=bw, pcie_ceiling_env_steps_per_s=ceiling,
                copy_bandwidth_bidirectional_all_ranks_gbs=bidir, pcie_ceiling_bidirectional_env_steps_per_s=ceiling_bidir,
                learner_thread_ms_per_step={k: v * 1e3 / steps for k, v in phase.items()},
                actor_groups=int(os.environ.get('PARL_B200_ACTOR_GROUPS', 0)) or 'auto', actor_last_sample_ms=last_sample_ms,
                sample_dict_bytes=nbytes, last_losses=[float(x) for x in losses])


if __name__ == '__main__':
    main()
