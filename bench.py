"""Benchmark of the hot path (BASELINE.json metric: env-steps/sec, update ms, % roofline).

    python bench.py --gpus 1 --steps 5 --warmup 3            # PPO, BASELINE configs[1] (default)
    python bench.py --workload sac --steps 20 --warmup 5      # BASELINE configs[2]
    python bench.py --workload td3 | ddpg                     # BASELINE configs[3] (per-GPU shard)
    python bench.py --impl reference --steps 2 --warmup 1     # reference arm (CPU oracle port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # weak scaling

PPO (default): one "step" = one PPO iteration of BASELINE.json configs[1]: a rollout of
T=128 vector steps of N=4096 synthetic HalfCheetah-shape envs per GPU (obs 17, act 6) followed
by the full update (value evaluation, lambda-returns, advantage normalisation, E=10 epochs x
32 minibatches of 16384 of clipped-ratio actor + value-regression critic updates with Adam,
2x256 tanh MLPs).  Nothing is skipped in the timed region.

Off-policy workloads: one "step" = one vector step of the collector with a FULL device replay
(obs / act shapes and env counts of BASELINE configs[2] / [3]) followed by the reference's
update cadence: `steps_between_batches = 50` <= N, so every vector step runs one update of 50
iterations x batch 100 (replays/buffers.py:8-12; `--offpolicy-batch B` scales the batch).

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  update_ms    CUDA-event time of one update (ppo.py:20-59 / ddpg.py:86-103) inside the timed run
  roofline     dominant GEMM entry point: achieved TFLOP/s from CUDA-event timing of every
               launch (an instrumented pass of the same steps) against MEASURED_PEAKS.json;
               `hbm_kernels`: achieved GB/s and fraction of the measured HBM peak for the
               memory-bound kernels (env step, lambda-returns, advantages, Adam, moments,
               policy loss, permutation; off-policy: Q target, soft update)
  cpu_baseline the oracle port (CPU restatement of the reference, pinned to the reference's
               golden vectors) timed on this box's host cores
  e2e          same metric through the reference-facing protocol with HOST numpy arrays
               crossing the boundary every vector step
  multi_rank_parity  (N > 1) the teacher-forced golden scenarios reproduced by the N ranks
               before timing ("ok" / error text)

`--dump-outputs DIR` writes what the timed path computed in its last step as DIR/<name>.npy
(rank 0), so that two builds run with the same arguments (same seeded inputs) can be compared
output for output.

The benchmark runs the library that `__graft_entry__.build()` left in the tree; it compiles
nothing and writes nothing there.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the tree may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OBS, ACT, ENVS_PER_GPU, SEGMENT, EPOCHS, MINIBATCHES, HIDDEN = 17, 6, 4096, 128, 10, 32, 256
MAX_EPISODE_STEPS = 1000
# BASELINE.json configs[2] / configs[3]: (agent, env preset, obs, act, envs per GPU)
OFF_POLICY = {'sac': ('SAC', 'Humanoid', 376, 17, 2048),
              'td3': ('TD3', 'Ant', 111, 8, 1024),
              'ddpg': ('DDPG', 'Ant', 111, 8, 1024)}
REPLAY_SIZE = int(1e6)


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=p.get('bf16_tflops_sustained', 1441.0), hbm=p.get('hbm_gbs', 6574.1),
                    source='MEASURED_PEAKS.json (sustained bf16 / copy bandwidth)')
    return dict(tflops=1400.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


def ncu_traffic():
    """dram read+write bytes per launch of the 16384-row critic minibatch kernels, from the
    committed warm-cache `ncu` capture (profiles/r2_chain_traffic.json, written by
    scratch/summarize_ncu.py); None when no capture of this round is committed."""
    path = os.path.join(ROOT, 'profiles', 'r2_chain_traffic.json')
    if os.path.exists(path):
        return json.load(open(path))
    return {}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""

    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(
                    ['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                     '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([c.strip() for c in out.strip().split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import numpy as np
        good = [s for s in self.samples if len(s) == 6 and s[0].isdigit()]
        if not good:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == 'Active' for s in good)]
        return dict(sm_mhz=float(np.median([int(s[0]) for s in good])),
                    sm_max_mhz=float(good[0][1]), reasons=reasons, samples=len(good))


# ------------------------------------------------------------------- shared plumbing
class Run:
    """Process-group, barrier and timing helpers of one bench process (one rank)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', 1))
        self.rank = int(os.environ.get('RANK', 0))
        self.local_rank = int(os.environ.get('LOCAL_RANK', 0))
        assert self.world == args.gpus, \
            f'launch with torchrun for --gpus {args.gpus} (WORLD_SIZE={self.world})'
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group('nccl', device_id=torch.device('cuda', self.local_rank))
        from tonic_b200 import _lib
        _lib.load()         # raises when the library has not been built

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, value):
        t = self.torch.tensor([value], device='cuda', dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps):
        """K calls of fn bracketed by barrier + synchronize, CUDA events, max over ranks."""
        torch = self.torch
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        # `ncu --profile-from-start off` captures exactly the timed region (launch list of the SAME
        # command under profiles/; a number printed by such a run is never a bench value)
        profiled = os.environ.get('TB_BENCH_CUDA_PROFILER') == '1'
        if profiled:
            torch.cuda.profiler.start()
        start.record()
        for _ in range(steps):
            fn()
        end.record()
        self.barrier()
        if profiled:
            torch.cuda.profiler.stop()
        return self.max_over_ranks(start.elapsed_time(end))


class UpdateTimer:
    """CUDA events around agent._update (no synchronisation: read after the run)."""

    def __init__(self, agent):
        import torch
        self.events = []
        inner = agent._update

        def timed(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = inner(*a, **k)
            e.record()
            self.events.append((s, e))
            return out
        agent._update = timed

    def reset(self):
        self.events.clear()

    def mean_ms(self):
        if not self.events:
            return None
        return sum(s.elapsed_time(e) for s, e in self.events) / len(self.events)


def hbm_table(prof, bytes_per_launch, hbm_peak):
    """entry point -> achieved GB/s of the memory-bound kernels (algorithmic bytes per launch
    / CUDA-event time per launch) and the fraction of the measured HBM peak."""
    out = {}
    for name, nbytes in bytes_per_launch.items():
        if name in prof and prof[name][0] > 0 and prof[name][1] > 0:
            count, ms = prof[name]
            us = ms / count * 1e3
            gbs = nbytes / (us * 1e-6) / 1e9
            out[name] = dict(launches=count, avg_launch_us=round(us, 2), bytes_per_launch=int(nbytes),
                             achieved_gbs=round(gbs, 1), frac=round(gbs / hbm_peak, 4))
    return out


DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much
DUMP_ENVS = 1024            # environment columns of the PPO segment in the dump (fixed seeded sample)


def dump_outputs(out_dir, tensors):
    """Writes every tensor as out_dir/<name>.npy: float64 stays float64, everything else becomes
    float32."""
    import numpy as np
    arrays = {}
    for name, t in tensors.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES, f'--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte limit'
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def model_outputs(agent, stats):
    """What an update hands back: the model's state_dict (the reference's key names, as in a
    checkpoint) and the per-minibatch statistics block the logger reads."""
    out = {'model.' + k: v for k, v in agent.model.state_dict().items()}
    out['update_stats'] = stats
    return out


# ----------------------------------------------------------------------------- PPO
def build_ppo(envs_local, total_envs, seed=0):
    import torch
    import tonic_b200
    import tonic_b200.torch
    m, n = tonic_b200.torch.models, tonic_b200.torch.normalizers
    spec = tonic_b200.environments.SynthControl('HalfCheetah', max_episode_steps=MAX_EPISODE_STEPS)
    env = tonic_b200.environments.distribute(lambda: spec, 1, total_envs)
    assert env.workers == envs_local
    env.initialize(seed=seed)
    model = m.ActorCritic(
        actor=m.Actor(encoder=m.ObservationEncoder(), torso=m.MLP((HIDDEN, HIDDEN), torch.nn.Tanh),
                      head=m.DetachedScaleGaussianPolicyHead()),
        critic=m.Critic(encoder=m.ObservationEncoder(), torso=m.MLP((HIDDEN, HIDDEN), torch.nn.Tanh),
                        head=m.ValueHead()),
        observation_normalizer=n.MeanStd())
    batch = total_envs * SEGMENT // MINIBATCHES     # GLOBAL minibatch (weak scaling)
    replay = tonic_b200.replays.Segment(size=SEGMENT, batch_iterations=EPOCHS, batch_size=batch)
    agent = tonic_b200.torch.agents.PPO(model=model, replay=replay)
    agent.initialize(env.observation_space, env.action_space, seed=seed)
    return agent, env, batch


def ppo_outputs(agent, env):
    """The last PPO iteration on a fixed seeded sample of environment columns: the segment it
    collected with the values, returns and advantages of its update, and the observations the
    next iteration starts from; then the updated model and the update's statistics."""
    import numpy as np
    import torch
    n = env.workers
    cols = np.sort(np.random.RandomState(0).choice(n, min(DUMP_ENVS, n), replace=False))
    cols = torch.as_tensor(cols, device=env.observations.device)
    out = {'segment.' + k: v.index_select(1, cols) for k, v in agent.replay.buffers.items()}
    out['env.observations'] = env.observations.index_select(0, cols)
    out.update(model_outputs(agent, agent._update_buffers[0]))
    return out


def multi_rank_parity(run):
    """N > 1: every rank reproduces its share of the teacher-forced golden scenarios
    (tests/multi_rank_scenario.py, the checker the 2-GPU test uses) before anything is timed."""
    if run.world == 1:
        return None
    try:
        from tests import multi_rank_scenario
        multi_rank_scenario.check_all()
        verdict = 'ok'
    except Exception as exc:        # report, do not hide the throughput numbers
        verdict = f'FAILED: {type(exc).__name__}: {str(exc)[:300]}'
    flags = [None] * run.world
    run.dist.all_gather_object(flags, verdict)
    bad = [f for f in flags if f != 'ok']
    return 'ok' if not bad else bad[0]


def run_ppo(args):
    import torch
    run = Run(args)
    world, rank = run.world, run.rank
    from tonic_b200 import _lib, config, graphs, kernels
    from tonic_b200.utils import logger
    parity = multi_rank_parity(run)
    iterations = dict(actor=0, critic=0)          # statistics are still read back every update

    def capture(key, value, stats=False, **kw):
        if key.endswith('/iterations'):
            iterations[key.split('/')[0]] += int(value)
    logger.store = capture
    logger.store_aggregate = lambda *a, **k: None

    total_envs = ENVS_PER_GPU * world
    config.noise = 'device'      # Philox action noise inside the kernels (no host traffic)
    config.indices = args.indices
    agent, env, batch = build_ppo(ENVS_PER_GPU, total_envs)
    update_timer = UpdateTimer(agent)
    env.start()

    def iteration():
        done = agent.rollout(env, SEGMENT)       # fills the segment, then runs the update
        assert done == SEGMENT

    for _ in range(args.warmup):
        iteration()
    run.barrier()
    sampler = ClockSampler(run.local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count() + graphs.replayed_launches
    iterations.update(actor=0, critic=0)
    update_timer.reset()
    elapsed_ms = run.timed(iteration, args.steps)
    sampler.stop_flag = True
    update_ms = run.max_over_ranks(update_timer.mean_ms() or 0.0)
    launches = _lib.launch_count() + graphs.replayed_launches - launches0
    timed_iterations = dict(iterations)
    env_steps = args.steps * SEGMENT * total_envs
    value = env_steps / (elapsed_ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ppo_outputs(agent, env))

    if args.quick:
        if rank == 0:
            print(json.dumps(dict(value=round(value, 1), ms_per_step=round(elapsed_ms / args.steps, 3),
                                  update_ms=round(update_ms, 3), gpu_launches=launches,
                                  minibatch_updates=timed_iterations, multi_rank_parity=parity,
                                  quick=True)))
        return
    # ---- e2e: the reference-facing protocol with HOST arrays ------------------------
    def host_iteration(observations, steps_count):
        for _ in range(SEGMENT):
            actions = agent.step(observations, steps_count)
            observations, infos = env.step(actions)
            agent.update(**infos, steps=steps_count)
            steps_count += ENVS_PER_GPU
        return observations, steps_count

    def measure(iters, warm):
        """The reference's protocol with numpy arrays crossing the boundary every vector step."""
        agent.replay.index = 0
        observations = env.start(host=True)
        steps_count = 0
        for _ in range(warm):
            observations, steps_count = host_iteration(observations, steps_count)
        torch.cuda.synchronize()
        run.barrier()
        kernels.transfers['h2d'] = kernels.transfers['d2h'] = 0
        iterations.update(actor=0, critic=0)
        update_timer.reset()
        t0 = time.time()
        for _ in range(iters):
            observations, steps_count = host_iteration(observations, steps_count)
        torch.cuda.synchronize()
        dt = run.max_over_ranks(time.time() - t0)      # slowest rank
        detail = dict(update_ms=round(run.max_over_ranks(update_timer.mean_ms() or 0.0), 3),
                      minibatch_updates_per_iteration={k: v // iters for k, v in iterations.items()})
        detail['protocol_us_per_vector_step'] = round(
            (dt / iters * 1e3 - detail['update_ms']) / SEGMENT * 1e3, 1)
        return (iters * SEGMENT * total_envs / dt, kernels.transfers['h2d'] // iters,
                kernels.transfers['d2h'] // iters, detail)
    # product configuration: device Philox noise + device permutations, update replayed as a
    # CUDA graph (3 warm iterations: 2 eager executions size the workspaces, 1 captures)
    e2e_iters = max(1, min(args.steps, 3))
    fast, h2d, d2h, e2e_detail = measure(e2e_iters, 3)
    # parity configuration: host torch RNG noise + numpy-compatible MT19937 permutations
    parity_value = None
    if world == 1:
        config.noise = config.indices = 'host'
        parity_value, _, _, _ = measure(1, 1)
        config.noise, config.indices = 'device', args.indices
        parity_value = round(parity_value, 1)
    e2e = dict(value=round(fast, 1), unit='env-steps/s', h2d_bytes_per_step=h2d,
               d2h_bytes_per_step=d2h, steps=e2e_iters, parity_mode_value=parity_value, **e2e_detail,
               note='agent.step / environment.step / agent.update called with numpy arrays '
                    'every vector step (pinned staging, copies inside the timed region; bytes '
                    'are per rank and per PPO iteration of 128 vector steps); value = product configuration '
                    '(device noise and permutations, graph-replayed update), parity_mode_value '
                    '= host torch RNG noise + host MT19937 permutations (bit-compatible streams); measured '
                    'right after the device-resident timed pass (same training phase: the number of actor '
                    'minibatches before the KL early stop grows with training and is reported beside '
                    'update_ms); protocol_us_per_vector_step = (iteration - update) / 128')

    # ---- instrumented pass: CUDA events around every launch (same workload, same kernels:
    # graphs off so that the C entry points record per-launch events, and the per-step rollout
    # chain the graph replays -- not the FFMA persistent-rollout kernel) ----------------------
    config.graphs = False
    saved_rollout = config.fused_rollout
    if saved_rollout == 'auto':
        config.fused_rollout = False
    kernels.flops.clear()
    iterations.update(actor=0, critic=0)
    kernels.profile_begin()
    t0 = time.time()
    for _ in range(args.steps):
        iteration()
    prof = kernels.profile_end()
    config.graphs = True
    config.fused_rollout = saved_rollout
    prof_wall_ms = (time.time() - t0) * 1e3
    total_kernel_ms = sum(ms for _, ms in prof.values())
    profiled_iterations = dict(iterations)
    pk = peaks()
    # FLOPs of launches that the device-side KL flag turned into no-ops are not counted:
    # the skipped actor minibatches are known from the logged iteration counters
    skipped = profiled_iterations['critic'] - profiled_iterations['actor']
    rows_local = batch // world
    gemm_names = ('tb_tc_mlp_train', 'tb_tc_mlp_forward', 'tb_tc_mlp_backward', 'tb_tc_gemm256_fwd',
                  'tb_tc_gemm256_bwd', 'tb_tc_wgrad256', 'tb_mlp_wgrad_fused', 'tb_mlp_forward',
                  'tb_mlp_backward', 'tb_mlp_wgrad')
    # algorithmic FLOPs of ONE skipped launch (they are actor-minibatch launches)
    actor_launch_flops = {
        'tb_tc_mlp_train': 2.0 * rows_local * (OBS * HIDDEN + HIDDEN * HIDDEN + HIDDEN * ACT)
        + 2.0 * rows_local * HIDDEN * (ACT + HIDDEN),
        'tb_tc_mlp_forward': 2.0 * rows_local * (OBS * HIDDEN + HIDDEN * HIDDEN + HIDDEN * ACT),
        'tb_tc_mlp_backward': 2.0 * rows_local * HIDDEN * (ACT + HIDDEN),
        'tb_mlp_wgrad_fused': 2.0 * rows_local * (HIDDEN * HIDDEN + HIDDEN * (OBS + 2)
                                                  + 2 * ACT * (HIDDEN + 1))}
    # rollout launches of the forward kernel evaluate 4096 rows, not a minibatch: count separately
    # entry points the skipped actor minibatches went through (device flag -> no-op launches)
    if 'tb_tc_mlp_train' in prof:
        skip_names = ('tb_tc_mlp_train', 'tb_mlp_wgrad_fused')
    else:
        skip_names = tuple(n for n in gemm_names if n not in ('tb_tc_mlp_train',))

    def executed_flops(name):
        total = kernels.flops.get(name, 0.0)
        if name in skip_names:
            per_launch = actor_launch_flops.get(name, 2.0 * rows_local * HIDDEN * HIDDEN)
            if name in ('tb_mlp_forward', 'tb_mlp_backward', 'tb_mlp_wgrad'):
                per_launch = total / max(prof.get(name, (1, 0))[0], 1)
            total -= skipped * per_launch
        return max(total, 0.0)
    gemms = [k for k in prof if k in gemm_names]
    top = max(gemms, key=lambda k: prof[k][1])
    top_count, top_ms = prof[top]
    top_flops = executed_flops(top)
    achieved = top_flops / (top_ms / 1e3) / 1e12 if top_ms > 0 else 0.0
    passes = {'tf32x3': 3, 'tf32': 1}.get(config.gemm, 0)
    P_actor = OBS * HIDDEN + HIDDEN + HIDDEN * HIDDEN + HIDDEN + ACT * HIDDEN + ACT + ACT
    P_critic = OBS * HIDDEN + HIDDEN + HIDDEN * HIDDEN + HIDDEN + HIDDEN + 1
    TN = SEGMENT * ENVS_PER_GPU
    hbm = hbm_table(prof, {
        # SURVEY 8(d): env state read+write 2*4*O + segment row write 4*(2O+A+4)
        'tb_env_step': (8 * OBS + 4 * (2 * OBS + ACT + 4)) * ENVS_PER_GPU,
        'tb_gauss_sample': 4 * (2 * ACT + 2 * ACT + 1) * ENVS_PER_GPU,      # minibatch launches differ: mixed
        'tb_moments_record': 4 * OBS * ENVS_PER_GPU,
        # sample + record + step in one launch: state read once, loc read, actions / log-probs /
        # obs / next_obs / flags written (the separate kernels' bytes minus the re-read rows)
        'tb_act_env_step': (4 * OBS + 4 * ACT + 4 * (2 * OBS + OBS + ACT + 1 + 3) + 12) * ENVS_PER_GPU,
        'tb_lambda_returns': 4 * 6 * TN,
        'tb_advantages': 4 * 3 * TN,               # per phase: read returns / values or advantages, write
        'tb_permutation': 8 * TN,
        'tb_gauss_policy_loss': (4 * (ACT + ACT + 2 + 2 * ACT) + 8) * rows_local,
        'tb_adam_step': 28 * (P_actor + P_critic) / 2,
    }, pk['hbm'])
    traffic = ncu_traffic()
    roofline = dict(
        kernel=top, bound='tensor', achieved=round(achieved, 3), peak=pk['tflops'],
        unit='TFLOP/s', frac=round(achieved / pk['tflops'], 5),
        traffic=traffic.get(top), peak_source=pk['source'], launches=top_count,
        executed_launches=top_count - (skipped if top in skip_names else 0),
        avg_launch_us=round(top_ms / max(top_count - (skipped if top in skip_names else 0), 1) * 1e3, 2),
        share_of_kernel_time=round(top_ms / total_kernel_ms, 4),
        flops_per_launch=round(top_flops / max(top_count - (skipped if top in skip_names else 0), 1), 1),
        tensor_pipe_tflops=round(achieved * max(passes, 1), 3),
        note=('dominant GEMM entry point by CUDA-event time in an eager (graphs off) pass of the '
              'same K steps with the same kernels; achieved = algorithmic fp32-equivalent FLOPs of the '
              'executed launches (forward->loss->backward kernel: 2*rows*(d_in*256 + 256*256 + 256*n_out) + '
              '2*rows*256*(n_out + 256); weight-gradient + Adam kernel: 2*rows*(256*256 + '
              '256*(d_in+2) + (n_out+extras)*257)) / event time; ' +
              ('FP32 FFMA kernels' if passes == 0 else
               f'tcgen05 kind::tf32 with {passes} MMA pass(es) per product, so the tensor pipe '
               f'itself runs {passes}x the achieved figure (tensor_pipe_tflops)') +
              '; peak = measured dense bf16 tensor throughput; traffic = dram read+write bytes per '
              'launch from the committed warm-cache ncu capture of the minibatch chain (profiles/)'),
        kernels={k: dict(launches=c, ms=round(ms, 3),
                         tflops=round(executed_flops(k) / (ms / 1e3) / 1e12, 3) if ms and k in gemm_names else None)
                 for k, (c, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1])},
        hbm_kernels=hbm, hbm_peak_gbs=pk['hbm'],
        hbm_note='memory-bound kernels: algorithmic bytes per launch (SURVEY 8d) / CUDA-event time per '
                 'launch; at these sizes (<= 12 MB per launch) they are launch-latency bound, not HBM bound')

    # ---- off-policy configurations (BASELINE configs[2] / [3]) measured in the same run ------
    offpolicy = None
    if world == 1 and not args.no_offpolicy:
        del agent, env
        torch.cuda.empty_cache()
        offpolicy = {}
        for name in ('sac', 'td3', 'ddpg'):
            try:
                offpolicy[name] = measure_offpolicy(run, name, steps=10, warmup=3, batch=100)
            except Exception as exc:
                offpolicy[name] = dict(error=f'{type(exc).__name__}: {str(exc)[:200]}')
    if rank != 0:
        return
    cpu = cpu_baseline() if world == 1 else None
    line = dict(
        metric='env-steps/sec (PPO, 4096 envs per GPU, 2x256 MLP)', value=round(value, 1),
        unit='env-steps/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=round(elapsed_ms / args.steps, 3), higher_is_better=True, scaling='weak',
        vs_baseline=None, dtype='f32', data='synthetic',
        config=dict(workload='PPO, synthetic HalfCheetah-shape env (obs=17, act=6), 4096 envs '
                             'per GPU, T=128 segment, E=10 epochs x 32 minibatches, 2x256 tanh MLP',
                    envs_per_gpu=ENVS_PER_GPU, segment=SEGMENT, epochs=EPOCHS, minibatch=batch,
                    hidden=HIDDEN, parallelism=f'dp{world} (envs sharded, grad all-reduce)',
                    l2='working set per iteration (segment 92 MB + activations 69 MB/minibatch) '
                       'exceeds the 126 MB L2; no explicit flush',
                    gemm=config.gemm, cuda_graphs=bool(config.graphs), noise='device Philox',
                    indices=('device Feistel permutation' if args.indices == 'device'
                             else 'host MT19937 (numpy-compatible)')),
        clocks=sampler.summary(), gpu_launches=launches, update_ms=round(update_ms, 3),
        minibatch_updates=dict(
            critic=timed_iterations['critic'], actor=timed_iterations['actor'],
            note='actor updates stop early inside an iteration when KL > 0.015 (reference '
                 'default, ppo.py:45-46): a device flag turns the remaining actor kernels of '
                 'that iteration into no-ops; critic updates always run'),
        multi_rank_parity=parity,
        e2e=e2e, roofline=roofline, offpolicy=offpolicy,
        cpu_baseline=cpu,
        profiled_pass=dict(kernel_ms_per_step=round(total_kernel_ms / args.steps, 3),
                           wall_ms_per_step=round(prof_wall_ms / args.steps, 3),
                           note='graphs off, per-launch CUDA events; same kernels as the timed pass'))
    print(json.dumps(line))


# ------------------------------------------------------------------------ off-policy
def build_offpolicy(name, envs_local, total_envs, batch, seed=0):
    import torch
    import tonic_b200
    import tonic_b200.torch
    kind, preset, obs, act, _ = OFF_POLICY[name]
    m, n = tonic_b200.torch.models, tonic_b200.torch.normalizers
    spec = tonic_b200.environments.SynthControl(preset, max_episode_steps=MAX_EPISODE_STEPS)
    env = tonic_b200.environments.distribute(lambda: spec, 1, total_envs)
    assert env.workers == envs_local
    env.initialize(seed=seed)
    critic = m.Critic(encoder=m.ObservationActionEncoder(), torso=m.MLP((HIDDEN, HIDDEN), torch.nn.ReLU),
                      head=m.ValueHead())
    if kind == 'SAC':
        head = m.GaussianPolicyHead(loc_activation=torch.nn.Identity,
                                    distribution=m.SquashedMultivariateNormalDiag)
    else:
        head = m.DeterministicPolicyHead()
    actor = m.Actor(encoder=m.ObservationEncoder(), torso=m.MLP((HIDDEN, HIDDEN), torch.nn.ReLU), head=head)
    wrapper = m.ActorCriticWithTargets if kind == 'DDPG' else m.ActorTwinCriticWithTargets
    model = wrapper(actor=actor, critic=critic, observation_normalizer=n.MeanStd())
    # the ring is local to the rank: 1M transitions per GPU (BASELINE configs[2])
    replay = tonic_b200.replays.Buffer(size=REPLAY_SIZE, batch_iterations=50, batch_size=batch,
                                       steps_before_batches=1 << 60,      # the bench fills the ring first
                                       steps_between_batches=50)
    if kind == 'SAC':
        exploration = tonic_b200.explorations.NoActionNoise(start_steps=0)
    else:
        exploration = tonic_b200.explorations.NormalActionNoise(start_steps=0)
    agent = getattr(tonic_b200.torch.agents, kind)(model=model, replay=replay, exploration=exploration)
    agent.initialize(env.observation_space, env.action_space, seed=seed)
    return agent, env


def offpolicy_outputs(agent, env):
    """The last vector step: the actions, what the environment returned for them (the transition
    stored in the ring), the updated model and the update's statistics."""
    out = {'actions': agent._staged_actions}
    for k in ('observations', 'next_observations', 'rewards', 'resets', 'terminations'):
        out['env.' + k] = getattr(env, k)
    out.update(model_outputs(agent, agent._update_stats))
    return out


def measure_offpolicy(run, name, steps, warmup, batch, dump_dir=None):
    """Fills the device ring (untimed: collector only), then times `steps` vector steps, each
    followed by the reference's update (50 iterations x batch); `dump_dir`: writes the outputs
    of the last timed step there."""
    import torch
    from tonic_b200 import _lib, config, kernels
    from tonic_b200.utils import logger
    kind, preset, obs, act, envs = OFF_POLICY[name]
    world = run.world
    batch = batch * world                    # GLOBAL batch (every rank contributes `batch` rows)
    config.noise, config.indices = 'device', 'device'
    saved = logger.store, logger.store_aggregate
    logger.store = lambda *a, **k: None
    logger.store_aggregate = lambda *a, **k: None
    from tonic_b200 import graphs
    agent, env = build_offpolicy(name, envs, envs * world, batch)
    env.start()
    state = dict(steps=1)

    def vector_step():
        # the fused driver of tonic_b200.Trainer: act -> environment -> store -> record -> update,
        # device resident, replayed as a CUDA graph once captured
        agent.rollout(env, 1, steps=state['steps'])
        state['steps'] += envs * world

    fill = -(-REPLAY_SIZE // envs)           # vector steps that fill the ring (no update yet)
    for _ in range(fill):
        vector_step()
    assert agent.replay.size == agent.replay.max_size
    collect_ms = run.timed(vector_step, steps) / steps       # collector only (ring full, no update)
    agent.replay.steps_before_batches = 0    # from here on: one update per vector step
    for _ in range(max(warmup, 3)):          # 2 eager executions size the workspaces, 1 captures
        vector_step()
    launches0 = _lib.launch_count() + graphs.replayed_launches
    ms = run.timed(vector_step, steps)
    launches = _lib.launch_count() + graphs.replayed_launches - launches0
    if dump_dir and run.rank == 0:
        dump_outputs(dump_dir, offpolicy_outputs(agent, env))
    update_ms = ms / steps - collect_ms      # device time added by the update to one vector step
    # instrumented pass (graphs off: per-launch events)
    config.graphs = False
    kernels.flops.clear()
    kernels.profile_begin()
    for _ in range(min(steps, 5)):
        vector_step()
    prof = kernels.profile_end()
    config.graphs = True
    n_prof = min(steps, 5)
    pk = peaks()
    nets = agent.model.networks()
    P_total = sum(n.params.numel() for n in nets)
    row_bytes = 4 * (2 * obs + act + 2)        # SURVEY 8(d): gathered bytes per sampled transition
    hbm = hbm_table(prof, {
        'tb_env_step': (8 * obs + 4 * (2 * obs + act + 4)) * envs,
        'tb_q_target': (4 * 5 + 8) * (batch // world),
        'tb_soft_update': 12 * P_total / max(len(nets) // 2, 1),
        'tb_adam_step': 28 * P_total / max(len(nets), 1),
        'tb_moments_record': 4 * obs * envs,
    }, pk['hbm'])
    gemm_ms = sum(ms_ for k, (c, ms_) in prof.items() if 'mlp' in k or 'gemm' in k or 'wgrad' in k)
    gemm_flops = sum(v for k, v in kernels.flops.items()
                     if k in ('tb_mlp_forward', 'tb_mlp_forward_tc', 'tb_mlp_backward', 'tb_mlp_backward_tc',
                              'tb_mlp_wgrad', 'tb_mlp_wgrad_tc', 'tb_mlp_wgrad_fused'))
    out = dict(
        workload=f'{kind}, synthetic {preset}-shape env (obs={obs}, act={act}), {envs} envs per GPU, '
                 f'device replay {REPLAY_SIZE} transitions per GPU (full), 2x256 ReLU MLPs, '
                 f'50 iterations x batch {batch} per update (replays/buffers.py:8-12), one update per '
                 'vector step',
        value=round(steps * envs * world / (ms / 1e3), 1), unit='env-steps/s',
        ms_per_vector_step=round(ms / steps, 3), update_ms=round(update_ms, 3),
        collect_ms=round(collect_ms, 4), cuda_graphs=bool(config.graphs),
        update_iterations=50, batch=batch, gpu_launches_per_step=launches // steps,
        replay_bytes=int(agent.replay.max_size * envs * 4 * (2 * obs + act + 3)),
        sampled_bytes_per_update=50 * batch * row_bytes,
        gemm=dict(ms_per_update=round(gemm_ms / n_prof, 3),
                  tflops=round(gemm_flops / max(gemm_ms, 1e-9) / 1e9, 3),
                  note='all MLP forward / backward / weight-gradient launches of one update (algorithmic '
                       'fp32 FLOPs / CUDA-event time); at 100 rows per launch they are launch-latency bound'),
        hbm_kernels=hbm,
        kernels={k: dict(launches=c // n_prof, ms=round(ms_ / n_prof, 4))
                 for k, (c, ms_) in sorted(prof.items(), key=lambda kv: -kv[1][1])[:12]})
    logger.store, logger.store_aggregate = saved
    del agent, env
    torch.cuda.empty_cache()
    return out


def run_offpolicy(args):
    run = Run(args)
    from tonic_b200 import config
    name = args.workload
    kind, preset, obs, act, envs = OFF_POLICY[name]
    sampler = ClockSampler(run.local_rank)
    if run.rank == 0:
        sampler.start()
    res = measure_offpolicy(run, name, args.steps, args.warmup, args.offpolicy_batch, args.dump_outputs)
    sampler.stop_flag = True
    if run.rank != 0:
        return
    cpu = cpu_baseline_offpolicy(name) if run.world == 1 and not args.quick else None
    pk = peaks()
    top = max(res['hbm_kernels'].items(), key=lambda kv: kv[1]['avg_launch_us'] * kv[1]['launches'],
              default=(None, None))
    line = dict(
        metric=f'env-steps/sec ({kind}, {envs} envs per GPU, 2x256 MLP, device replay 1M)',
        value=res['value'], unit='env-steps/s', n_gpus=run.world, steps=args.steps, warmup=args.warmup,
        ms_per_step=res['ms_per_vector_step'], higher_is_better=True, scaling='weak', vs_baseline=None,
        dtype='f32', data='synthetic',
        config=dict(workload=res['workload'], envs_per_gpu=envs, gemm=config.gemm,
                    parallelism=f'dp{run.world} (envs + replay columns sharded, grad all-reduce)',
                    l2='the 1M-transition ring (3.1 GB at 376/17) is far larger than L2: sampled rows come from HBM'),
        clocks=sampler.summary(), gpu_launches=res['gpu_launches_per_step'] * args.steps,
        update_ms=res['update_ms'],
        roofline=dict(kernel=top[0], bound='hbm', unit='GB/s', peak=pk['hbm'],
                      achieved=top[1]['achieved_gbs'] if top[1] else None,
                      frac=top[1]['frac'] if top[1] else None, traffic=None, peak_source=pk['source'],
                      hbm_kernels=res['hbm_kernels'], gemm=res['gemm'], kernels=res['kernels']),
        e2e=None, cpu_baseline=cpu, offpolicy=res)
    print(json.dumps(line))


# ------------------------------------------------------------------------- reference
def _set_threads(n):
    import torch
    torch.set_num_threads(max(1, int(n)))


def oracle_iteration_factory(envs, seed=0, groups=1):
    """The oracle port's PPO on the same workload shape (bounded number of envs); `groups` > 1:
    the reference's forked `--parallel groups --sequential envs/groups` worker grid."""
    from oracle import port
    if groups > 1:
        env = port.ParallelVectorEnv(OBS, ACT, groups, envs // groups, MAX_EPISODE_STEPS)
    else:
        env = port.VectorEnv(OBS, ACT, envs, MAX_EPISODE_STEPS)
    env.initialize(seed)
    batch = envs * SEGMENT // MINIBATCHES
    agent = port.OnPolicyOracle('PPO', (HIDDEN, HIDDEN),
                                dict(size=SEGMENT, batch_iterations=EPOCHS, batch_size=batch))
    agent.initialize(env.observation_space, env.action_space, seed=seed)
    state = dict(obs=env.start(), steps=0)

    def iteration():
        for _ in range(SEGMENT):         # trainer.py:44-50
            actions = agent.step(state['obs'], state['steps'])
            state['obs'], infos = env.step(actions)
            agent.update(**infos, steps=state['steps'])
            state['steps'] += envs
    iteration.close = getattr(env, 'close', lambda: None)
    return iteration


def host_cores():
    """Physical cores this process may use (hyper-threads halved when visible)."""
    try:
        logical = len(os.sched_getaffinity(0))
    except AttributeError:
        logical = os.cpu_count() or 1
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = logical
    return min(logical, physical), logical


CPU_ENVS = int(os.environ.get('TB_BENCH_CPU_ENVS', 256))   # bounded sample: the reference steps envs in a per-env Python loop, so
                      # env-steps/s is flat in the number of envs (BASELINE.md section 2)


def cpu_grid(seconds_budget=45.0):
    """env-steps/s of the oracle port (one PPO iteration of CPU_ENVS envs per sample) for
    torch intra-op threads in {1, 8, all physical cores} and for the forked worker grid
    `--parallel C' --sequential CPU_ENVS/C'`; best of up to 3 samples each, pinned thread
    counts (64 unpinned threads on 256-row GEMMs swung 5x between boxes in round 1)."""
    import torch
    physical, logical = host_cores()
    results = []
    configs = [('sequential', 1, 1), ('sequential', min(8, physical), 1)]
    if physical > 8:
        configs.append(('sequential', physical, 1))
    groups = max(2, min(16, physical // 2))
    while CPU_ENVS % groups:
        groups -= 1
    configs.append(('parallel', max(1, min(8, physical - groups)), groups))
    t_start = time.time()
    for mode, threads, grp in configs:
        _set_threads(threads)
        iteration = oracle_iteration_factory(CPU_ENVS, groups=grp)
        try:
            iteration()                       # warm-up (allocations, first update)
            best = None
            for _ in range(3):
                t0 = time.time()
                iteration()
                dt = time.time() - t0
                best = dt if best is None else min(best, dt)
                if time.time() - t_start > seconds_budget * (len(results) + 1) / len(configs):
                    break
        finally:
            iteration.close()
        results.append(dict(mode=(f'--parallel {grp} --sequential {CPU_ENVS // grp}' if grp > 1
                                  else f'--parallel 1 --sequential {CPU_ENVS}'),
                            torch_threads=threads, env_steps_per_s=round(SEGMENT * CPU_ENVS / best, 1),
                            seconds=round(best, 2)))
    _set_threads(physical)
    return results, physical, logical


def cpu_baseline():
    grid, physical, logical = cpu_grid()
    best = max(grid, key=lambda r: r['env_steps_per_s'])
    return dict(value=best['env_steps_per_s'], unit='env-steps/s', cores=best['torch_threads'],
                host_cores=dict(physical=physical, logical=logical), kind='port',
                sample=f'best of up to 3 x 1 PPO iteration of {CPU_ENVS} envs x {SEGMENT} steps + full '
                       f'update (E={EPOCHS}, {MINIBATCHES} minibatches/epoch, 2x256 MLP) per '
                       'configuration; bounded sample of the 4096-env workload: the reference steps '
                       'envs in a per-env Python loop, so steps/s is flat in the number of envs',
                best=best['mode'], grid=grid)


def cpu_baseline_offpolicy(name, envs=64, vector_steps=12):
    """The oracle port's off-policy agent: `vector_steps` vector steps of `envs` envs, one update
    (50 x batch 100) per vector step, replay pre-filled with 2000 transitions."""
    from oracle import port
    kind, preset, obs, act, _ = OFF_POLICY[name]
    physical, _ = host_cores()
    _set_threads(min(8, physical))
    env = port.VectorEnv(obs, act, envs, MAX_EPISODE_STEPS)
    env.initialize(0)
    agent = port.OffPolicyOracle(kind, (HIDDEN, HIDDEN),
                                 dict(size=REPLAY_SIZE, batch_iterations=50, batch_size=100,
                                      steps_before_batches=envs * 32, steps_between_batches=50),
                                 start_steps=0)
    agent.initialize(env.observation_space, env.action_space, seed=0)
    state = dict(obs=env.start(), steps=1)

    def vector_step():
        actions = agent.step(state['obs'], state['steps'])
        state['obs'], infos = env.step(actions)
        agent.update(**infos, steps=state['steps'])
        state['steps'] += envs
    for _ in range(34):
        vector_step()
    t0 = time.time()
    for _ in range(vector_steps):
        vector_step()
    dt = time.time() - t0
    return dict(value=round(vector_steps * envs / dt, 1), unit='env-steps/s', cores=min(8, physical),
                kind='port', update_ms=None,
                sample=f'{vector_steps} vector steps of {envs} envs, one update (50 x batch 100) per '
                       'vector step; the update dominates, so env-steps/s scales with the number of '
                       f'envs per vector step (GPU arm: {OFF_POLICY[name][4]})',
                seconds=round(dt, 2))


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm (oracle port -- the Python
    reference cannot travel to the GPU box) on the host cores, all the threads it can use:
    the fastest configuration of the thread / worker-grid sweep is the one timed."""
    if int(os.environ.get('RANK', 0)) != 0:
        return
    grid, physical, logical = cpu_grid(seconds_budget=60.0)
    best = max(grid, key=lambda r: r['env_steps_per_s'])
    groups = 1
    if best['mode'].startswith('--parallel') and not best['mode'].startswith('--parallel 1 '):
        groups = int(best['mode'].split()[1])
    _set_threads(best['torch_threads'])
    iteration = oracle_iteration_factory(CPU_ENVS, groups=groups)
    try:
        for _ in range(args.warmup):
            iteration()
        t0 = time.time()
        for _ in range(args.steps):
            iteration()
        dt = time.time() - t0
    finally:
        iteration.close()
    value = round(args.steps * SEGMENT * CPU_ENVS / dt, 1)
    sample = (f'each step = 1 PPO iteration of {CPU_ENVS} envs x {SEGMENT} steps + full update '
              f'(E={EPOCHS}, {MINIBATCHES} minibatches/epoch, 2x256 MLP), configuration {best["mode"]} '
              f'with {best["torch_threads"]} torch threads (fastest of the sweep in `grid`)')
    print(json.dumps(dict(
        impl='reference', metric='env-steps/sec (PPO, 4096 envs per GPU, 2x256 MLP)', value=value,
        unit='env-steps/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
        ms_per_step=round(dt / args.steps * 1e3, 3), higher_is_better=True, scaling='weak',
        vs_baseline=None, dtype='f32', data='synthetic',
        config=dict(workload='PPO, synthetic HalfCheetah-shape env (obs=17, act=6), bounded '
                             f'sample of {CPU_ENVS} envs, T=128, E=10 x 32 minibatches, 2x256 tanh MLP'),
        cpu_baseline=dict(value=value, unit='env-steps/s', cores=best['torch_threads'],
                          host_cores=dict(physical=physical, logical=logical), kind='port',
                          sample=sample, grid=grid),
        e2e=dict(value=value, unit='env-steps/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--gpus', type=int, default=1)
    parser.add_argument('--steps', type=int, default=5)
    parser.add_argument('--warmup', type=int, default=3)
    parser.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    parser.add_argument('--workload', default='ppo', choices=['ppo', 'sac', 'td3', 'ddpg'])
    parser.add_argument('--offpolicy-batch', type=int, default=100,
                        help='batch size of the off-policy updates (reference default 100)')
    parser.add_argument('--no-offpolicy', action='store_true',
                        help='PPO workload: skip the short SAC / TD3 / DDPG measurements')
    parser.add_argument('--indices', default='device', choices=['host', 'device'],
                        help="minibatch permutations: 'device' (Feistel, on the GPU) or 'host' "
                             "(numpy-compatible MT19937 stream, bit-identical to the reference)")
    parser.add_argument('--quick', action='store_true',
                        help='timed region only (for runs under ncu): no e2e / cpu_baseline / profile pass')
    parser.add_argument('--dump-outputs', metavar='DIR',
                        help='write the outputs of the last timed step as DIR/<name>.npy')
    args = parser.parse_args()
    if args.steps < 1:
        parser.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        parser.error('--dump-outputs covers the GPU implementation only')
    if args.impl == 'reference':
        run_reference(args)
    else:
        assert args.warmup >= 3 or os.environ.get('TB_ALLOW_SHORT_WARMUP'), 'W >= 3 warm-up steps'
        if args.workload == 'ppo':
            run_ppo(args)
        else:
            run_offpolicy(args)


if __name__ == '__main__':
    main()
