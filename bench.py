#!/usr/bin/env python
"""bench.py - headline benchmark of the ProMP hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--workload point|cheetah] [--impl reference] [--dump-outputs DIR]

A "step" is ONE FULL META-ITERATION of the hot path over one batch of synthetic tasks
(BASELINE.json configs[1]: MetaPointEnvCorner, 40 tasks x 20 envs x H=100, ProMP, 2x(64) Gaussian MLP):
  update_tasks -> [rollout -> returns/baseline/GAE] -> inner adapt -> [rollout -> processing]
  -> ProMP outer step (5 Adam epochs of the second-order meta-gradient + stats pass).
metric = env-steps/s = (M*E*H*2 env steps per meta-iteration) / (time per meta-iteration), whole job.

  value : device-resident loop (reset states drawn in-kernel, nothing logged to the host), CUDA events, one CUDA-graph replay
          of the ~29 launches of a meta-iteration per step.
  e2e   : the same iteration through the DEFAULT entry point of a run script, promp_b200.meta_trainer.Trainer(...).train():
          per iteration numpy-drawn tasks + reset states (reference RNG order) -> pinned -> ONE H2D copy, graph replay (captured
          automatically), ONE D2H of the logged scalars, every reference logger key emitted, logger.dumpkvs().
          e2e.eager = Trainer(use_cuda_graph=False).train_iteration(itr, log=True): what configurations with a host decision
          inside the iteration get.
  other_configs : short measurements, in the same run and through Trainer.train(), of the other BASELINE.json configurations:
          HalfCheetah surrogate (configs[2] per GPU = configs[4] at N = 8, weak scaling), MAML-TRPO on PointEnv (configs[3]:
          40 tasks in total, STRONG scaling over the N GPUs) and, at N = 1, ProMP with adaptive_inner_kl_penalty=True (the
          reference class default; the rule runs on the device, so the iteration is still one graph replay).
  roofline     : dominant kernel (policy_grad / policy_hvp).  These kernels are issue / latency-bound (AI ~ 1 kFLOP/B, inputs
                 L2-resident): bound = "issue", achieved / peak / frac = algorithmic fp32 TFLOP/s over the fp32-SIMT peak; the HBM
                 view (SURVEY.md 8d bytes per sample / launch time over the MEASURED_PEAKS.json copy bandwidth) is in roofline.hbm,
                 and the HBM-side stage (process_fused_kernel) in roofline.process_kernel.
  cpu_baseline : the CPU oracle port of the reference (oracle/) on the host cores: numpy half in min(tasks, cores) worker
                 processes (like the reference's parallel=True executor), TF1 half on PyTorch-CPU threads.

--impl reference times the reference's CPU implementation (oracle port: /root/reference is absent on the
GPU box and TF1 is not installable) on the same metric; launched for N GPUs it processes 40*N tasks on min(40*N, cores)
workers, so the N > 1 ratios are like for like.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    'point': dict(env='MetaPointEnvCorner', M=40, E=20, H=100, Do=2, Da=2,
                  name='ProMP MetaPointEnvCorner meta_batch=40 x envs_per_task=20, H=100 (BASELINE.json configs[1])'),
    'cheetah': dict(env='HalfCheetahRandDirecEnv', M=40, E=20, H=200, Do=17, Da=6,
                    name='ProMP HalfCheetahRandDirec-surrogate meta_batch=40 x 20, H=200 (BASELINE.json configs[2])'),
}
PROMP = dict(inner_lr=0.1, learning_rate=1e-3, num_ppo_steps=5, clip_eps=0.3, target_inner_step=0.01,
             init_inner_kl_penalty=5e-4, adaptive_inner_kl_penalty=False, num_inner_grad_steps=1)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, sm_max_mhz=1965.0), 'fallback'


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                       '-lms', '100'], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        os.unlink(self.f.name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(max(mx)) if mx else None,
                    samples=len(sm), reasons=sorted(reasons))


# ------------------------------------------------------------------------------------------- GPU arm
TRPO = dict(step_size=0.01, inner_type='log_likelihood', inner_lr=0.1, num_inner_grad_steps=1)    # maml_run_mujoco.py defaults


def build_stack(wl, reset_mode, task_shard=None, algo='promp', tasks=None, **trainer_kw):
    from promp_b200.envs import normalize, MetaPointEnvCorner, HalfCheetahRandDirecEnv
    from promp_b200.policies import MetaGaussianMLPPolicy
    from promp_b200.samplers import MetaSampler, MetaSampleProcessor
    from promp_b200.baselines import LinearFeatureBaseline
    from promp_b200.meta_algos import ProMP, TRPOMAML
    from promp_b200.meta_trainer import Trainer
    M = wl['M'] if tasks is None else tasks
    env = normalize(MetaPointEnvCorner() if wl['env'] == 'MetaPointEnvCorner' else HalfCheetahRandDirecEnv())
    policy = MetaGaussianMLPPolicy(name="meta-policy", obs_dim=wl['Do'], action_dim=wl['Da'], meta_batch_size=M,
                                   hidden_sizes=(64, 64))
    sampler = MetaSampler(env=env, policy=policy, rollouts_per_meta_task=wl['E'], meta_batch_size=M,
                          max_path_length=wl['H'], parallel=True, reset_mode=reset_mode, seed=1, task_shard=task_shard)
    proc = MetaSampleProcessor(baseline=LinearFeatureBaseline(), discount=0.99, gae_lambda=1, normalize_adv=True)
    if algo in ('promp', 'promp_adaptive_kl'):
        alg = ProMP(policy=policy, inner_lr=PROMP['inner_lr'], meta_batch_size=M,
                    num_inner_grad_steps=PROMP['num_inner_grad_steps'], learning_rate=PROMP['learning_rate'],
                    num_ppo_steps=PROMP['num_ppo_steps'], clip_eps=PROMP['clip_eps'],
                    target_inner_step=PROMP['target_inner_step'], init_inner_kl_penalty=PROMP['init_inner_kl_penalty'],
                    adaptive_inner_kl_penalty=True if algo == 'promp_adaptive_kl' else PROMP['adaptive_inner_kl_penalty'])
    else:
        alg = TRPOMAML(policy=policy, step_size=TRPO['step_size'], inner_type=TRPO['inner_type'], inner_lr=TRPO['inner_lr'],
                       meta_batch_size=M, num_inner_grad_steps=TRPO['num_inner_grad_steps'], exploration=False)
    trainer = Trainer(algo=alg, policy=policy, env=env, sampler=sampler, sample_processor=proc, n_itr=1,
                      num_inner_grad_steps=PROMP['num_inner_grad_steps'], **trainer_kw)
    return trainer


DUMP_LIMIT_BYTES = 64 << 20
PHASE_OUTPUTS = ('obs', 'act', 'mean', 'log_std', 'rew', 'returns', 'adv', 'coeffs', 'stats')


def dump_outputs(out_dir, policy, phases):
    """Write what one timed meta-iteration hands its caller as out_dir/<name>.npy: the updated policy parameters (theta)
    and, per sampling phase s, the trajectories, the policy's distribution parameters, returns, advantages, baseline
    coefficients and path statistics (phase<s>_<name>).  Inputs are seeded, so two builds run with the same arguments can
    be compared array by array."""
    arrays = {'theta': policy.theta}
    for s, ph in enumerate(phases):
        arrays.update(('phase%d_%s' % (s, name), getattr(ph, name)) for name in PHASE_OUTPUTS)
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


class LaunchCounter(object):
    """Counts OUR kernel launches by wrapping the ctypes entry points (kernels per call from the .cu files)."""
    KERNELS = dict(promp_rollout=1, promp_env_step=1, promp_env_observe=1, promp_process_samples=1,
                   promp_adj_avg_rewards=1, promp_policy_grad=1, promp_policy_hvp=1, promp_reduce_tasks=1,
                   promp_adam_tf1=2, promp_policy_forward=1, promp_counter_add=1, promp_meta_loss_terms=1,
                   promp_policy_grad_ragged=1, promp_policy_hvp_ragged=1, promp_process_samples_ragged=1,
                   promp_vec_axpy=1, promp_cg_init=1, promp_cg_step=1, promp_trpo_step=1, promp_trpo_select=1,
                   promp_allreduce_p2p=1, promp_baseline_fit=1, promp_baseline_predict=1,
                   promp_meta_update=1, promp_meta_loss_terms_p2p=1, promp_policy_grad_ex=1, promp_rollout_early_term=1,
                   promp_paths_finalize=4, promp_phase_log_terms=1, promp_promp_log_terms=1,
                   promp_policy_chain=1, promp_adapt_kl_coeff=1)
    # entry points that launch the same kernel are timed under one name
    ALIAS = dict(promp_policy_grad_ex='promp_policy_grad', promp_policy_grad_ragged='promp_policy_grad',
                 promp_policy_hvp_ragged='promp_policy_hvp', promp_process_samples_ragged='promp_process_samples')

    def __init__(self, time_kernels=False):
        from promp_b200 import _lib
        self._lib = _lib
        self.count = 0
        self.calls = {}
        self.time_kernels = time_kernels
        self.events = {}
        self._orig = _lib.call

    def __enter__(self):
        import torch
        orig, me = self._orig, self

        def call(name, *args):
            k = me.KERNELS.get(name, 0)
            if name == 'promp_policy_chain':     # one dataflow kernel or one kernel per stage: ask the library which
                k = me._lib.load().promp_policy_chain_num_launches(args[0], args[1], args[2], args[3], args[5], args[6])
            me.count += k
            me.calls[name] = me.calls.get(name, 0) + 1
            if me.time_kernels and k:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                orig(name, *args)
                b.record()
                me.events.setdefault(me.ALIAS.get(name, name), []).append((a, b))
            else:
                orig(name, *args)
        self._lib.call = call
        return self

    def __exit__(self, *exc):
        self._lib.call = self._orig

    def kernel_ms(self):
        import torch
        torch.cuda.synchronize()
        return {n: [a.elapsed_time(b) for a, b in ev] for n, ev in self.events.items()}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from promp_b200 import _lib
    from promp_b200.utils import logger
    logger.set_quiet(True)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    _lib.require_cuda()
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        import datetime
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank), timeout=datetime.timedelta(seconds=120))
        from promp_b200.utils.dist import enable_p2p_allreduce
        p2p = enable_p2p_allreduce()
    wl = WORKLOADS[args.workload]
    M, E, H = wl['M'], wl['E'], wl['H']
    steps_per_iter = M * E * H * (PROMP['num_inner_grad_steps'] + 1) * world      # weak scaling: M tasks per GPU
    shard = (rank, world) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(trainer, log, n_warm, n_steps, step_fn=None):
        """(device ms, wall ms, what the last timed step returned)"""
        run = step_fn if step_fn is not None else (lambda: trainer.train_iteration(0, log=log))
        for i in range(n_warm):
            run()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for i in range(n_steps - 1):
            run()
        last = run()        # only the last result is kept: holding each one into the next step would double the eager buffers
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = a.elapsed_time(b)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), last

    # ---- value: device-resident loop --------------------------------------------------------------
    np.random.seed(1)
    tr_dev = build_stack(wl, 'device', shard)
    clocks = ClockSampler(local_rank) if rank == 0 else None
    use_graph = not args.no_graph       # N > 1: the all-reduce inside the graph is the P2P kernel (promp_allreduce_p2p)
    with LaunchCounter() as lc:
        ms_eager, wall_eager, last = timed(tr_dev, False, args.warmup, args.steps)
    launches = lc.count // (args.warmup + args.steps)
    if use_graph:
        # the same ~40 launches per meta-iteration captured once into a CUDA graph and replayed
        step_fn = tr_dev.capture_graph(warmup=2)
        ms_dev, wall_dev, phases = timed(tr_dev, False, args.warmup, args.steps, step_fn)
    else:
        ms_dev, wall_dev = ms_eager, wall_eager
        phases = [samples[0].phase for samples in last]
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr_dev.policy, phases)
    # ---- e2e: the default entry point of a run script - Trainer.train() - with host inputs / logged outputs ----------
    def timed_train(trainer, n_warm, n_steps):
        """Time n_steps meta-iterations of trainer.train() (device events + wall clock, max over ranks) after n_warm."""
        trainer.start_itr, trainer.n_itr = 0, n_warm
        trainer.train()                                   # warm-up iterations (captures the CUDA graph when possible)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        trainer.start_itr, trainer.n_itr = n_warm, n_warm + n_steps
        t0 = time.perf_counter()
        a.record()
        trainer.train()
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        t = torch.tensor([a.elapsed_time(b), wall * 1e3], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    np.random.seed(1)
    tr_e2e = build_stack(wl, 'numpy', shard)              # Trainer defaults: use_cuda_graph='auto', prefetch_host_inputs=True
    sd = tr_e2e.sampler.spec
    S = PROMP['num_inner_grad_steps'] + 1
    if use_graph:
        ms_e2e, wall_e2e = timed_train(tr_e2e, args.warmup, args.steps)
        h2d, d2h = tr_e2e.graph_h2d_bytes, tr_e2e.graph_d2h_bytes
        e2e_api = ('promp_b200.meta_trainer.Trainer(...).train() with its defaults - the call an unchanged run script makes '
                   '(run_scripts/pro-mp_run_point_mass.py:66-77): per iteration numpy-drawn tasks + reset states in the reference RNG '
                   'order (reset_mode=numpy, next iteration drawn into a second pinned slot while the GPU runs), H2D from pinned memory, '
                   'one CUDA-graph replay of the device part (captured automatically: fixed-horizon env, fixed KL coefficient), one D2H '
                   'of the logged scalars, logger.logkv of every reference key, logger.dumpkvs()')
    else:
        ms_e2e, wall_e2e, _ = timed(tr_e2e, True, args.warmup, args.steps)
        h2d = 4 * (M * sd['task_dim'] + S * M * E * sd['state_dim'])
        d2h = S * (M * 8 * 8 + M * sd['act_dim'] * 4 + (2 * M * E * H * 4 * 2 if sd['env_kind'] == 2 else 0)) + 4 * (3 + S - 1)
        e2e_api = 'promp_b200.meta_trainer.Trainer.train_iteration(log=True), reset_mode=numpy'
    # the same iteration WITHOUT graph replay: Trainer.train_iteration(log=True), what configurations with a host decision
    # inside the iteration get (adaptive KL coefficient, early-terminating envs, E-MAML)
    np.random.seed(1)
    tr_eager = build_stack(wl, 'numpy', shard, use_cuda_graph=False)
    ms_e2e_eager, wall_e2e_eager, _ = timed(tr_eager, True, args.warmup, args.steps)

    # ---- the other BASELINE.json configurations, measured in the same run (short): HalfCheetah surrogate (configs[2] per GPU =
    #      configs[4] at N = 8, weak scaling) and TRPO-MAML on PointEnv (configs[3]: 40 tasks in total, STRONG scaling)
    extras = {}
    if not args.no_extras:
        def extra(key, wl_x, algo, tasks_per_gpu, scaling, n_steps):
            np.random.seed(1)
            tr = build_stack(wl_x, 'numpy', shard, algo=algo, tasks=tasks_per_gpu)
            ms, wall = timed_train(tr, 3, n_steps)
            n_env = tasks_per_gpu * world * wl_x['E'] * wl_x['H'] * 2
            wl_name = {'promp': wl_x['name'],
                       'promp_adaptive_kl': wl_x['name'] + ' with adaptive_inner_kl_penalty=True (the reference CLASS default, pro_mp.py:40; '
                                            'the run script sets False): halve / double rule applied on the device'}.get(
                algo, 'MAML-TRPO (maml_run_mujoco.py config: step_size 0.01, inner_type log_likelihood) on MetaPointEnvCorner, '
                      'meta_batch=40 in total (BASELINE.json configs[3])')
            extras[key] = dict(workload=wl_name,
                               algo=algo, scaling=scaling, tasks_per_gpu=tasks_per_gpu, tasks_total=tasks_per_gpu * world,
                               n_gpus=world, steps=n_steps, ms_per_step=ms / n_steps, wall_ms_per_step=wall / n_steps,
                               value=n_env * n_steps / (ms * 1e-3), unit='env-steps/s', meta_iters_per_sec=n_steps / (ms * 1e-3),
                               api='Trainer.train() (default entry point; e2e with host-drawn inputs and logged outputs)',
                               launch_mode='cuda_graph_replay' if tr.graph_capturable() else 'eager')
            if algo == 'trpo':
                extras[key]['last_step'] = {k: v for k, v in tr.algo.optimizer.last.items()}
        other = 'cheetah' if args.workload == 'point' else 'point'
        extra(other + '_promp_weak', WORKLOADS[other], 'promp', WORKLOADS[other]['M'], 'weak', max(5, args.steps // 2))
        if 40 % world == 0:
            extra('point_trpo_strong', WORKLOADS['point'], 'trpo', 40 // world, 'strong', max(3, args.steps // 4))
        if world == 1:
            extra('point_promp_adaptive_kl', WORKLOADS['point'], 'promp_adaptive_kl', WORKLOADS['point']['M'], 'weak', max(5, args.steps // 2))

    out = None
    # ---- per-kernel timing pass (instrumented, not part of the timed loops; every rank runs it because the
    #      iteration contains the all-reduce) --------------------------------------------------------------
    # stand-alone launches of the policy kernels here (promp_policy_chain would time a whole gradient chain as one unit; at this
    # size it launches the same kernels one after the other anyway - see promp_policy_chain_num_launches)
    tr_dev.algo.use_chain = False
    with LaunchCounter(time_kernels=True) as lk:
        for i in range(3):
            tr_dev.train_iteration(i, log=False)
        kms = lk.kernel_ms()
    barrier()
    if rank == 0:
        def _stat(name, v):
            # a launch that skipped itself (promp_policy_grad_ex launch re-use: the whole grid returns at once) is not a
            # sample of the kernel's duration: average over the launches that did the work, count the others separately
            v = np.asarray(v, dtype=np.float64)
            full = v[v > 0.25 * np.median(v)]
            if name == 'promp_policy_chain':
                # launches of different composition share the entry point (Adam epochs: grad + grad + HVP; first epoch with
                # the re-used inner pass; statistics pass: grad + values only): the roofline entry is the full epoch chain
                full = v[v > 0.85 * v.max()]
            return dict(launches_per_iter=len(v) // 3, avg_ms=float(np.mean(full)), total_ms_per_iter=float(np.sum(v) / 3),
                        skipped_launches_per_iter=float(len(v) - len(full)) / 3)
        per_kernel = {n: _stat(n, v) for n, v in kms.items()}
        peaks, peak_src = measured_peaks()
        N = E * H
        # dominant kernels: promp_policy_grad (13 launches / iteration) and promp_policy_hvp (5).  Algorithmic bytes per
        # launch (SURVEY.md section 8d "inner adapt / outer epoch" rows): obs + act + adv + old_mean per sample, once,
        # + per-task params (+ direction) and output.  Algorithmic FLOPs: the dense MLP chain (fwd + bwd [+ tangents]).
        P = _lib.load().promp_num_params(wl['Do'], wl['Da'], 64)
        Do_, Da_ = wl['Do'], wl['Da']
        alg = {
            'promp_policy_grad': dict(
                bytes=M * N * 4 * (Do_ + 2 * Da_ + 1),
                flops=M * N * (3 * 2 * 64 * 64 + 2 * 2 * Do_ * 64 + 3 * 2 * 64 * Da_),
                gemm_flops=M * N * 3 * 2 * 64 * 64, ncu='policy_grad'),
            'promp_policy_hvp': dict(
                bytes=M * N * 4 * (Do_ + 2 * Da_ + 1),
                flops=M * N * (8 * 2 * 64 * 64 + 6 * 2 * Do_ * 64 + 8 * 2 * 64 * Da_),
                gemm_flops=M * N * 8 * 2 * 64 * 64, ncu='policy_hvp'),
        }
        # the dataflow launch of one Adam epoch = inner gradient + outer gradient + HVP over the same per-sample bytes
        alg['promp_policy_chain'] = dict(
            bytes=2 * alg['promp_policy_grad']['bytes'] + alg['promp_policy_hvp']['bytes'],
            flops=2 * alg['promp_policy_grad']['flops'] + alg['promp_policy_hvp']['flops'],
            gemm_flops=2 * alg['promp_policy_grad']['gemm_flops'] + alg['promp_policy_hvp']['gemm_flops'], ncu='policy_chain')
        try:    # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture (tools/profile_all.sh)
            km_file = [f for f in ('r02_kernel_metrics.json', 'r01_kernel_metrics.json')
                       if os.path.exists(os.path.join(ROOT, 'profiles', f))][0]
            km = json.load(open(os.path.join(ROOT, 'profiles', km_file)))[args.workload]
        except Exception:
            km_file, km = None, {}
        iter_ms = max(sum(k['total_ms_per_iter'] for k in per_kernel.values()), 1e-9)
        fp32_peak = 148 * 128 * 2 * peaks.get('sm_max_mhz', 1965.0) * 1e6 / 1e12

        def kernel_roof(name):
            """The policy kernels are issue / latency-bound (AI ~ 1 kFLOP/B, inputs L2-resident): `frac` is the compute-side
            fraction (algorithmic fp32 FLOP/s over the fp32-SIMT peak 148 SM x 128 lanes x 2 x f_max); the HBM view
            (SURVEY.md section 8d bytes per sample x samples / launch time over the measured copy bandwidth) sits beside it."""
            a_, pk = alg[name], per_kernel.get(name, {})
            ms = pk.get('avg_ms', float('nan'))
            tfl = a_['flops'] / (ms * 1e-3) / 1e12
            gbs = a_['bytes'] / (ms * 1e-3) / 1e9
            kk = [k for k in km if k.startswith(a_['ncu'])]
            traffic = (km[kk[0]].get('dram_read_bytes', 0.0) + km[kk[0]].get('dram_write_bytes', 0.0)) if kk else None
            return dict(kernel=(kk[0] if kk else a_['ncu'] + '_kernel'), bound='issue', achieved=tfl, peak=fp32_peak, unit='TFLOP/s',
                        frac=tfl / fp32_peak, peak_source='derived: 148 SM x 128 fp32 lanes x 2 x sm_max_mhz (no measured fp32 peak in MEASURED_PEAKS.json)',
                        traffic=traffic,
                        traffic_source=('profiles/%s (cold-cache ncu replay; in the live loop the inputs are L2 hits)' % km_file) if kk else None,
                        hbm={'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'], 'peak_source': peak_src,
                             'algorithmic_bytes_per_launch': a_['bytes'],
                             'bytes_rule': 'SURVEY.md 8(d): 4*(Do+2*Da+1) B per sample per pass x M*N samples (x 3 passes for the epoch chain)'},
                        algorithmic_flops_per_launch=a_['flops'], avg_launch_ms=ms,
                        launches_per_iter=pk.get('launches_per_iter'), share_of_iteration=pk.get('total_ms_per_iter', 0.0) / iter_ms,
                        tensor={'executed_tf32_tflops': 3 * a_['gemm_flops'] / (ms * 1e-3) / 1e12,
                                'peak_bf16_tflops': peaks.get('bf16_tflops'),
                                'note': 'layer GEMMs run as 3xTF32 tcgen05.mma (weight gradients: mma.sync); 3 MMAs per algorithmic GEMM'})
        dom = max(alg, key=lambda n: per_kernel.get(n, {}).get('total_ms_per_iter', 0.0))
        roof = kernel_roof(dom)
        roof['note'] = ('arithmetic intensity ~ %d FLOP/B with everything L2/smem resident: neither HBM- nor tensor-peak-bound; the kernel is '
                        'issue/latency-bound at 1 CTA/SM (see DESIGN.md section 3 phase table); the HBM fraction (roofline.hbm) is small by construction'
                        % (alg[dom]['flops'] / alg[dom]['bytes']))
        others = [n for n in alg if n != dom and n in per_kernel]
        if others:
            roof['other_policy_kernel'] = kernel_roof(others[0])
        # HBM-bound scan kernel for reference: promp_process_samples reads obs twice + rew twice, writes ret + adv
        proc_bytes = M * N * (8 + 4 * (wl['Do'] + 1) + 4 * (wl['Do'] + 2) + 12)
        proc_ms = per_kernel.get('promp_process_samples', {}).get('avg_ms', float('nan'))
        roof['process_kernel'] = dict(kernel='process_fused_kernel', bound='hbm', unit='GB/s', peak=peaks['hbm_gbs'],
                                      achieved=proc_bytes / (proc_ms * 1e-3) / 1e9, frac=proc_bytes / (proc_ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
                                      algorithmic_bytes_per_launch=proc_bytes, avg_launch_ms=proc_ms,
                                      bytes_rule='SURVEY.md 8(d): returns 8 + Gram 4*(Do+1) + predict/GAE 4*(Do+2) + normalise 12 B per env-step',
                                      note='2.5-20 MB per launch: latency-bound (one short wave), far from the bandwidth roof by size')
        ro_bytes = M * N * (4 * (wl['Do'] + 2 * wl['Da'] + 1) + 1 + (8 if wl['Da'] == 6 else 0))
        ro_ms = per_kernel.get('promp_rollout', {}).get('avg_ms', float('nan'))
        roof['rollout_kernel'] = dict(achieved=ro_bytes / (ro_ms * 1e-3) / 1e9, frac=ro_bytes / (ro_ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
                                      algorithmic_bytes_per_launch=ro_bytes, avg_launch_ms=ro_ms,
                                      env_steps_per_s=M * N / (ro_ms * 1e-3))
        cpu = None
        if not args.no_cpu_baseline and world == 1:       # the CPU baseline is reported at N = 1 only (rank 0)
            # a separate process: the CPU arm forks worker processes, which must not inherit this process's CUDA context
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--workload', args.workload,
                                    '--steps', '2', '--warmup', '1'], capture_output=True, text=True, timeout=300,
                                   env=dict(os.environ, CUDA_VISIBLE_DEVICES='', RANK='0', WORLD_SIZE='1'))
                cpu = json.loads(r.stdout.strip().splitlines()[-1])['cpu_baseline']
            except Exception as e:      # keep the bench line: fall back to the in-process single-worker port
                sys.stderr.write('cpu_baseline subprocess failed (%r); single-process fallback\n' % (e,))
                cpu = run_cpu_baseline(wl, steps=2, warmup=1, m_sample=10, parallel=False)
        value = steps_per_iter * args.steps / (ms_dev * 1e-3)
        e2e_val = steps_per_iter * args.steps / (ms_e2e * 1e-3)
        out = {
            'metric': 'env_steps_per_sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'tasks_per_gpu': M, 'envs_per_task': E, 'max_path_length': H,
                       'algo': 'ProMP num_promp_steps=5 inner_lr=0.1 lr=1e-3 clip_eps=0.3 (pro-mp_run_point_mass.py defaults)',
                       'step_definition': 'one full meta-iteration (2 sampling+processing phases, inner adapt, 5 Adam epochs + stats pass)',
                       'parallelism': 'task-sharded dp%d, one all-reduce of the flat meta-gradient per Adam epoch (P2P peer-memory kernel over NVLink, inside the CUDA graph)' % world,
                       'l2_note': 'every iteration rewrites all trajectory buffers from fresh rollouts (inputs are produced, not re-read); no L2 flush needed'},
            'meta_iters_per_sec': world * 0 + args.steps / (ms_dev * 1e-3),
            'wall_ms_per_step': wall_dev / args.steps,
            'launch_mode': 'cuda_graph_replay' if use_graph else 'eager', 'eager_ms_per_step': ms_eager / args.steps,
            'e2e': {'value': e2e_val, 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': ms_e2e / args.steps, 'wall_ms_per_step': wall_e2e / args.steps,
                    'api': e2e_api,
                    'eager': {'value': steps_per_iter * args.steps / (ms_e2e_eager * 1e-3), 'ms_per_step': ms_e2e_eager / args.steps,
                              'wall_ms_per_step': wall_e2e_eager / args.steps,
                              'api': 'Trainer(use_cuda_graph=False).train_iteration(itr, log=True): ~35 kernel launches per iteration '
                                     'issued one by one, a D2H read of the logged statistics per sampling phase'}},
            'other_configs': extras,
            'gpu_launches': launches * args.steps, 'gpu_launches_per_step': launches,
            'clocks': clk, 'roofline': roof, 'kernels': per_kernel, 'cpu_baseline': cpu,
        }
    if world > 1:
        p2p.check()
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out))


# ------------------------------------------------------------------------------------------- CPU arm
def pick_torch_threads(fn):
    """The CPU stand-in for TF1's executor is sensitive to the thread count (BASELINE.md section 2):
    sweep and keep the fastest."""
    import torch
    best, best_t = None, None
    cands = sorted(set([1, 2, 4, 8, os.cpu_count() or 1]))
    for nt in cands:
        if nt > (os.cpu_count() or 1):
            continue
        torch.set_num_threads(nt)
        t = time.perf_counter()
        fn()
        dt = time.perf_counter() - t
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def cpu_meta_iteration(wl, m_sample, state):
    """One meta-iteration of the reference algorithm on the CPU (oracle port), m_sample tasks."""
    import torch
    from oracle import numpy_half as nh, tf_half as th, cheetah_surrogate as cs
    Do, Da, E, H = wl['Do'], wl['Da'], wl['E'], wl['H']
    dims = (Do, Da, (64, 64))
    if 'sampler' not in state:
        env = nh.NormalizedEnv(nh.PointEnvCorner() if wl['env'] == 'MetaPointEnvCorner' else cs.HalfCheetahRandDirecSurrogate())
        policy = th.OraclePolicy(m_sample, Do, Da)
        state.update(policy=policy, sampler=nh.Sampler(env, policy, E, m_sample, H),
                     proc=nh.SampleProcessor(nh.LinearFeatureBaseline(), 0.99, 1, True), adam=th.TF1Adam(policy.theta.size))
    policy, sampler, proc, adam = state['policy'], state['sampler'], state['proc'], state['adam']

    def to_phase(data):
        f = lambda a: torch.tensor(np.stack(a), dtype=torch.float32)
        return dict(obs=f([d['observations'] for d in data]), act=f([d['actions'] for d in data]),
                    adv=f([d['advantages'] for d in data]), mean=f([d['agent_infos']['mean'] for d in data]),
                    log_std=f([d['agent_infos']['log_std'] for d in data]))
    spans = {}
    t0 = time.perf_counter()
    sampler.update_tasks()
    policy.switch_to_pre_update()
    phases = []
    for step in range(2):
        t = time.perf_counter()
        paths = sampler.obtain_samples()
        spans['sampling'] = spans.get('sampling', 0) + time.perf_counter() - t
        t = time.perf_counter()
        data = proc.process_samples(paths)
        phases.append(to_phase(data))
        spans['sample_proc'] = spans.get('sample_proc', 0) + time.perf_counter() - t
        if step == 0:
            t = time.perf_counter()
            new = th.adapt(torch.tensor(policy.theta_tasks), phases[0], dims, PROMP['inner_lr'])
            policy.update_task_parameters(new.numpy())
            spans['inner_step'] = time.perf_counter() - t
    t = time.perf_counter()
    theta, _ = th.promp_optimize(torch.tensor(policy.theta), phases, dims, adam, PROMP['inner_lr'], PROMP['clip_eps'],
                                 [PROMP['init_inner_kl_penalty']], PROMP['num_ppo_steps'])
    policy.theta = theta.numpy()
    spans['outer_step'] = time.perf_counter() - t
    spans['itr'] = time.perf_counter() - t0
    return spans


# ---- multi-process numpy half: the reference's parallel=True runs one worker process per task (MetaParallelEnvExecutor,
#      samplers/vectorized_env_executor.py:88-202); here every worker owns a contiguous block of tasks and runs the oracle's
#      sampler + sample processor for them (policy forward included, so there is no per-step pipe traffic: a stronger CPU
#      arm than the reference's own layout).
_WORKER = {}


def _cpu_worker_phase(job):
    wl_key, goals, theta_tasks, pre_update, seed = job
    import warnings
    warnings.filterwarnings('ignore')
    from oracle import numpy_half as nh, tf_half as th, cheetah_surrogate as cs
    wl = WORKLOADS[wl_key]
    m_sub = len(goals)
    key = (wl_key, m_sub)
    if key not in _WORKER:
        try:
            import torch
            torch.set_num_threads(1)
        except Exception:
            pass
        env = nh.NormalizedEnv(nh.PointEnvCorner() if wl['env'] == 'MetaPointEnvCorner' else cs.HalfCheetahRandDirecSurrogate())
        policy = th.OraclePolicy(m_sub, wl['Do'], wl['Da'])
        _WORKER[key] = (policy, nh.Sampler(env, policy, wl['E'], m_sub, wl['H']),
                        nh.SampleProcessor(nh.LinearFeatureBaseline(), 0.99, 1, True))
    policy, sampler, proc = _WORKER[key]
    np.random.seed(seed)
    sampler.vec_env.set_tasks(list(goals))
    if pre_update:
        policy.theta = np.asarray(theta_tasks[0], dtype=np.float32)
        policy.switch_to_pre_update()
    else:
        policy.update_task_parameters(np.asarray(theta_tasks, dtype=np.float32))
    data = proc.process_samples(sampler.obtain_samples())
    f = lambda a: np.stack(a).astype(np.float32)
    return dict(obs=f([d['observations'] for d in data]), act=f([d['actions'] for d in data]),
                adv=f([d['advantages'] for d in data]), mean=f([d['agent_infos']['mean'] for d in data]),
                log_std=f([d['agent_infos']['log_std'] for d in data]))


def cpu_meta_iteration_parallel(wl_key, m_sample, state, pool, n_workers):
    """One meta-iteration on the CPU with the numpy half sharded over `n_workers` processes."""
    import torch
    from oracle import numpy_half as nh, tf_half as th, cheetah_surrogate as cs
    wl = WORKLOADS[wl_key]
    dims = (wl['Do'], wl['Da'], (64, 64))
    if 'theta' not in state:
        env = nh.PointEnvCorner() if wl['env'] == 'MetaPointEnvCorner' else cs.HalfCheetahRandDirecSurrogate()
        state.update(env=env, theta=th.init_params(*dims), adam=th.TF1Adam(th.num_params(*dims)), itr=0)
    env, adam = state['env'], state['adam']
    chunks = np.array_split(np.arange(m_sample), n_workers)
    chunks = [c for c in chunks if len(c)]
    spans = {}
    t0 = time.perf_counter()
    tasks = env.sample_tasks(m_sample)
    theta = np.asarray(state['theta'], dtype=np.float32)
    theta_tasks = np.tile(theta, (m_sample, 1))
    phases = []
    for step in range(2):
        t = time.perf_counter()
        jobs = [(wl_key, [tasks[i] for i in c], theta_tasks[c], step == 0, 1000003 * state['itr'] + 7919 * step + int(c[0]) + 1)
                for c in chunks]
        parts = pool.map(_cpu_worker_phase, jobs)
        phases.append({k: torch.from_numpy(np.concatenate([p[k] for p in parts])) for k in parts[0]})
        spans['sampling'] = spans.get('sampling', 0) + time.perf_counter() - t       # sampling + sample processing + IPC
        if step == 0:
            t = time.perf_counter()
            theta_tasks = th.adapt(torch.from_numpy(theta_tasks), phases[0], dims, PROMP['inner_lr']).numpy()
            spans['inner_step'] = time.perf_counter() - t
    t = time.perf_counter()
    new_theta, _ = th.promp_optimize(torch.from_numpy(theta), phases, dims, adam, PROMP['inner_lr'], PROMP['clip_eps'],
                                     [PROMP['init_inner_kl_penalty']], PROMP['num_ppo_steps'])
    state['theta'] = new_theta.numpy()
    state['itr'] += 1
    spans['outer_step'] = time.perf_counter() - t
    spans['sample_proc'] = 0.0
    spans['itr'] = time.perf_counter() - t0
    return spans


def run_cpu_baseline(wl, steps, warmup, m_sample, parallel=True, n_tasks=None):
    """CPU arm: the oracle port of the reference's path on this box's host cores.  parallel=True: the numpy half runs in
    min(tasks, cores) worker processes (like the reference's parallel=True executor), the TF1 half (PyTorch-CPU) with the
    fastest thread count; the whole M-task workload is timed.  parallel=False: single process, `m_sample` tasks."""
    import torch
    import warnings
    warnings.filterwarnings('ignore')
    wl_key = [k for k, v in WORKLOADS.items() if v is wl][0]
    cores = os.cpu_count() or 1
    pool, n_workers = None, 1
    if parallel and cores > 1:
        import multiprocessing as mp
        m_sample = wl['M'] if n_tasks is None else n_tasks        # like for like with an N-GPU run: 40*N tasks
        n_workers = max(1, min(m_sample, cores))
        pool = mp.get_context('fork').Pool(n_workers)        # forked BEFORE the parent touches torch's thread pool
    try:
        state = {}
        np.random.seed(1)
        # choose the torch thread count on a gradient evaluation of the right shape
        from oracle import tf_half as th
        dims = (wl['Do'], wl['Da'], (64, 64))
        N = wl['E'] * wl['H']
        g = torch.Generator().manual_seed(0)
        fake = dict(obs=torch.randn(m_sample, N, wl['Do'], generator=g), act=torch.randn(m_sample, N, wl['Da'], generator=g),
                    adv=torch.randn(m_sample, N, generator=g), mean=torch.randn(m_sample, N, wl['Da'], generator=g),
                    log_std=torch.zeros(m_sample, N, wl['Da']))
        theta = torch.tensor(th.init_params(*dims))

        def probe():
            t = theta.clone().requires_grad_(True)
            obj, _, _ = th.meta_objective(t, [fake, fake], dims, 0.1, 'promp', 0.3, [5e-4])
            torch.autograd.grad(obj, t)
        nthreads = pick_torch_threads(probe)
        if pool is not None:
            run = lambda: cpu_meta_iteration_parallel(wl_key, m_sample, state, pool, n_workers)
        else:
            run = lambda: cpu_meta_iteration(wl, m_sample, state)
        for _ in range(warmup):
            run()
        all_spans = [run() for _ in range(steps)]
    finally:
        if pool is not None:
            pool.close()
            pool.join()
    itr = float(np.median([s['itr'] for s in all_spans]))
    steps_per_iter = m_sample * wl['E'] * wl['H'] * 2
    med = {k: float(np.median([s[k] for s in all_spans])) for k in all_spans[0]}
    if pool is not None:
        sample = ('all %d tasks x %d envs x H=%d, full meta-iteration; numpy half (per-env Python stepping like the reference, '
                  'sampling + sample processing) sharded over %d worker processes, TF1 half = PyTorch-CPU restatement batched over '
                  'tasks with %d threads; median of %d' % (m_sample, wl['E'], wl['H'], n_workers, nthreads, steps))
    else:
        sample = ('%d of %d tasks x %d envs x H=%d, full meta-iteration (tasks are independent; numpy half = per-env Python '
                  'stepping like the reference, TF1 half = PyTorch-CPU restatement batched over tasks), median of %d'
                  % (m_sample, wl['M'], wl['E'], wl['H'], steps))
    return dict(value=steps_per_iter / itr, unit='env-steps/s', cores=max(n_workers, nthreads), host_cores=cores, worker_processes=n_workers,
                torch_threads=nthreads, kind='port', sample=sample, sec_per_iter=itr, spans_sec=med,
                sampling_env_steps_per_sec=steps_per_iter / med['sampling'])


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port) on this box's cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    world = int(os.environ.get('WORLD_SIZE', '1'))
    # the GPU arm is weak-scaled (wl['M'] tasks per GPU): the CPU arm gets the same wl['M'] * N tasks, on min(tasks, cores) workers
    cpu = run_cpu_baseline(wl, steps=args.steps, warmup=args.warmup, m_sample=10, parallel=not args.cpu_serial,
                           n_tasks=wl['M'] * world)
    out = {
        'impl': 'reference', 'metric': 'env_steps_per_sec', 'value': cpu['value'], 'unit': 'env-steps/s',
        'n_gpus': int(os.environ.get('WORLD_SIZE', '1')), 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': cpu['sec_per_iter'] * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 (TF half) / f64 (numpy half)', 'data': 'synthetic',
        'config': {'workload': wl['name'], 'tasks_total': wl['M'] * world, 'sample': cpu['sample'],
                   'note': 'reference = jonasrothfuss/ProMP CPU path; /root/reference and TF1 are absent on the GPU box, so the '
                           'oracle port (pinned to the reference by tests/golden) is what runs'},
        'cpu_baseline': cpu,
        'e2e': {'value': cpu['value'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='promp_b200', choices=['promp_b200', 'reference'])
    ap.add_argument('--workload', default='point', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the short cheetah / TRPO-MAML measurements (other_configs)')
    ap.add_argument('--cpu-serial', action='store_true', help='CPU arm: single process on a 10-task sample instead of one worker process per task')
    ap.add_argument('--no-graph', action='store_true', help='time the device-resident loop eagerly instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed meta-iteration computed as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl != 'reference' else max(args.warmup, 1)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
