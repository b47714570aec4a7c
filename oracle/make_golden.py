"""Generate tests/golden/*.npz by running the UNMODIFIED reference numpy half.

Runs only in the build container (needs /root/reference, which is read-only and absent on the GPU
box).  The reference modules are imported from where they lie, with the stub packages in
oracle/stubs standing in for gym / pyprind / rand_param_envs (absent, no network).  Nothing from
the reference is copied: only its numeric outputs are stored.

    python oracle/make_golden.py          # rewrites tests/golden/
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = '/root/reference'
OUT = os.path.join(ROOT, 'tests', 'golden')


def _import_reference():
    if not os.path.isdir(REF):
        raise SystemExit("reference tree %s not present: golden vectors can only be regenerated in the build container" % REF)
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'stubs'))
    sys.path.insert(0, REF)
    sys.path.insert(0, ROOT)


def gen_point_corner_steps():
    """normalize(MetaPointEnvCorner).step over scripted actions for the three reward types."""
    from meta_policy_search.envs.point_envs.point_env_2d_corner import MetaPointEnvCorner
    from meta_policy_search.envs.normalized_env import normalize
    out = {}
    T, n_env = 60, 24
    rng = np.random.RandomState(7)
    # policy-space actions in [-10,10]-ish, biased toward a random corner so that the sparse
    # reward's three branches (inside radius / goal is nearest corner / other corner) all occur
    drift = rng.choice([-1.0, 1.0], size=(n_env, 2)) * 4.0
    actions = drift[None] + 6.0 * rng.randn(T, n_env, 2)
    actions[::7] *= 3.0          # exercise the clip at the action bounds
    out['actions'] = actions
    for rtype in ('sparse', 'dense', 'dense_squared'):
        env = normalize(MetaPointEnvCorner(reward_type=rtype))
        np.random.seed(11)
        tasks = env.sample_tasks(n_env)
        obs0 = np.zeros((n_env, 2))
        obs = np.zeros((T, n_env, 2))
        rew = np.zeros((T, n_env))
        import copy
        envs = [copy.deepcopy(env) for _ in range(n_env)]
        for i, e in enumerate(envs):
            e.set_task(tasks[i])
            obs0[i] = e.reset()
        for t in range(T):
            for i, e in enumerate(envs):
                o, r, d, info = e.step(actions[t, i])
                assert d is False and info == {}
                obs[t, i], rew[t, i] = o, r
        out['goals'] = np.asarray(tasks, dtype=np.float64)
        out['obs0'] = obs0
        out['next_obs_' + rtype] = obs
        out['rewards_' + rtype] = rew
    np.savez_compressed(os.path.join(OUT, 'point_corner_steps.npz'), **out)


def gen_point_env_steps():
    """MetaPointEnv (tests' PointEnv: origin goal, early done) under normalize."""
    from meta_policy_search.envs.point_envs.point_env_2d import MetaPointEnv
    from meta_policy_search.envs.normalized_env import normalize
    T, n_env = 80, 8
    np.random.seed(3)
    envs = [normalize(MetaPointEnv()) for _ in range(n_env)]
    obs0 = np.asarray([e.reset() for e in envs])
    obs = np.zeros((T, n_env, 2)); rew = np.zeros((T, n_env)); done = np.zeros((T, n_env), dtype=bool)
    acts = np.zeros((T, n_env, 2))
    cur = obs0.copy()
    for t in range(T):
        for i, e in enumerate(envs):
            a = -cur[i] * 100.0 / 2.0          # head to the origin (policy-space: a_env = a/100 -> clip 0.1)
            acts[t, i] = a
            o, r, d, _ = e.step(a)
            obs[t, i], rew[t, i], done[t, i] = o, r, d
            cur[i] = o
    np.savez_compressed(os.path.join(OUT, 'point_env_steps.npz'), obs0=obs0, actions=acts, next_obs=obs,
                        rewards=rew, dones=done)


def gen_process_samples():
    """MetaSampleProcessor + LinearFeatureBaseline on synthetic paths (several settings)."""
    from meta_policy_search.samplers.meta_sample_processor import MetaSampleProcessor
    from meta_policy_search.baselines.linear_baseline import LinearFeatureBaseline
    from collections import OrderedDict
    out = {}
    cases = dict(
        a=dict(M=3, E=4, H=20, Do=2, Da=2, discount=0.99, gae_lambda=1.0, normalize_adv=True, positive_adv=False),
        b=dict(M=2, E=5, H=33, Do=2, Da=2, discount=0.95, gae_lambda=0.9, normalize_adv=False, positive_adv=False),
        c=dict(M=2, E=6, H=25, Do=17, Da=6, discount=0.99, gae_lambda=0.97, normalize_adv=True, positive_adv=True),
        d=dict(M=4, E=20, H=100, Do=2, Da=2, discount=0.99, gae_lambda=1.0, normalize_adv=True, positive_adv=False),
        e=dict(M=2, E=20, H=200, Do=17, Da=6, discount=0.99, gae_lambda=1.0, normalize_adv=True, positive_adv=False),
    )
    for name, c in cases.items():
        rng = np.random.RandomState(ord(name) + 5)
        M, E, H, Do, Da = c['M'], c['E'], c['H'], c['Do'], c['Da']
        # float32-representable inputs (the CUDA path holds trajectories in float32)
        obs = np.cumsum(0.3 * rng.randn(M, E, H, Do), axis=2)
        if name == 'c':
            obs[0, 0, :5] *= 40.0        # exercise the +-10 feature clip
        obs = obs.astype(np.float32).astype(np.float64)
        act = rng.randn(M, E, H, Da).astype(np.float32).astype(np.float64)
        rew = (rng.randn(M, E, H) * (rng.rand(M, E, H) < 0.6)).astype(np.float32).astype(np.float64)
        mean = rng.randn(M, E, H, Da).astype(np.float32).astype(np.float64)
        log_std = np.tile(rng.randn(M, 1, 1, Da) * 0.1, (1, E, H, 1)).astype(np.float32).astype(np.float64)
        paths = OrderedDict()
        for m in range(M):
            paths[m] = [dict(observations=obs[m, e], actions=act[m, e], rewards=rew[m, e], env_infos={},
                             agent_infos=dict(mean=mean[m, e], log_std=log_std[m, e])) for e in range(E)]
        proc = MetaSampleProcessor(baseline=LinearFeatureBaseline(), discount=c['discount'], gae_lambda=c['gae_lambda'],
                                   normalize_adv=c['normalize_adv'], positive_adv=c['positive_adv'])
        # capture the per-task coefficients: the shared baseline is re-fitted inside the task loop
        coeffs = []
        orig_fit = proc.baseline.fit

        def fit_and_record(paths_, target_key='returns'):
            orig_fit(paths_, target_key=target_key)
            coeffs.append(np.array(proc.baseline._coeffs))
        proc.baseline.fit = fit_and_record
        data = proc.process_samples(paths, log=False)
        pre = 'case_%s_' % name
        for k, v in c.items():
            out[pre + 'cfg_' + k] = np.asarray(v)
        out[pre + 'obs'], out[pre + 'act'], out[pre + 'rew'] = obs.astype(np.float32), act.astype(np.float32), rew.astype(np.float32)
        out[pre + 'returns'] = np.stack([d['returns'] for d in data])
        out[pre + 'advantages'] = np.stack([d['advantages'] for d in data])
        out[pre + 'adj_avg_rewards'] = np.stack([d['adj_avg_rewards'] for d in data])
        if name == 'a':
            out[pre + 'observations_stacked'] = np.stack([d['observations'] for d in data]).astype(np.float32)
        out[pre + 'coeffs'] = np.stack(coeffs)
        assert len(data[0].keys()) == 8
    np.savez_compressed(os.path.join(OUT, 'process_samples.npz'), **out)


def gen_point_variants_steps():
    """MetaPointEnvWalls (dense / dense_squared) and MetaPointEnvMomentum (three reward types) under normalize:
    seeded tasks (pins the RNG order of sample_tasks), resets and closed-loop steps under a random walk that is
    strong enough to hit both walls."""
    import copy
    from meta_policy_search.envs.point_envs.point_env_2d_walls import MetaPointEnvWalls
    from meta_policy_search.envs.point_envs.point_env_2d_momentum import MetaPointEnvMomentum
    from meta_policy_search.envs.normalized_env import normalize
    out = {}
    T, n_env = 150, 12
    rng = np.random.RandomState(21)
    drift = rng.randn(1, n_env, 2) * 4.0                          # per-env outward drift so that the walls get crossed
    actions = (drift + 6.0 * rng.randn(T, n_env, 2)).astype(np.float32).astype(np.float64)
    out['walls_actions'] = actions
    for rtype in ('dense', 'dense_squared'):
        env = normalize(MetaPointEnvWalls(reward_type=rtype))
        np.random.seed(17)
        tasks = env.sample_tasks(n_env)
        envs = [copy.deepcopy(env) for _ in range(n_env)]
        obs0 = np.zeros((n_env, 2)); obs = np.zeros((T, n_env, 2)); rew = np.zeros((T, n_env))
        for i, e in enumerate(envs):
            e.set_task(tasks[i])
            obs0[i] = e.reset()
        for t in range(T):
            for i, e in enumerate(envs):
                o, r, d, info = e.step(actions[t, i])
                assert d is False and info == {}
                obs[t, i], rew[t, i] = o, r
        out['walls_tasks'] = np.stack([np.concatenate([tk['goal'], tk['gap_1'], tk['gap_2']]) for tk in tasks]).astype(np.float64)
        out['walls_obs0'] = obs0
        out['walls_next_obs_' + rtype] = obs
        out['walls_rewards_' + rtype] = rew
    out['walls_rng_probe_after'] = np.random.uniform(size=3)
    T2 = 60
    actions = (3.0 * rng.randn(T2, n_env, 2)).astype(np.float32).astype(np.float64)
    out['momentum_actions'] = actions
    for rtype in ('sparse', 'dense', 'dense_squared'):
        env = normalize(MetaPointEnvMomentum(reward_type=rtype))
        np.random.seed(19)
        tasks = env.sample_tasks(n_env)
        envs = [copy.deepcopy(env) for _ in range(n_env)]
        obs0 = np.zeros((n_env, 4)); obs = np.zeros((T2, n_env, 4)); rew = np.zeros((T2, n_env))
        for i, e in enumerate(envs):
            e.set_task(tasks[i])
            obs0[i] = e.reset()
        for t in range(T2):
            for i, e in enumerate(envs):
                o, r, d, info = e.step(actions[t, i])
                assert d is False and info == {}
                obs[t, i], rew[t, i] = o, r
        out['momentum_goals'] = np.asarray(tasks, dtype=np.float64)
        out['momentum_obs0'] = obs0
        out['momentum_next_obs_' + rtype] = obs
        out['momentum_rewards_' + rtype] = rew
    np.savez_compressed(os.path.join(OUT, 'point_variants_steps.npz'), **out)


def gen_tf_half_numpy_known():
    """The numpy-executable pieces of the reference's TF1 half (TensorFlow itself is absent; `import tensorflow` inside
    these modules is satisfied by the inert oracle/stubs_tf stand-in, which these functions never touch):
    DiagonalGaussian.kl / log_likelihood / entropy (policies/distributions/diagonal_gaussian.py:46-69, 111-127, 142-153)
    and conjugate_gradients (optimizers/conjugate_gradient_optimizer.py:325-354)."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'stubs_tf'))      # import-only TensorFlow stand-in (nothing of it is executed)
    from meta_policy_search.policies.distributions.diagonal_gaussian import DiagonalGaussian
    if not hasattr(np, 'cast'):          # removed in NumPy 2; the optimizer module evaluates np.cast['float32'](1e-5) at import
        class _Cast(dict):
            def __missing__(self, k):
                return lambda x: np.asarray(x, dtype=k)
        np.cast = _Cast()
    from meta_policy_search.optimizers.conjugate_gradient_optimizer import conjugate_gradients
    rng = np.random.RandomState(31)
    out = {}
    for Da, N in ((2, 257), (6, 140)):
        pre = 'dist%d_' % Da
        old_mean, new_mean = rng.randn(N, Da), rng.randn(N, Da)
        old_ls, new_ls = 0.3 * rng.randn(N, Da) - 0.5, 0.3 * rng.randn(N, Da) - 0.5
        new_ls[:5] = np.log(1e-6)                      # the clip floor of gaussian_mlp_policy.py:71
        x = old_mean + np.exp(old_ls) * rng.randn(N, Da)
        dist = DiagonalGaussian(Da)
        old, new = dict(mean=old_mean, log_std=old_ls), dict(mean=new_mean, log_std=new_ls)
        out[pre + 'old_mean'], out[pre + 'old_ls'], out[pre + 'new_mean'], out[pre + 'new_ls'], out[pre + 'x'] = \
            old_mean, old_ls, new_mean, new_ls, x
        out[pre + 'kl'] = dist.kl(old, new)
        out[pre + 'll_old'] = dist.log_likelihood(x, old)
        out[pre + 'll_new'] = dist.log_likelihood(x, new)
        out[pre + 'entropy'] = dist.entropy(new)
    n = 60
    A = rng.randn(n, n)
    A = (A @ A.T / n + 0.5 * np.eye(n)).astype(np.float32)
    b = rng.randn(n).astype(np.float32)
    out['cg_A'], out['cg_b'] = A, b
    out['cg_x10'] = conjugate_gradients(lambda p: A.dot(p), b, cg_iters=10)
    out['cg_x3'] = conjugate_gradients(lambda p: A.dot(p), b, cg_iters=3)
    out['cg_x_tol'] = conjugate_gradients(lambda p: A.dot(p), b, cg_iters=200, residual_tol=1e-6)
    # adaptive inner-KL penalty rule (meta_algos/pro_mp.py:201-214), incl. the exact thresholds
    from meta_policy_search.meta_algos.pro_mp import _adapt_kl_coeff
    target = 0.01
    kls = np.concatenate([rng.uniform(0.0, 0.03, size=40), [target / 1.5, target * 1.5, 0.0, target]])
    coeffs = np.concatenate([rng.uniform(1e-4, 1e-2, size=40), [5e-4, 5e-4, 5e-4, 5e-4]])
    out['klc_target'], out['klc_kl'], out['klc_in'] = np.asarray(target), kls, coeffs
    out['klc_out'] = np.asarray([_adapt_kl_coeff(float(c), float(k), target) for c, k in zip(coeffs, kls)])
    np.savez_compressed(os.path.join(OUT, 'tf_half_known.npz'), **out)



def _np_cast_shim():
    if not hasattr(np, 'cast'):          # removed in NumPy 2; the optimizer module evaluates np.cast['float32'](1e-5) at import
        class _Cast(dict):
            def __missing__(self, k):
                return lambda x: np.asarray(x, dtype=k)
        np.cast = _Cast()


def _build_reference_algo(case, torch_dtype):
    """UNMODIFIED reference policy + algorithm graph for one oracle/tf_cases.py case, on the torch-backed tensorflow
    stand-in.  Returns (tf, sess, policy, algo)."""
    import tensorflow as tf
    from oracle import tf_cases
    from meta_policy_search.policies.meta_gaussian_mlp_policy import MetaGaussianMLPPolicy
    from meta_policy_search.meta_algos.pro_mp import ProMP
    from meta_policy_search.meta_algos.trpo_maml import TRPOMAML
    from meta_policy_search.meta_algos.vpg_maml import VPGMAML
    H = tf_cases.HYPER
    tf.reset_default_graph()
    tf.set_compute_dtype(torch_dtype)
    M = case['M']
    policy = MetaGaussianMLPPolicy(name='meta-policy', obs_dim=case['Do'], action_dim=case['Da'], meta_batch_size=M,
                                   hidden_sizes=(case['hidden'], case['hidden']))
    S1 = case['S'] - 1
    if case['algo'] == 'promp':
        algo = ProMP(policy=policy, inner_lr=H['inner_lr'], meta_batch_size=M, num_inner_grad_steps=S1,
                     learning_rate=H['learning_rate'], num_ppo_steps=H['num_ppo_steps'], clip_eps=H['clip_eps'],
                     target_inner_step=0.01, init_inner_kl_penalty=H['init_inner_kl_penalty'], adaptive_inner_kl_penalty=False)
    elif case['algo'] == 'trpo':
        algo = TRPOMAML(policy=policy, step_size=H['step_size'], inner_type=case['inner_type'], inner_lr=H['inner_lr'],
                        meta_batch_size=M, num_inner_grad_steps=S1, exploration=case.get('exploration', False))
    else:
        algo = VPGMAML(policy=policy, learning_rate=H['learning_rate'], inner_type=case['inner_type'], inner_lr=H['inner_lr'],
                       meta_batch_size=M, num_inner_grad_steps=S1, exploration=case.get('exploration', False))
    sess = tf.Session()
    sess.__enter__()
    uninit = [v for v in tf.global_variables() if not sess.run(tf.is_variable_initialized(v))]     # meta_trainer.py:75-76
    sess.run(tf.variables_initializer(uninit))
    policy.set_params(tf_cases.unflatten(case['theta'], case['Do'], case['Da'], case['hidden']))
    return tf, sess, policy, algo


def gen_tf_half_graph(only=None):
    """Golden OUTPUTS of the reference's TF1 graph half, produced by running its UNMODIFIED graph-building code
    (policies/*, meta_algos/{base,pro_mp,trpo_maml,vpg_maml}.py, optimizers/*) on the torch-backed `tensorflow`
    stand-in (oracle/stubs_tf): inner adapt step, meta-objective, inner / outer KL, second-order meta-gradient,
    the K-epoch TF1-Adam trajectory end point, TRPO-MAML loss / constraint gradients, finite-difference Hx, CG direction
    and accepted step.  Each case is evaluated twice: float32 (the reference's dtype) and float64 (same graph, no rounding).
    Inputs come from oracle/tf_cases.py seeds and are not stored."""
    import torch
    torch.set_num_threads(1)          # many tiny ops: intra-op threading only adds synchronisation cost
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'stubs_tf'))
    _np_cast_shim()
    from oracle import tf_cases
    from meta_policy_search.utils import logger
    from meta_policy_search.optimizers.conjugate_gradient_optimizer import conjugate_gradients
    logger.set_level(logger.DISABLED) if hasattr(logger, 'set_level') else None
    path = os.path.join(OUT, 'tf_half_graph.npz')
    out = dict(np.load(path)) if (only and os.path.exists(path)) else {}
    for name in tf_cases.CASES:
        if only and name not in only:
            continue
        case = tf_cases.make_case(name)
        samples = tf_cases.reference_samples(case)
        M, P, big = case['M'], case['P'], case['M'] >= 40
        keep_tasks = [0, 13, M - 1] if big else list(range(M))
        for tag, tdt in (('f32', torch.float32), ('f64', torch.float64)):
            pre = '%s/%s/' % (name, tag)
            tf, sess, policy, algo = _build_reference_algo(case, tdt)
            try:
                flat = lambda od: np.concatenate([np.asarray(v, dtype=np.float64).reshape(-1) for v in od.values()])
                # ---- inner adapt steps (meta_algos/base.py:217-242), from the pre-update parameters
                policy.switch_to_pre_update()
                for s in range(case['S'] - 1):
                    algo._adapt(samples[s])
                    tp = np.stack([flat(od) for od in policy.policies_params_vals])            # [M, P]
                    delta = tp - case['theta'].astype(np.float64)[None]
                    out[pre + 'adapt%d_tasks' % s] = tp[keep_tasks]
                    out[pre + 'adapt%d_delta_sum' % s] = delta.sum(1)
                    out[pre + 'adapt%d_delta_norm' % s] = np.sqrt((delta ** 2).sum(1))
                out[name + '/keep_tasks'] = np.asarray(keep_tasks)
                # ---- outer objective / gradient at theta
                inp = algo._extract_input_dict_meta_op(samples, algo._optimization_keys)
                params = list(policy.get_params().values())
                opt = algo.optimizer
                if case['algo'] == 'promp':
                    inp['inner_kl_coeff'] = algo.inner_kl_coeff
                    inp['clip_eps'] = algo.clip_eps
                    feed = opt.create_feed_dict(inp)
                    loss, ikl, okl, grads = sess.run([opt._loss, opt._inner_kl, opt._outer_kl, tf.gradients(opt._loss, params)], feed)
                    out[pre + 'loss'], out[pre + 'inner_kl'], out[pre + 'outer_kl'] = np.float64(loss), np.asarray(ikl, np.float64), np.float64(okl)
                    out[pre + 'grad'] = np.concatenate([np.asarray(g, np.float64).reshape(-1) for g in grads])
                    algo.optimize_policy(samples, log=False)                                       # pro_mp.py:165-199, K = 5 epochs
                    out[pre + 'theta_after_adam5'] = flat(policy.get_param_values())
                    la, ikl2, okl2 = opt.compute_stats(inp)
                    out[pre + 'loss_after'], out[pre + 'inner_kl_after'], out[pre + 'outer_kl_after'] = \
                        np.float64(la), np.asarray(ikl2, np.float64), np.float64(okl2)
                    if not big:
                        # first epoch alone (fresh graph = fresh Adam slots; only the epoch count of the optimizer changes)
                        sess.__exit__(None, None, None)
                        tf, sess, policy, algo = _build_reference_algo(case, tdt)
                        algo.optimizer._max_epochs = 1
                        algo.optimize_policy(samples, log=False)
                        out[pre + 'theta_after_adam1'] = flat(policy.get_param_values())
                elif case['algo'] == 'trpo':
                    out[pre + 'loss'] = np.float64(opt.loss(inp))
                    out[pre + 'outer_kl'] = np.float64(opt.constraint_val(inp))
                    g = opt.gradient(inp)
                    out[pre + 'grad'] = np.asarray(g, np.float64)
                    out[pre + 'kl_grad'] = np.asarray(opt._hvp_approach.constraint_gradient(inp), np.float64)
                    x = (g / (np.linalg.norm(g) + 1e-12)).astype(g.dtype)
                    out[pre + 'hx_dir'] = np.asarray(x, np.float64)
                    out[pre + 'hx'] = np.asarray(opt._hvp_approach.Hx(inp, x), np.float64)           # conjugate_gradient_optimizer.py:59-89
                    if not big or tag == 'f64':
                        Hx = opt._hvp_approach.build_eval(inp)
                        out[pre + 'cg_dir'] = np.asarray(conjugate_gradients(Hx, g, cg_iters=10), np.float64)
                    algo.optimize_policy(samples, log=False)                                         # trpo_maml.py:161-192
                    out[pre + 'theta_after'] = flat(policy.get_param_values())
                    out[pre + 'loss_after'] = np.float64(opt.loss(inp))
                    out[pre + 'kl_after'] = np.float64(opt.constraint_val(inp))
                else:
                    feed = opt.create_feed_dict(inp)
                    loss, grads = sess.run([opt._loss, tf.gradients(opt._loss, params)], feed)
                    out[pre + 'loss'] = np.float64(loss)
                    out[pre + 'grad'] = np.concatenate([np.asarray(g, np.float64).reshape(-1) for g in grads])
                    algo.optimize_policy(samples, log=False)                                         # vpg_maml.py:147-166 (1 Adam step)
                    out[pre + 'theta_after'] = flat(policy.get_param_values())
            finally:
                sess.__exit__(None, None, None)
            print('tf_half_graph', name, tag, 'done', flush=True)
        # values of the float32 evaluation are float32 numbers: store them as such
        out = {k: (v.astype(np.float32) if ('/f32/' in k and np.asarray(v).dtype == np.float64) else v) for k, v in out.items()}
        np.savez_compressed(path, **out)



def gen_trainer_run():
    """End-to-end pin: the UNMODIFIED reference Trainer (meta_trainer.py:59-152) driving the unmodified reference
    MetaSampler(parallel=False) / MetaSampleProcessor / LinearFeatureBaseline / MetaGaussianMLPPolicy / ProMP on
    normalize(MetaPointEnvCorner) at BASELINE.json configs[0] (5 tasks x 4 envs x H=100, run-script hyper-parameters)
    for 3 meta-iterations.  TensorFlow is the torch-backed stand-in (oracle/stubs_tf); its tf.random_normal draws are
    recorded so the CUDA path can be fed the same action noise.  Stored: theta_0, the noise, per-iteration goals,
    theta after every iteration and the logged scalars."""
    import torch
    torch.set_num_threads(1)
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'stubs_tf'))
    _np_cast_shim()
    import tensorflow as tf
    from oracle import tf_cases
    from meta_policy_search.baselines.linear_baseline import LinearFeatureBaseline
    from meta_policy_search.envs.point_envs.point_env_2d_corner import MetaPointEnvCorner
    from meta_policy_search.envs.normalized_env import normalize
    from meta_policy_search.meta_algos.pro_mp import ProMP
    from meta_policy_search.meta_trainer import Trainer
    from meta_policy_search.samplers.meta_sampler import MetaSampler
    from meta_policy_search.samplers.meta_sample_processor import MetaSampleProcessor
    from meta_policy_search.policies.meta_gaussian_mlp_policy import MetaGaussianMLPPolicy
    from meta_policy_search.utils import logger
    M, E, H, n_itr = 5, 4, 100, 3
    out = {}
    for rtype in ('sparse', 'dense'):
        tf.reset_default_graph()
        tf.set_compute_dtype(torch.float32)
        draws = []
        noise_rng = np.random.RandomState(77)

        def normal_hook(shape):
            a = noise_rng.standard_normal(shape).astype(np.float32)
            draws.append(a)
            return a
        tf.set_random_normal_hook(normal_hook)
        try:
            env = normalize(MetaPointEnvCorner(reward_type=rtype))
            baseline = LinearFeatureBaseline()
            policy = MetaGaussianMLPPolicy(name='meta-policy', obs_dim=2, action_dim=2, meta_batch_size=M, hidden_sizes=(64, 64))
            sampler = MetaSampler(env=env, policy=policy, rollouts_per_meta_task=E, meta_batch_size=M, max_path_length=H,
                                  parallel=False)
            proc = MetaSampleProcessor(baseline=baseline, discount=0.99, gae_lambda=1, normalize_adv=True)
            algo = ProMP(policy=policy, inner_lr=0.1, meta_batch_size=M, num_inner_grad_steps=1, learning_rate=1e-3,
                         num_ppo_steps=5, clip_eps=0.3, target_inner_step=0.01, init_inner_kl_penalty=5e-4,
                         adaptive_inner_kl_penalty=False)
            sess = tf.Session()
            with sess.as_default():
                sess.run(tf.global_variables_initializer())
                theta0 = tf_cases.make_case('promp_iter0')['theta']          # a fixed, seeded parameter vector (P = 4484)
                policy.set_params(tf_cases.unflatten(theta0, 2, 2, 64))
            thetas, kvs, goals = [], [], []
            flat = lambda od: np.concatenate([np.asarray(v, dtype=np.float64).reshape(-1) for v in od.values()])
            orig_opt, orig_update = algo.optimize_policy, sampler.update_tasks

            def optimize_and_record(*a, **k):
                orig_opt(*a, **k)
                thetas.append(flat(policy.get_param_values()))
                kvs.append({k_: float(v) for k_, v in logger.getkvs().items() if not k_.startswith('Time')})

            def update_and_record():
                orig_update()
                goals.append(np.asarray([e.get_task() for e in sampler.vec_env.envs[::E]], dtype=np.float64))
            algo.optimize_policy, sampler.update_tasks = optimize_and_record, update_and_record
            trainer = Trainer(algo=algo, env=env, sampler=sampler, sample_processor=proc, policy=policy, n_itr=n_itr,
                              num_inner_grad_steps=1, sess=sess)
            np.random.seed(1)
            trainer.train()
            rng_probe = np.random.uniform(size=4)
        finally:
            tf.set_random_normal_hook(None)
        # reassemble the recorded draws: per iteration, phase 0 (pre-update) = H draws of [M*E, Da];
        # phase 1 (post-update) = H x M draws of [E, Da] in task order
        noise = np.zeros((n_itr, 2, M, E, H, 2), np.float32)
        k = 0
        for it in range(n_itr):
            for t in range(H):
                noise[it, 0, :, :, t] = draws[k].reshape(M, E, 2); k += 1
            for t in range(H):
                for m in range(M):
                    noise[it, 1, m, :, t] = draws[k]; k += 1
        assert k == len(draws), (k, len(draws))
        pre = rtype + '_'
        out[pre + 'theta0'], out[pre + 'noise'], out[pre + 'goals'] = theta0, noise, np.stack(goals)
        out[pre + 'thetas'] = np.stack(thetas)
        keys = sorted(kvs[0])
        out[pre + 'log_keys'] = np.asarray(keys)
        out[pre + 'log_vals'] = np.asarray([[kv[k_] for k_ in keys] for kv in kvs])
        out[pre + 'rng_probe_after'] = rng_probe
    np.savez_compressed(os.path.join(OUT, 'trainer_run.npz'), **out)


def gen_process_samples_ragged():
    """MetaSampleProcessor + LinearFeatureBaseline on VARIABLE-LENGTH paths (early termination,
    meta_sampler.py:116-125): per task a different number of paths and samples.  Stored flat with offsets."""
    from meta_policy_search.samplers.meta_sample_processor import MetaSampleProcessor
    from meta_policy_search.baselines.linear_baseline import LinearFeatureBaseline
    from collections import OrderedDict
    out = {}
    cases = dict(
        r1=dict(M=3, Do=2, Da=2, discount=0.99, gae_lambda=1.0, normalize_adv=True, positive_adv=False,
                lens=[[5, 17, 1, 30, 12], [40, 3], [9, 9, 9, 25, 2, 2, 31]]),
        r2=dict(M=2, Do=17, Da=6, discount=0.95, gae_lambda=0.9, normalize_adv=True, positive_adv=True,
                lens=[[60, 45, 80, 100, 33], [100, 100, 7, 64]]),
        r3=dict(M=4, Do=2, Da=2, discount=0.99, gae_lambda=0.97, normalize_adv=False, positive_adv=False,
                lens=[[100] * 3, [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 50], [77], [20, 20, 20, 20, 20, 20]]),
    )
    for name, c in cases.items():
        rng = np.random.RandomState(sum(map(ord, name)))
        M, Do, Da = c['M'], c['Do'], c['Da']
        paths = OrderedDict()
        flat = dict(obs=[], act=[], rew=[], mean=[])
        log_std = (rng.randn(M, Da) * 0.1).astype(np.float32)
        for m in range(M):
            paths[m] = []
            for L in c['lens'][m]:
                obs = np.cumsum(0.3 * rng.randn(L, Do), axis=0).astype(np.float32).astype(np.float64)
                act = rng.randn(L, Da).astype(np.float32).astype(np.float64)
                rew = (rng.randn(L) * (rng.rand(L) < 0.7)).astype(np.float32).astype(np.float64)
                mean = rng.randn(L, Da).astype(np.float32).astype(np.float64)
                paths[m].append(dict(observations=obs, actions=act, rewards=rew, env_infos={},
                                     agent_infos=dict(mean=mean, log_std=np.tile(log_std[m].astype(np.float64), (L, 1)))))
                for k, v in (('obs', obs), ('act', act), ('rew', rew), ('mean', mean)):
                    flat[k].append(v.astype(np.float32))
        proc = MetaSampleProcessor(baseline=LinearFeatureBaseline(), discount=c['discount'], gae_lambda=c['gae_lambda'],
                                   normalize_adv=c['normalize_adv'], positive_adv=c['positive_adv'])
        coeffs = []
        orig_fit = proc.baseline.fit

        def fit_and_record(paths_, target_key='returns'):
            orig_fit(paths_, target_key=target_key)
            coeffs.append(np.array(proc.baseline._coeffs))
        proc.baseline.fit = fit_and_record
        data = proc.process_samples(paths, log=False)
        pre = 'case_%s_' % name
        for k in ('M', 'Do', 'Da', 'discount', 'gae_lambda', 'normalize_adv', 'positive_adv'):
            out[pre + 'cfg_' + k] = np.asarray(c[k])
        out[pre + 'n_paths'] = np.asarray([len(l) for l in c['lens']], dtype=np.int32)
        out[pre + 'path_len'] = np.concatenate([np.asarray(l, dtype=np.int32) for l in c['lens']])
        out[pre + 'log_std'] = log_std
        for k in flat:
            out[pre + k] = np.concatenate(flat[k])
        out[pre + 'returns'] = np.concatenate([d['returns'] for d in data])
        out[pre + 'advantages'] = np.concatenate([d['advantages'] for d in data])
        out[pre + 'observations_stacked'] = np.concatenate([d['observations'] for d in data]).astype(np.float32)
        out[pre + 'coeffs'] = np.stack(coeffs)
    np.savez_compressed(os.path.join(OUT, 'process_samples_ragged.npz'), **out)


def gen_sampler_rollout():
    """Reference MetaSampler(parallel=False) + normalize(MetaPointEnvCorner) driven by the oracle's
    numpy policy with injected action noise: pins RNG consumption order, index mapping, rollouts."""
    from meta_policy_search.samplers.meta_sampler import MetaSampler
    from meta_policy_search.envs.point_envs.point_env_2d_corner import MetaPointEnvCorner
    from meta_policy_search.envs.normalized_env import normalize
    from oracle.tf_half import OraclePolicy, init_params
    M, E, H = 5, 4, 100          # BASELINE.json configs[0]
    rng = np.random.RandomState(123)
    theta = init_params(2, 2, (64, 64), rng=rng)
    noise = rng.randn(2, H, M, E, 2).astype(np.float32)
    np.random.seed(1)
    env = normalize(MetaPointEnvCorner())
    out = dict(theta=theta, noise=noise)
    phase = [0]
    policy = OraclePolicy(M, 2, 2, theta=theta, noise=lambda t, shape: noise[phase[0], t])
    sampler = MetaSampler(env=env, policy=policy, rollouts_per_meta_task=E, meta_batch_size=M,
                          max_path_length=H, parallel=False)
    for it in range(2):
        sampler.update_tasks()
        goals = np.asarray([e.get_task() for e in sampler.vec_env.envs[::E]], dtype=np.float64)
        policy.switch_to_pre_update()
        phase[0] = it
        paths = sampler.obtain_samples()
        pre = 'it%d_' % it
        out[pre + 'goals'] = goals
        out[pre + 'obs'] = np.stack([np.stack([p['observations'] for p in paths[m]]) for m in range(M)])
        out[pre + 'act'] = np.stack([np.stack([p['actions'] for p in paths[m]]) for m in range(M)])
        out[pre + 'rew'] = np.stack([np.stack([p['rewards'] for p in paths[m]]) for m in range(M)])
        out[pre + 'mean'] = np.stack([np.stack([p['agent_infos']['mean'] for p in paths[m]]) for m in range(M)])
    out['rng_probe_after'] = np.random.uniform(size=4)     # pins how many draws were consumed
    np.savez_compressed(os.path.join(OUT, 'sampler_rollout.npz'), **out)


def gen_baseline_known():
    """discount_cumsum / feature matrix known answers straight from the reference utils."""
    from meta_policy_search.utils import utils
    from meta_policy_search.baselines.linear_baseline import LinearFeatureBaseline
    rng = np.random.RandomState(0)
    x = rng.randn(37)
    obs = rng.randn(9, 3) * 8
    b = LinearFeatureBaseline()
    np.savez_compressed(os.path.join(OUT, 'utils_known.npz'), x=x, dc_099=utils.discount_cumsum(x, 0.99),
                        dc_05=utils.discount_cumsum(x, 0.5), obs=obs, feats=b._features(dict(observations=obs)),
                        norm_adv=utils.normalize_advantages(x), pos_adv=utils.shift_advantages_to_positive(x))


def gen_stack_tensor_dict_list():
    """utils.stack_tensor_dict_list (utils/utils.py:144-159) on per-step info dicts with a nested dict: the trajectory
    bookkeeping of the stepwise sampler.  The inputs are re-drawn by the test from the same seed."""
    from meta_policy_search.utils import utils
    rng = np.random.RandomState(0)
    steps = [dict(mean=rng.randn(3), log_std=rng.randn(3), nested=dict(a=rng.randn(2), b=float(i))) for i in range(7)]
    got = utils.stack_tensor_dict_list(steps)
    np.savez_compressed(os.path.join(OUT, 'stack_tensor_dict_list.npz'), keys=np.asarray(sorted(got)),
                        nested_keys=np.asarray(sorted(got['nested'])), mean=got['mean'], log_std=got['log_std'],
                        nested_a=got['nested']['a'], nested_b=got['nested']['b'])


def gen_trainer_protocol():
    """What the UNMODIFIED reference Trainer (meta_trainer.py:59-152) asks of the objects it drives: the sequence of
    method calls it makes on recording doubles (2 iterations, 1 inner step), and the TensorFlow names it uses, with
    promp_b200/tf_shim imported as `tensorflow` (INTEGRATION.md section 1)."""
    import importlib.util
    import types
    spec = importlib.util.spec_from_file_location(
        'tensorflow', os.path.join(ROOT, 'promp_b200', 'tf_shim', 'tensorflow', '__init__.py'))
    shim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(shim)
    tf_used, session_used, calls = set(), set(), []

    class RecordingSession(shim.Session):
        def __getattribute__(self, k):
            if not k.startswith('_'):
                session_used.add(k)
            return object.__getattribute__(self, k)

    class RecordingTF(types.ModuleType):
        def __getattr__(self, k):
            tf_used.add(k)
            return RecordingSession if k == 'Session' else getattr(shim, k)

    class Rec(object):
        def __init__(self, name):
            self._n = name

        def __getattr__(self, k):
            def f(*a, **kw):
                calls.append(self._n + '.' + k)
                if k == 'obtain_samples':
                    return {0: [dict(x=1)], 1: [dict(x=2)]}
                if k == 'process_samples':
                    return ['samples']
                return None
            return f

    saved = {k: sys.modules.pop(k) for k in ('tensorflow', 'meta_policy_search.meta_trainer') if k in sys.modules}
    sys.modules['tensorflow'] = RecordingTF('tensorflow')
    try:
        from meta_policy_search.meta_trainer import Trainer
    finally:
        sys.modules.pop('tensorflow')
        sys.modules.pop('meta_policy_search.meta_trainer', None)
        sys.modules.update(saved)
    sampler = Rec('sampler')
    sampler.total_timesteps_sampled = 0
    proc = Rec('proc')
    proc.baseline = Rec('baseline')
    Trainer(algo=Rec('algo'), env=Rec('env'), sampler=sampler, sample_processor=proc, policy=Rec('policy'), n_itr=2,
            num_inner_grad_steps=1).train()
    np.savez_compressed(os.path.join(OUT, 'trainer_protocol.npz'), calls=np.asarray(calls),
                        tf_names=np.asarray(sorted(tf_used)), session_methods=np.asarray(sorted(session_used)))


if __name__ == '__main__':
    _import_reference()
    os.makedirs(OUT, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == 'tf_half_graph':      # python oracle/make_golden.py tf_half_graph [case ...]
        gen_tf_half_graph(only=sys.argv[2:] or None)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] in ('trainer_run', 'stack_tensor_dict_list', 'trainer_protocol'):
        globals()['gen_' + sys.argv[1]]()
        sys.exit(0)
    gen_point_corner_steps()
    gen_point_env_steps()
    gen_process_samples()
    gen_sampler_rollout()
    gen_baseline_known()
    gen_stack_tensor_dict_list()
    gen_trainer_protocol()
    gen_process_samples_ragged()
    gen_point_variants_steps()
    gen_tf_half_numpy_known()
    gen_tf_half_graph()
    gen_trainer_run()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
