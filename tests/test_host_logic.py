"""CPU tests: the C-ABI library loads and exports every symbol the header declares (no compute calls
without a GPU), host-side logic, the TF1-half oracle's own validation, the world_size-2 gloo path and
the reference's unchanged Trainer driving reference-shaped objects through the tf shim."""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_header_symbols():
    import __graft_entry__ as ge
    ge.build()
    from promp_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'promp_b200.h')).read()
    declared = set(re.findall(r'\b(promp_[a-z0-9_]+)\s*\(', header))
    declared -= {'promp_status'}
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    # pure host helpers (no kernel launch)
    assert lib.promp_num_params(2, 2, 64) == 4484 and lib.promp_num_params(17, 6, 64) == 5708
    assert lib.promp_env_state_dim(_lib.ENV_CHEETAH_DIR) == 18 and lib.promp_env_task_dim(_lib.ENV_POINT_CORNER) == 2
    assert lib.promp_version() >= 100
    assert lib.promp_process_workspace_bytes(40, 20, 100, 2) >= 40 * 2 * 2000 * 8
    # argument validation happens before any CUDA call
    assert lib.promp_reduce_tasks(0, 0, None, 1.0, None, None) == -1
    assert b'bad arguments' in lib.promp_last_error()


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from promp_b200 import _lib
    from promp_b200.policies import MetaGaussianMLPPolicy
    from promp_b200.envs import normalize, MetaPointEnvCorner
    from promp_b200.samplers import MetaDeviceEnvExecutor
    with pytest.raises(_lib.PrompLibraryError):
        MetaGaussianMLPPolicy(meta_batch_size=2, obs_dim=2, action_dim=2, hidden_sizes=(64, 64))
    with pytest.raises(_lib.PrompLibraryError):
        MetaDeviceEnvExecutor(normalize(MetaPointEnvCorner()), 2, 2, 10)
    with pytest.raises(_lib.PrompLibraryError):
        _lib.ptr(torch.zeros(3))


def test_env_host_side_matches_reference_rng_order():
    """Task / reset draws of the device env descriptions consume numpy exactly like the oracle's envs."""
    from promp_b200.envs import MetaPointEnvCorner, HalfCheetahRandDirecEnv, normalize
    from oracle import numpy_half as nh
    np.random.seed(5)
    a = MetaPointEnvCorner().sample_tasks(7)
    s = MetaPointEnvCorner().host_reset_states(6)
    np.random.seed(5)
    o = nh.PointEnvCorner()
    b = o.sample_tasks(7)
    r = np.stack([o.reset() for _ in range(6)])
    assert all(np.array_equal(x, y) for x, y in zip(a, b)) and np.array_equal(s, r)
    env = normalize(MetaPointEnvCorner('dense'))
    assert env.reward_type == 1 and env.device_spec()['normalized'] and env.action_space.low[0] == -10
    assert env.observation_space.shape == (2,) and HalfCheetahRandDirecEnv().device_spec()['state_dim'] == 18
    with pytest.raises(NotImplementedError):
        normalize(MetaPointEnvCorner(), normalize_obs=True)
    with pytest.raises(TypeError):
        normalize(object())


def test_adapt_kl_coeff_rule():
    from promp_b200.meta_algos.pro_mp import _adapt_kl_coeff
    from oracle.tf_half import adapt_kl_coeff
    assert _adapt_kl_coeff(1.0, 0.001, 0.01) == 0.5 and _adapt_kl_coeff(1.0, 0.02, 0.01) == 2.0
    assert _adapt_kl_coeff(1.0, 0.01, 0.01) == 1.0
    np.testing.assert_array_equal(adapt_kl_coeff([1.0, 1.0], [0.001, 0.1], 0.01), [0.5, 2.0])


def test_logger_and_lazy_containers():
    from promp_b200.utils import logger
    logger.set_quiet(True)
    logger.logkv('a', 1.0)
    logger.dumpkvs()
    assert logger.last_dump()['a'] == 1.0 and len(logger.getkvs()) == 0
    from promp_b200.samplers.device_data import SamplesData
    assert len(SamplesData(None, 0).keys()) == 8 and 'adj_avg_rewards' in SamplesData(None, 0)


# ------------------------------------------------------------------ the TF1-half oracle validates itself
@pytest.mark.parametrize('algo', ['promp', 'trpo'])
@pytest.mark.parametrize('inner', ['likelihood_ratio', 'log_likelihood'])
def test_tf_half_oracle_finite_differences(algo, inner):
    """fp64 central differences of the restated meta objective vs its autograd gradient (2 inner steps)."""
    import torch
    from oracle import tf_half as th
    torch.manual_seed(0)
    M, N, Do, Da = 3, 40, 2, 2
    dims = (Do, Da, (64, 64))
    theta = torch.tensor(th.init_params(*dims, rng=np.random.RandomState(0), dtype=np.float64))
    theta = theta + 0.05 * torch.randn_like(theta)

    def mk():
        obs = torch.randn(M, N, Do, dtype=torch.float64)
        mean, ls = th.dist_info(theta.unsqueeze(0).expand(M, -1), obs, dims)
        act = mean + torch.randn_like(mean) * torch.exp(ls)
        return dict(obs=obs, act=act, adv=torch.randn(M, N, dtype=torch.float64),
                    mean=(mean + 0.05 * torch.randn_like(mean)).detach(), log_std=(ls.expand_as(mean) + 0.02).detach().clone())
    data = [mk(), mk(), mk()]
    kw = dict(inner_type=inner) if algo == 'trpo' else {}
    t = theta.clone().requires_grad_(True)
    obj, ikl, okl = th.meta_objective(t, data, dims, 0.1, algo, 0.3, [5e-4, 1e-3], **kw)
    (g,) = torch.autograd.grad(obj, t)
    for seed in range(3):
        v = torch.randn(theta.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(seed))
        eps = 1e-6
        fp = th.meta_objective(theta + eps * v, data, dims, 0.1, algo, 0.3, [5e-4, 1e-3], **kw)[0]
        fm = th.meta_objective(theta - eps * v, data, dims, 0.1, algo, 0.3, [5e-4, 1e-3], **kw)[0]
        fd = float((fp - fm) / (2 * eps))
        assert abs(fd - float(g @ v)) < 1e-7 * max(1.0, abs(fd)), (fd, float(g @ v))


def test_tf_half_oracle_reference_identities():
    """Restated reference tests: likelihood ratio == 1 when pi_old == pi_new (tests/test_integration.py:150-175);
    get_actions' agent_infos == distribution info of the same observations (tests/test_policies.py:43-64)."""
    import torch
    from oracle import tf_half as th
    M, E, Do, Da = 4, 6, 2, 2
    pol = th.OraclePolicy(M, Do, Da, hidden_sizes=(16, 16))
    pol.switch_to_pre_update()
    obs = [np.random.randn(E, Do) for _ in range(M)]
    actions, infos = pol.get_actions(obs)
    mean, ls = th.dist_info(torch.tensor(pol.theta_tasks), torch.tensor(np.stack(obs), dtype=torch.float32), (Do, Da, (16, 16)),
                            min_log_std=math.log(1e-6))
    got = np.stack([[i['mean'] for i in task] for task in infos])
    np.testing.assert_allclose(got, mean.numpy(), rtol=1e-5, atol=1e-5)
    a = torch.tensor(np.stack(actions), dtype=torch.float32)
    lr = th.likelihood_ratio(a, mean, ls.expand_as(mean), mean, ls)
    assert np.allclose(lr.numpy(), 1)
    # TF1 Adam: first step moves every coordinate by lr * sign(g) (m/sqrt(v) = 1 up to eps)
    adam = th.TF1Adam(5)
    out = adam.step(torch.zeros(5), torch.tensor([1., -2., 3., -4., 5.]))
    np.testing.assert_allclose(out.numpy(), -1e-3 * np.sign([1., -2., 3., -4., 5.]), rtol=1e-4)


def test_cheetah_surrogate_spec_properties():
    from oracle import cheetah_surrogate as cs
    rng = np.random.RandomState(0)
    qpos, qvel = cs.reset_state(rng)
    assert np.abs(qpos).max() <= 0.1 and cs.get_obs(qpos, qvel).shape == (17,)
    u = rng.uniform(-1, 1, size=6)
    q1, v1, r, rr, rc = cs.step(qpos, qvel, u, 1.0)
    q2, v2, r2, rr2, rc2 = cs.step(qpos, qvel, u, -1.0)
    assert np.allclose(q1, q2) and rr == -rr2 and rc == rc2 and np.isclose(r, rr + rc)       # direction only flips reward_run
    assert np.isclose(rc, -0.05 * np.sum(u ** 2))
    # float32 evaluation tracks float64
    q32, v32, r32, _, _ = cs.step(qpos.astype(np.float32), qvel.astype(np.float32), u.astype(np.float32), np.float32(1.0))
    np.testing.assert_allclose(q32, q1, atol=1e-6)
    # bounded under sustained random torques
    for _ in range(400):
        qpos, qvel, _, _, _ = cs.step(qpos, qvel, rng.uniform(-1, 1, size=6), 1.0)
    assert np.abs(qpos[1:]).max() < 5 and np.abs(qvel).max() < 20


# ------------------------------------------------------------------ multi-rank host path (gloo, CPU)
def test_two_rank_gloo_sharding_and_allreduce():
    env = dict(os.environ, MASTER_ADDR='127.0.0.1')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29533', os.path.join(ROOT, 'tests', '_gloo_worker.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert 'rank 0 ok' in r.stdout and 'rank 1 ok' in r.stdout


# ------------------------------------------------------------------ the reference's unchanged Trainer
def test_reference_trainer_drives_promp_classes_unchanged(golden_dir):
    """The driver protocol of meta_policy_search/meta_trainer.py (unmodified): tests/golden/trainer_protocol.npz holds the
    method calls the reference Trainer makes on recording doubles over 2 iterations with one inner step, and the
    TensorFlow names it uses with promp_b200/tf_shim imported as `tensorflow` (oracle/make_golden.py::gen_trainer_protocol).
    promp_b200's Trainer must make the same calls in the same order (plus the sampler capability probe that decides on
    CUDA-graph replay), and the shim must provide every name the reference Trainer takes from TensorFlow."""
    import importlib.util
    from promp_b200.meta_trainer import Trainer
    from promp_b200.utils import logger
    g = np.load(os.path.join(golden_dir, 'trainer_protocol.npz'))
    calls = []

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
    sampler = Rec('sampler')
    sampler.total_timesteps_sampled = 0
    proc = Rec('proc')
    proc.baseline = Rec('baseline')
    logger.set_quiet(True)
    Trainer(algo=Rec('algo'), env=Rec('env'), sampler=sampler, sample_processor=proc, policy=Rec('policy'), n_itr=2,
            num_inner_grad_steps=1).train()
    assert calls[0] == 'sampler._fused_ok', calls
    assert calls[1:] == list(g['calls']), calls
    spec = importlib.util.spec_from_file_location(
        'tf_shim', os.path.join(ROOT, 'promp_b200', 'tf_shim', 'tensorflow', '__init__.py'))
    tf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tf)
    for name in g['tf_names']:
        assert callable(getattr(tf, str(name), None)), name
    sess = tf.Session()
    for name in g['session_methods']:
        assert callable(getattr(sess, str(name), None)), name
    with sess.as_default() as s:
        assert s is sess and s.run(tf.variables_initializer(tf.global_variables())) is None
    sess.close()


def test_logger_file_formats_and_snapshot_modes(tmp_path):
    """utils/logger.py:37-146, 376-427 behaviours: progress.csv grows its header and pads earlier rows when new keys
    appear, progress.json holds one object per dump, log.txt the printed table; snapshot_mode all / last / gap /
    last_gap / none choose the file names the reference uses."""
    import csv
    import json
    from promp_b200.utils import logger
    d = str(tmp_path / 'run')
    try:
        logger.configure(dir=d, format_strs=['log', 'csv', 'json'], snapshot_mode='gap', snapshot_gap=2)
        logger.logkv('Itr', 0); logger.logkv('Step_0-AverageReturn', np.float32(-1.5)); logger.dumpkvs()
        logger.logkv('Itr', 1); logger.logkv('Step_0-AverageReturn', -1.25); logger.logkv('KLCoeffInner', 5e-4); logger.dumpkvs()
        logger.log('hello', ' world')
        assert logger.save_itr_params(1, dict(itr=1)) is None
        p = logger.save_itr_params(2, dict(itr=2, x=np.arange(3)))
        assert os.path.basename(p) == 'itr_2.pkl' and logger.load_snapshot(p)['itr'] == 2
        rows = list(csv.reader(open(os.path.join(d, 'progress.csv'))))
        assert rows[0] == ['Itr', 'Step_0-AverageReturn', 'KLCoeffInner']
        assert rows[1] == ['0', '-1.5', ''] and rows[2] == ['1', '-1.25', '0.0005']
        js = [json.loads(l) for l in open(os.path.join(d, 'progress.json'))]
        assert js[0] == {'Itr': 0, 'Step_0-AverageReturn': -1.5} and js[1]['KLCoeffInner'] == 5e-4
        txt = open(os.path.join(d, 'log.txt')).read()
        assert '| Itr ' in txt and 'hello world' in txt and txt.count('-1.5') == 1
        for mode, itr, want in (('all', 3, 'itr_3.pkl'), ('last', 3, 'params.pkl'), ('last_gap', 4, 'params.pkl'), ('none', 4, None)):
            logger.configure(dir=d, format_strs=['json'], snapshot_mode=mode, snapshot_gap=2)
            got = logger.save_itr_params(itr, dict(itr=itr))
            assert (got and os.path.basename(got)) == want
        with pytest.raises(ValueError):
            logger.configure(dir=d, format_strs=['tensorboard'])
    finally:
        logger.reset()


def test_ragged_phase_path_table():
    """RaggedPhaseData (variable-length paths): prefix-sum path table, per-task counts, padding to a multiple of 4 rows -
    the host-side contract promp_process_samples_ragged / promp_policy_*_ragged read (include/promp_b200.h)."""
    import torch
    from promp_b200.samplers.device_data import RaggedPhaseData
    lens = [[5, 17, 1], [40], [9, 9, 9, 25, 2]]
    ph = RaggedPhaseData(lens, 2, 2, torch.device('cpu'))
    assert ph.M == 3 and ph.E == 5 and ph.N == 56 and ph.N % 4 == 0          # Pmax = 5, Nmax = max(23, 40, 54) -> 56
    np.testing.assert_array_equal(ph.n_valid_host, [23, 40, 54])
    np.testing.assert_array_equal(ph.n_paths_host, [3, 1, 5])
    np.testing.assert_array_equal(ph.path_off_host, [[0, 5, 22, 23, 23, 23], [0, 40, 40, 40, 40, 40], [0, 9, 18, 27, 52, 54]])
    assert ph.path_off.dtype == torch.int32 and ph.n_valid.dtype == torch.int32 and ph.total_paths == 9
    assert ph.obs.shape == (3, 56, 2) and float(ph.obs.abs().sum()) == 0.0       # padding rows start zeroed


def test_path_stacking_matches_reference_utils(golden_dir):
    """Trajectory bookkeeping of the stepwise sampler (SURVEY row a8): per-step info dicts -> one dict of stacked arrays,
    nested dicts included, exactly like utils.stack_tensor_dict_list (meta_policy_search/utils/utils.py) of the unmodified
    reference on the same seeded steps (tests/golden/stack_tensor_dict_list.npz)."""
    from promp_b200.samplers.meta_sampler import _stack
    want = np.load(os.path.join(golden_dir, 'stack_tensor_dict_list.npz'))
    rng = np.random.RandomState(0)
    steps = [dict(mean=rng.randn(3), log_std=rng.randn(3), nested=dict(a=rng.randn(2), b=float(i))) for i in range(7)]
    got = _stack(steps)
    assert sorted(got) == list(want['keys']) and sorted(got['nested']) == list(want['nested_keys'])
    for k in ('mean', 'log_std'):
        np.testing.assert_array_equal(got[k], want[k])
    for k in ('a', 'b'):
        np.testing.assert_array_equal(got['nested'][k], want['nested_' + k])
    assert _stack([]) == {} and _stack([{}, {}]) == {}


def test_policy_chain_plan_host_side():
    """promp_policy_chain's host-side planning (no GPU work): which shapes the automatic choice sends to the dataflow kernel
    (one to three 128-sample tiles per SM and stage; the SM count falls back to 148 without a device), the workspace bound, and
    argument validation through the C ABI."""
    import ctypes
    from promp_b200 import _lib
    lib = _lib.load()

    def stages(kinds, N):
        arr = (_lib.PolicyStage * len(kinds))()
        for i, k in enumerate(kinds):
            arr[i].kind, arr[i].N = k, N
        return arr, ctypes.cast(arr, ctypes.c_void_p)
    full = [0, 0, 1]
    for (Do, Da, hid, M, N, want) in [(2, 2, 64, 10, 2000, 1), (2, 2, 64, 20, 2000, 1), (2, 2, 64, 40, 2000, 3),
                                      (2, 2, 64, 5, 2000, 3), (17, 6, 64, 10, 4000, 1), (17, 6, 64, 40, 4000, 3),
                                      (2, 2, 32, 10, 2000, 3)]:          # hidden 32: no tensor-core kernels, always per stage
        arr, ptr = stages(full, N)
        assert lib.promp_policy_chain_num_launches(Do, Da, hid, M, 3, ptr) == want, (Do, Da, hid, M, N)
        ws = lib.promp_policy_chain_workspace_bytes(Do, Da, hid, M, 3, ptr)
        assert ws >= lib.promp_policy_workspace_bytes(M, N, Do, Da, hid) > 0
    try:
        _lib.set_option('chain', 1)
        arr, ptr = stages(full, 2000)
        assert lib.promp_policy_chain_num_launches(2, 2, 64, 40, 3, ptr) == 1
        _lib.set_option('chain', 0)
        assert lib.promp_policy_chain_num_launches(2, 2, 64, 10, 3, ptr) == 3
    finally:
        _lib.set_option('chain', -1)
    arr, ptr = stages(full, 2000)
    assert lib.promp_policy_chain_num_launches(2, 2, 64, 10, 7, ptr) < 0          # more than 6 stages
    assert lib.promp_policy_chain_workspace_bytes(3, 3, 64, 10, 3, ptr) < 0       # unsupported dimensions
    # the launch entry validates before touching the device
    rc = lib.promp_policy_chain(2, 2, 64, 10, ctypes.c_float(-13.8), 3, ptr, None, None, ctypes.c_void_p(16), 1 << 20, None)
    assert rc == -1 and 'null pointer' in _lib.last_error()


def test_policy_stage_struct_layout_matches_header(tmp_path):
    """The ctypes mirror of promp_policy_stage has the size and field offsets a C compiler gives the header's struct (the header
    is plain C: compiled here with gcc, no CUDA needed)."""
    import ctypes
    import shutil
    import subprocess
    from promp_b200 import _lib
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip("no gcc")
    fields = [name for name, _ in _lib.PolicyStage._fields_]
    src = tmp_path / 'layout.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "promp_b200.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(promp_policy_stage));\n' +
                   ''.join('  printf("%%zu\\n", offsetof(promp_policy_stage, %s));\n' % f for f in fields) +
                   '  return 0;\n}\n')
    exe = tmp_path / 'layout'
    subprocess.run([gcc, '-std=c99', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.PolicyStage)
    for f, off in zip(fields, out[1:]):
        assert getattr(_lib.PolicyStage, f).offset == off, f
