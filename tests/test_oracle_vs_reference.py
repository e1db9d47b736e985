"""Pins the oracle port and the product's host-side code against the UNMODIFIED reference.

The reference has no tests or golden vectors (SURVEY.md section 4), so the pin is: the reference's own collector +
buffer + PPO, off-policy agents, logger, networks, epoch loop, flags, helpers and host VecEnv were run from the seeds
and inputs below, and what they produced is stored in tests/golden/reference_pins.npz (`python -m oracle.make_golden
pins` regenerates it where the reference is importable).  The oracle port and the product must reproduce it exactly.
"""
import hashlib
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PPO_CASE = (4, 16, (16, 16), 4, 2, 3)          # N, T, hidden, batch rows, opt epochs, seed
PPO_MAX_FRAMES = (999, 7)
PPO_KEYS = ("obs", "next_obs", "acts", "values", "rewards", "terminals", "time_limits")
OFF_CASE = (11, 3, (24, 24), 48, 4)             # obs dim, act dim, hidden, batch, seed
ARGVS = [[], ["--seed", "3", "--vec_env_nums", "16", "--config", "c.json", "--id", "x", "--overwrite"],
         ["--no_cuda", "--device", "2", "--save_dir", "/tmp/s", "--log_dir", "/tmp/l",
          "--proc_nums", "8", "--eval_worker_nums", "1"]]
VEC_N, VEC_T, VEC_PARAM = 5, 14, {"reward_scale": 0.25}


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_pins.npz"))


def _infos(g, tag):
    return json.loads(str(g[tag + "_infos"]))


def _params(g, tag):
    return [g["%s_p%d" % (tag, i)] for i in range(int(g[tag + "_nparams"]))]


def _digest(a, dtype=None):
    """[shape, dtype, sha256 of the bytes]: pins bit-exact equality without storing the values."""
    a = np.ascontiguousarray(np.asarray(a, dtype=dtype))
    return [list(a.shape), str(a.dtype), hashlib.sha256(a.tobytes()).hexdigest()]


def _param_key(a):
    return [list(a.shape), float(np.abs(a).sum())]


class _NullLogger:
    def __init__(self):
        self.infos = []

    def add_update_info(self, info):
        self.infos.append(info)

    def add_epoch_info(self, *a, **k):
        pass

    def log(self, *a):
        pass

    def finish(self):
        pass


@pytest.mark.parametrize("max_frames", PPO_MAX_FRAMES)
def test_port_reproduces_reference_ppo(g, max_frames):
    """The oracle port, from the reference's seeding, gives identical rollouts, advantages, parameters, logged
    scalars and normaliser state over two epochs."""
    from oracle import ref_port
    N, T, hidden, rows, oe, seed = PPO_CASE
    tag = "ppo%d" % max_frames
    penv, pcol, pagent = ref_port.build_ppo(env_nums=N, horizon=T, hidden=hidden, batch_rows=rows, opt_epochs=oe,
                                            seed=seed, max_episode_frames=max_frames)
    ref = json.loads(str(g[tag + "_arrays"]))

    def check(name, a):                 # same values as the reference's float64 buffers, bit for bit
        assert _digest(a, dtype=ref[name][1]) == ref[name], name
    for epoch in range(2):
        pagent.current_epoch = epoch
        out = pcol.train_one_epoch()
        assert out["train_epoch_reward"] == g[tag + "_rewards"][epoch]
        for k in PPO_KEYS:
            check("e%d_%s" % (epoch, k), pagent.buffer.data[k])
        pagent.update_per_epoch()
        check("e%d_advs" % epoch, pagent.buffer.data["advs"])
        check("e%d_rets" % epoch, pagent.buffer.data["estimate_returns"])
    p_params = [p.detach().numpy() for p in list(pagent.pf.parameters()) + list(pagent.vf.parameters())]
    # the port keeps `logstd` after the net parameters; the reference registers it first
    assert json.loads(str(g[tag + "_param_keys"])) == sorted(map(_param_key, p_params))
    r_infos = _infos(g, tag)
    assert len(r_infos) == len(pagent.infos) == 2 * oe * (T // rows)
    for a, b in zip(r_infos, pagent.infos):
        assert a.keys() == b.keys()
        for k in a:
            assert a[k] == b[k], k
    np.testing.assert_array_equal(g[tag + "_norm_mean"], penv.norm.mean)
    np.testing.assert_array_equal(g[tag + "_norm_var"], penv.norm.var)
    assert g[tag + "_norm_count"] == penv.norm.count


def test_numpy_oracle_pieces_against_reference_functions(g):
    """Normalizer, quantile loss: ref_numpy vs the reference's own functions."""
    from oracle import ref_numpy as rn
    rs = np.random.RandomState(0)
    mine = rn.RunningNorm(5)
    for i in range(4):
        x = rs.randn(9, 5) * 3 + 1
        mine.update(x)
        np.testing.assert_array_equal(g["pieces_filt"][i], mine.filt(x))
    np.testing.assert_array_equal(g["pieces_mean"], mine.mean)
    np.testing.assert_array_equal(g["pieces_var"], mine.var)
    tau = (2 * np.arange(7) + 1) / 14.0
    src, tgt = rs.randn(6, 7), rs.randn(6, 7)
    assert abs(float(g["pieces_qr"]) - rn.quantile_regression_loss(tau, src, tgt)) < 1e-12


def _offpolicy_batches(o, a, B, n, seed):
    rs = np.random.RandomState(seed)
    return [{"obs": rs.randn(B, o), "next_obs": rs.randn(B, o), "acts": np.tanh(rs.randn(B, a)),
             "rewards": rs.randn(B, 1), "terminals": (rs.rand(B, 1) < 0.1).astype(np.float64)} for _ in range(n)]


def _check_updates(g, tag, port_infos, port_params):
    ref_infos, ref_params = _infos(g, tag), _params(g, tag)
    assert len(ref_infos) == len(port_infos)
    for x, y in zip(ref_infos, port_infos):
        assert x.keys() == y.keys()
        for k in x:
            assert x[k] == y[k], k
    assert len(ref_params) == len(port_params)
    for x, y in zip(ref_params, port_params):
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("kind", ["sac", "td3"])
def test_port_reproduces_reference_offpolicy_updates(g, kind):
    import torch
    import torch.nn as nn
    from oracle import ref_port
    o, a, hidden, B, seed = OFF_CASE
    batches = _offpolicy_batches(o, a, B, 4, seed)
    torch.manual_seed(seed)
    if kind == "sac":
        ppf = ref_port.TanhGaussianPolicy(o, a, list(hidden), nn.ReLU, state_dependent_std=True)
    else:
        ppf = ref_port.FixedNoisePolicy(o, a, list(hidden), nn.ReLU, norm_std_explore=0.1, tanh_action=True)
    pq1 = ref_port.QNet(o + a, 1, list(hidden), nn.ReLU)
    pq2 = ref_port.QNet(o + a, 1, list(hidden), nn.ReLU)
    if kind == "sac":
        port = ref_port.SACPort(ppf, pq1, pq2, a, std_reg=1e-3, mean_reg=1e-3)
        nets = [port.pf, port.qf1, port.qf2, port.tqf1, port.tqf2]
    else:
        port = ref_port.TD3Port(ppf, pq1, pq2, plr=1e-3, qlr=1e-3)
        nets = [port.pf, port.qf1, port.qf2, port.tpf, port.tqf1, port.tqf2]
    torch.manual_seed(100)
    port_infos = [port.update(b) for b in batches]
    _check_updates(g, kind, port_infos, [p.detach().numpy() for n_ in nets for p in n_.parameters()])


def test_port_reproduces_reference_ddpg_updates(g):
    import torch
    import torch.nn as nn
    from oracle import ref_port
    o, a, hidden, B, seed = OFF_CASE
    batches = _offpolicy_batches(o, a, B, 4, seed)
    torch.manual_seed(seed)
    ppf = ref_port.FixedNoisePolicy(o, a, list(hidden), nn.ReLU, norm_std_explore=0.1, tanh_action=True)
    pq = ref_port.QNet(o + a, 1, list(hidden), nn.ReLU)
    port = ref_port.DDPGPort(ppf, pq, plr=1e-3, qlr=1e-3)
    port_infos = [port.update(b) for b in batches]
    _check_updates(g, "ddpg", port_infos,
                   [p.detach().numpy() for n_ in (port.pf, port.qf, port.tpf, port.tqf) for p in n_.parameters()])


def _logger_inputs(rs):
    updates = [[{"Training/policy_loss": rs.randn(), "Training/vf_loss": abs(rs.randn()), "ratio/max": 1 + rs.rand()}
                for _ in range(5)] for _ in range(3)]
    epochs = [{"Running_Average_Rewards": rs.randn() * 100, "Train_Epoch_Reward": rs.randn() * 1e3,
               "eval_traj_length": 1000.0} for _ in range(3)]
    return updates, epochs


def _logger_params():
    return {"project": "p", "env_name": "SynthHalfCheetah-v0", "general_setting": {"discount": 0.99}}


def test_logger_files_match_reference(g, tmp_path, capsys):
    """utils/logger.py:17-158: same log.csv (titles, per-epoch values, Mean/Std/Max/Min aggregation of the
    per-update infos, "{:.5f}" formatting) and params.json from the product's Logger and the reference's."""
    from torchrl_b200.utils.logger import Logger
    updates, epochs = _logger_inputs(np.random.RandomState(0))
    lg = Logger("exp", "SynthHalfCheetah-v0", 3, _logger_params(), log_dir=str(tmp_path))
    for e in range(3):
        for info in updates[e]:
            lg.add_update_info(info)
        lg.add_epoch_info(e, (e + 1) * 4096, 1.5 * (e + 1), epochs[e])
    lg.finish()
    d = tmp_path / "exp" / "SynthHalfCheetah-v0" / "3"
    capsys.readouterr()
    ref_csv = str(g["logger_csv"])
    assert open(d / "log.csv").read() == ref_csv
    assert json.load(open(d / "params.json")) == json.loads(str(g["logger_params"]))
    assert ref_csv.count("\n") == 4 and "Training/policy_loss_Std" in ref_csv


def _build_nets(net_mod, pol_mod, seed):
    import torch
    import torch.nn as nn
    torch.manual_seed(seed)
    kw = dict(hidden_shapes=[32, 24], append_hidden_shapes=[], base_type=net_mod.MLPBase, activation_func=nn.Tanh)
    kw2 = dict(hidden_shapes=[32], append_hidden_shapes=[16], base_type=net_mod.MLPBase, activation_func=nn.ReLU)
    cnn = dict(hidden_shapes=[[16, [8, 8], [4, 4], [0, 0]], [32, [4, 4], [2, 2], [0, 0]]], append_hidden_shapes=[64],
               base_type=net_mod.CNNBase, activation_func=nn.ReLU)
    return [
        ("Net", net_mod.Net(input_shape=17, output_shape=1, **kw)),
        ("Net+append", net_mod.Net(input_shape=17, output_shape=3, **kw2)),
        ("QNet", net_mod.QNet(input_shape=23, output_shape=1, **kw)),
        ("BasicBias", pol_mod.GuassianContPolicyBasicBias(input_shape=17, output_shape=6, tanh_action=True, **kw)),
        ("Gaussian", pol_mod.GuassianContPolicy(input_shape=17, output_shape=12, tanh_action=True, **kw)),
        ("FixGaussian", pol_mod.FixGuassianContPolicy(input_shape=17, output_shape=6, norm_std_explore=0.1,
                                                    tanh_action=True, **kw)),
        ("Det", pol_mod.DetContPolicy(input_shape=17, output_shape=6, tanh_action=True, **kw)),
        ("CNN", net_mod.Net(input_shape=(4, 84, 84), output_shape=6, **cnn)),
    ]


def _forward_nets(nets):
    """CPU forward outputs of each net on inputs drawn from the torch generator right after the nets were built."""
    import torch
    x = torch.randn(5, 17)
    out = []
    for name, m in nets:
        with torch.no_grad():
            if name == "QNet":
                y = m([x, torch.randn(5, 6).fill_(0.3)])
            elif name == "CNN":
                y = m(torch.rand(2, 4, 84, 84))
            else:
                y = m(x)
        out.append((name, list(y) if isinstance(y, (tuple, list)) else [y]))
    return out


def test_networks_and_policies_are_state_dict_compatible_with_reference(g):
    """networks/{init,base,nets}.py, policies/continuous_policy.py: equal seeds give bit-identical parameters
    (same creation order and RNG consumption), identical state_dict keys / shapes (so `model_*.pth` snapshots load
    into either code base, algo/rl_algo.py:90-94) and identical CPU forward outputs.  The reference's parameters are
    stored as (shape, dtype, sha256 of the bytes)."""
    import torchrl_b200.networks as mnet
    import torchrl_b200.policies as mpol
    ref_state = json.loads(str(g["nets_state"]))
    nets = _build_nets(mnet, mpol, 7)
    for name, m in nets:
        mine = [[k, _digest(v.detach().numpy())] for k, v in m.state_dict().items()]
        assert [k for k, _ in ref_state[name]] == [k for k, _ in mine], name
        for (k, a), (_, b) in zip(ref_state[name], mine):
            assert a == b, (name, k)
    for name, ys in _forward_nets(nets):
        assert len(ys) == int(g["nets_out_%s_n" % name]), name
        for i, y in enumerate(ys):
            np.testing.assert_array_equal(y.numpy(), g["nets_out_%s_%d" % (name, i)], err_msg=name)


class _BookCol:
    epoch_frames = 64

    def __init__(self):
        self.k = self.e = 0
        self.terminated = False

    def train_one_epoch(self):
        self.k += 1
        return {"train_rewards": [float(self.k * 10 + i) for i in range(self.k % 3)],
                "train_epoch_reward": 1.5 * self.k}

    def eval_one_epoch(self):
        self.e += 1
        return {"eval_rewards": [(-1.0) ** self.e * 2.0 * self.e, float(self.e)], "eval_traj_length": 100.0 + self.e}

    def terminate(self):
        self.terminated = True


class _BookLog:
    def __init__(self):
        self.rows, self.finished = [], False

    def add_epoch_info(self, epoch, frames, seconds, infos, csv_write=True):
        self.rows.append((epoch, frames, list(infos.keys()),
                          {k: float(v) for k, v in infos.items() if "Time" not in k}))

    def add_update_info(self, info):
        pass

    def finish(self):
        self.finished = True


def _BookEnv():
    from oracle import reference_loader
    reference_loader.add_shims()
    import gym                                  # the oracle's stand-in (oracle/shims)

    class Env:
        action_space = gym.spaces.Box(-np.ones(3), np.ones(3))
        _obs_normalizer = None
    return Env()


def _instrument(cls):
    class Agent(cls):
        def snapshot(self, prefix, epoch):
            self.snaps.append(epoch)

        def update_per_epoch(self):
            self.updates += 1

        def finish_epoch(self):
            return {"extra/epoch": float(self.current_epoch)}

        def _device_sync(self):
            pass
    return Agent


def test_train_loop_bookkeeping_matches_reference(g, tmp_path):
    """RLAlgo.train (algo/rl_algo.py:96-165): with the same stub collector / logger the product's epoch loop makes the
    same calls in the same order -- epoch rows (keys, key order, values), evaluation cadence, best / periodic /
    final snapshots, running-average windows -- as the reference's."""
    import torch
    from torchrl_b200.algo.rl_algo import RLAlgo
    ref = json.loads(str(g["train_loop"]))
    col_m, log_m = _BookCol(), _BookLog()
    mine = object.__new__(_instrument(RLAlgo))
    mine.device = torch.device("cpu")
    mine._init_bookkeeping(_BookEnv(), None, col_m, log_m, None, 0.99, 7, 64, 3, 2, str(tmp_path / "m"))
    mine.snaps, mine.updates = [], 0
    mine.train()

    assert mine.snaps == ref["snaps"] and mine.updates == ref["updates"] == 7
    assert col_m.terminated and log_m.finished and col_m.e == ref["evals"]
    assert len(log_m.rows) == len(ref["rows"]) == 4
    for (e0, f0, k0, v0), (e1, f1, k1, v1) in zip(ref["rows"], log_m.rows):
        assert (e0, f0, k0) == (e1, f1, k1)
        for k in v0:
            assert v0[k] == v1[k] or (np.isnan(v0[k]) and np.isnan(v1[k])), k
    assert list(mine.episode_rewards) == ref["episode_rewards"]
    assert list(mine.training_episode_rewards) == ref["training_episode_rewards"]
    assert mine.best_eval == ref["best_eval"]


@pytest.mark.parametrize("argv", ARGVS)
def test_command_line_flags_match_reference(g, argv):
    """utils/args.py:6-46: same flags, types and defaults (the example scripts read the namespace).  The reference's
    `cuda` flag asks torch.cuda.is_available(); its flags were recorded for either answer."""
    import torch
    from torchrl_b200.utils.args import get_args
    ref = json.loads(str(g["args_cuda%d" % torch.cuda.is_available()]))[ARGVS.index(argv)]
    mine = vars(get_args(argv))
    assert mine == ref
    assert {k: type(v) for k, v in mine.items()} == {k: type(v) for k, v in ref.items()}


def _utils_nets():
    import copy
    import torch
    src = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Tanh(), torch.nn.Linear(5, 2))
    tgt_a = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Tanh(), torch.nn.Linear(5, 2))
    return src, tgt_a, copy.deepcopy(tgt_a)


def test_algo_utils_match_reference(g):
    """algo/utils.py:5-32: huber, quantile_regression_loss, Polyak / hard target updates and the linear LR
    schedule give bit-identical results."""
    import torch
    import torchrl_b200.algo.utils as mine
    torch.manual_seed(0)
    x = torch.randn(64) * 2
    assert torch.equal(torch.from_numpy(g["utils_huber"]), mine.huber(x))
    assert torch.equal(torch.from_numpy(g["utils_huber_03"]), mine.huber(x, 0.3))
    for dt in (torch.float32, torch.float64):
        tau = ((2 * torch.arange(9) + 1) / 18.0).to(dt)
        s, t = torch.randn(5, 9, dtype=dt), torch.randn(5, 9, dtype=dt)
        ref = torch.from_numpy(g["utils_qr_" + str(dt)[6:]])
        assert torch.equal(ref, mine.quantile_regression_loss(tau, s, t))
    src, _, tgt = _utils_nets()
    for _ in range(3):
        mine.soft_update_from_to(src, tgt, 0.005)
    ref_soft = _params(g, "utils_soft")
    assert len(ref_soft) == len(list(tgt.parameters()))
    for p, q in zip(ref_soft, tgt.parameters()):
        assert torch.equal(torch.from_numpy(p), q.detach())
    mine.copy_model_params_from_to(src, tgt)
    for q, r in zip(tgt.parameters(), src.parameters()):
        assert torch.equal(q, r)
    opt = torch.optim.Adam(tgt.parameters(), lr=1.0)
    for epoch, lr in zip((0, 17, 487), g["utils_lrs"]):
        mine.update_linear_schedule(opt, epoch, 488, 3e-4)
        assert opt.param_groups[0]["lr"] == lr


def test_epsilon_greedy_policy_matches_reference(g):
    """policies/discrete_policies.py:25-74: same exploration schedule and, with the reference's NumPy noise stream,
    the same decisions."""
    import torch
    import torchrl_b200.policies as mpol
    torch.manual_seed(0)
    qf = torch.nn.Linear(5, 4)
    mine = mpol.EpsilonGreedyDQNDiscretePolicy(qf=qf, start_epsilon=1.0, end_epsilon=0.1, decay_frames=20,
                                               action_shape=4)
    obs = torch.randn(30, 1, 5)
    mpol.set_noise_mode("reference_cpu")
    try:
        np.random.seed(3)
        a_mine = [(mine.explore(o)["action"].clone(), mine.epsilon) for o in obs]
    finally:
        mpol.set_noise_mode("philox")
    assert len(a_mine) == len(g["egreedy_acts"])
    for a0, e0, (a1, e1) in zip(g["egreedy_acts"], g["egreedy_eps"], a_mine):
        assert e0 == e1 and torch.equal(torch.from_numpy(a0), a1)
    assert mine.count == int(g["egreedy_count"]) == 30 and mine.epsilon == 0.1


def _shorten(env):
    """Reach the TimeLimit core of either wrapper chain and shorten its episodes."""
    core = env
    while not hasattr(core, "_max_episode_steps") or hasattr(core, "env") and hasattr(core.env, "_max_episode_steps"):
        core = core.env
    core._max_episode_steps = 6


@pytest.mark.parametrize("adt", [np.float32, np.float64])
def test_host_vecenv_and_wrapper_chain_match_reference(g, adt):
    """env/vecenv.py:6-78 + get_env.py:52-67 (NormAct, RewardShift, TimeLimitAugment): the product's host VecEnv over
    its one-object wrapper chain returns the same observations / rewards / flags, step for step, as the reference's
    VecEnv over the reference's stacked gym wrappers (same action dtype handed through)."""
    from oracle import synth_env
    from torchrl_b200.hostenv import VecEnv, get_single_env
    tag = "vecenv_" + np.dtype(adt).name
    mine = VecEnv(VEC_N, get_single_env, ["SynthHalfCheetah-v0", dict(VEC_PARAM), synth_env.make_env])
    for e in mine.envs:
        _shorten(e)
    mine.seed(9)
    np.testing.assert_array_equal(g[tag + "_reset"], mine.reset())
    rs = np.random.RandomState(1)
    for t in range(VEC_T):
        acts = rs.uniform(-1.4, 1.4, size=(VEC_N, 6)).astype(adt)
        o0, r0, d0, tl0 = (g["%s_%s" % (tag, k)][t] for k in ("obs", "rew", "done", "time_limit"))
        o1, r1, d1, i1 = mine.step(acts)
        np.testing.assert_array_equal(o0, o1)
        np.testing.assert_array_equal(r0, r1)
        np.testing.assert_array_equal(d0, d1)
        np.testing.assert_array_equal(tl0, i1["time_limit"])
        if d0.any():
            np.testing.assert_array_equal(g[tag + "_reset_rows"][t], mine.partial_reset(d1.squeeze(-1)))
        if t == 8:
            mine.eval()                    # RewardShift is train-only
    assert d0.dtype == d1.dtype and r0.shape == r1.shape == (VEC_N, 1)
