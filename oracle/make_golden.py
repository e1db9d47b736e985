"""Generate tests/golden/*.npz by executing the UNMODIFIED reference on CPU.

TEST INFRASTRUCTURE.  Run in the build container only (needs /root/reference):

    python -m oracle.make_golden            # regenerates every fixture

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so
the fixtures are outputs of the reference's own functions on seeded inputs.
Each fixture stores the inputs, or the seeds the tests draw them from, so the tests need nothing else.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def gae_inputs(T, N, seed=0, p_term=0.01, p_tl=0.005):
    """SURVEY.md section 8(d) recipe, in this exact draw order."""
    rs = np.random.RandomState(seed)
    values = rs.randn(T, N, 1)
    rewards = rs.randn(T, N, 1)
    terminals = (rs.rand(T, N, 1) < p_term)
    time_limits = (rs.rand(T, N, 1) < p_tl)
    last_value = rs.randn(N, 1)
    return values, rewards, terminals, time_limits, last_value


def golden_gae(trl):
    from torchrl.replay_buffers import OnPolicyReplayBuffer
    out = {}
    cases = [(128, 8, 0, 0.01, 0.005), (37, 5, 1, 0.2, 0.1), (1, 3, 2, 0.5, 0.5), (256, 33, 3, 0.02, 0.02)]
    for ci, (T, N, seed, pt, ptl) in enumerate(cases):
        values, rewards, terminals, time_limits, last_value = gae_inputs(T, N, seed, pt, ptl)
        for flt in (True, False):
            buf = OnPolicyReplayBuffer(max_replay_buffer_size=T * N, env_nums=N, time_limit_filter=flt)
            buf._values = values.astype(np.float64)
            buf._rewards = rewards.astype(np.float64)
            buf._terminals = terminals.astype(np.float64)
            buf._time_limits = time_limits.astype(np.float64)
            buf.generalized_advantage_estimation(last_value, 0.99, 0.95)
            tag = "c%d_f%d" % (ci, int(flt))
            out[tag + "_gae_advs"] = buf._advs.copy()
            out[tag + "_gae_rets"] = buf._estimate_returns.copy()
            buf.discount_reward(last_value, 0.99)
            out[tag + "_disc_advs"] = buf._advs.copy()
            out[tag + "_disc_rets"] = buf._estimate_returns.copy()
        out["c%d_values" % ci] = values
        out["c%d_rewards" % ci] = rewards
        out["c%d_terminals" % ci] = terminals
        out["c%d_time_limits" % ci] = time_limits
        out["c%d_last_value" % ci] = last_value
    out["ncases"] = np.array(len(cases))
    out["gamma_tau"] = np.array([0.99, 0.95])
    np.savez_compressed(os.path.join(GOLDEN, "gae.npz"), **out)
    print("gae.npz:", len(out), "arrays")


class _Quiet:
    """Logger stand-in for the reference agent (it only calls these)."""
    def add_update_info(self, info): pass
    def add_epoch_info(self, *a, **k): pass
    def log(self, *a): pass
    def finish(self): pass


def golden_hotpath(trl):
    """Seeded inputs -> outputs of the reference's OWN functions for the non-GAE rows of SURVEY.md 8(a):
    K2 Normalizer (env/base_wrapper.py:63-100), K3 TanhNormal.log_prob / entropy (policies/distribution.py:33-79),
    K7/K9 minibatch row order and uniform row indices (replay_buffers/on_policy.py:72-91, base.py:39-51),
    K8 PPO.update on one minibatch (algo/on_policy/ppo.py:41-150; the policy / value network OUTPUTS at the
    moment of the update are stored as the loss kernels' inputs), K10 quantile_regression_loss (algo/utils.py:5-13)."""
    import tempfile
    import torch
    import torchrl.networks as networks
    import torchrl.policies as policies
    from torchrl.algo import PPO
    from torchrl.algo.utils import quantile_regression_loss
    from torchrl.collector.on_policy import VecOnPolicyCollector
    from torchrl.env import get_vec_env
    from torchrl.env.base_wrapper import Normalizer
    from torchrl.policies.distribution import TanhNormal
    from torchrl.replay_buffers.on_policy import OnPolicyReplayBuffer
    from torchrl.replay_buffers.base import BaseReplayBuffer
    out = {}

    # ---- K2: running normaliser over 6 batches of (64, 17)
    rs = np.random.RandomState(11)
    batches = rs.randn(6, 64, 17) * rs.uniform(0.5, 3.0, size=(1, 1, 17)) + 2.0 * rs.randn(1, 1, 17)
    nrm = Normalizer((17,))
    means, vars_, counts, filts = [], [], [], []
    for k in range(6):
        nrm.update_estimate(batches[k])
        means.append(nrm._mean.copy()); vars_.append(nrm._var.copy()); counts.append(nrm._count)
        filts.append(nrm.filt(batches[k]))
    far = batches[0] * 50.0                              # filter-only call (eval mode) far outside: +-10 clip
    out.update(norm_batches=batches, norm_mean=np.array(means), norm_var=np.array(vars_),
               norm_count=np.array(counts), norm_filt=np.array(filts), norm_far=far, norm_far_filt=nrm.filt(far))

    # ---- K3: tanh-Gaussian log-density and entropy (float64 tensors: the formula, not fp32 noise)
    rs = np.random.RandomState(12)
    mean = rs.randn(512, 6)
    log_std = 0.3 * rs.randn(6) - 1.0
    std = np.exp(log_std)[None].repeat(512, 0)
    acts = np.tanh(mean + std * rs.randn(512, 6) * 1.2).astype(np.float32).astype(np.float64)
    dist = TanhNormal(torch.from_numpy(mean), torch.from_numpy(std))
    out.update(tn_mean=mean, tn_log_std=log_std, tn_acts=acts,
               tn_log_prob=dist.log_prob(torch.from_numpy(acts)).numpy(), tn_entropy=dist.entropy().numpy())

    # ---- K7 / K9: row order of one_iteration and row indices of random_batch from the global NumPy stream
    T, N = 24, 4
    buf = OnPolicyReplayBuffer(max_replay_buffer_size=T * N, env_nums=N)
    rows = np.arange(T, dtype=np.float64)[:, None, None].repeat(N, 1)
    buf._obs = rows.copy()
    buf._max_replay_buffer_size = T
    np.random.seed(5)
    order = []
    for _pass in range(2):
        for mb in buf.one_iteration(batch_size=6 * N, sample_key=["obs"], shuffle=True):
            order.append(mb["obs"].reshape(6, N)[:, 0])
    out["iter_rows"] = np.array(order).astype(np.int64)               # (2*T/6, 6) row indices, bit-exact contract
    ring = BaseReplayBuffer(max_replay_buffer_size=40 * N, env_nums=N)
    ring._obs = np.arange(40, dtype=np.float64)[:, None, None].repeat(N, 1)
    ring._size = 33
    np.random.seed(6)
    out["rand_rows"] = np.array([ring.random_batch(5 * N, ["obs"])["obs"].reshape(5, N)[:, 0] for _ in range(4)]
                                ).astype(np.int64)

    # ---- K8: one PPO minibatch update by the reference agent
    for tag, clipped in (("ppo", False), ("ppoc", True)):
        torch.manual_seed(21)
        np.random.seed(21)
        Nenv, B = 4, 256
        params = {"reward_scale": 1, "obs_norm": False}
        env = get_vec_env("SynthHalfCheetah-v0", dict(params), Nenv)
        eval_env = get_vec_env("SynthHalfCheetah-v0", dict(params), Nenv)
        rb = OnPolicyReplayBuffer(env_nums=Nenv, max_replay_buffer_size=8 * Nenv, time_limit_filter=True)
        net = dict(hidden_shapes=[32, 32], append_hidden_shapes=[], base_type=networks.MLPBase,
                   activation_func=torch.nn.Tanh)
        pf = policies.GuassianContPolicyBasicBias(input_shape=17, output_shape=6, tanh_action=True, **net)
        vf = networks.Net(input_shape=(17,), output_shape=1, **net)
        col = VecOnPolicyCollector(vf, env=env, eval_env=eval_env, pf=pf, replay_buffer=rb, device="cpu",
                                   train_render=False, epoch_frames=8 * Nenv, max_episode_frames=999, eval_episodes=1)
        agent = PPO(pf=pf, vf=vf, plr=3e-4, vlr=3e-4, clip_para=0.2, opt_epochs=1, tau=0.95, shuffle=True,
                    entropy_coeff=0.005, env=env, replay_buffer=rb, collector=col, logger=_Quiet(), discount=0.99,
                    num_epochs=10, batch_size=B, gae=True, device="cpu", save_dir=tempfile.mkdtemp(),
                    clipped_value_loss=clipped)
        with torch.no_grad():
            for prm in agent.target_pf.parameters():               # old policy != new policy: ratios leave 1 +- clip
                prm.add_(0.01 * torch.randn_like(prm))
        rs = np.random.RandomState(22)
        obs = rs.randn(B, 17)
        obs_t = torch.Tensor(obs)
        with torch.no_grad():
            mean_t, std_t, log_std_t = pf(obs_t)
        acts = np.tanh(mean_t.numpy() + std_t.numpy() * rs.randn(B, 6)).astype(np.float32).astype(np.float64)
        batch = {"obs": obs, "acts": acts, "advs": 2.0 * rs.randn(B, 1) + 0.3,
                 "values": rs.randn(B, 1), "estimate_returns": rs.randn(B, 1)}
        acts_t = torch.Tensor(batch["acts"])
        with torch.no_grad():
            old_lp = agent.target_pf.update(obs_t, acts_t)["log_prob"]
            v_t = vf(obs_t)
        info = agent.update(batch)
        for k, v in batch.items():
            out["%s_%s" % (tag, k)] = v
        out["%s_mean" % tag] = mean_t.numpy().astype(np.float64)
        out["%s_log_std" % tag] = log_std_t.numpy().astype(np.float64).reshape(-1)
        out["%s_old_logp" % tag] = old_lp.numpy().astype(np.float64)
        out["%s_v" % tag] = v_t.numpy().astype(np.float64)
        keys = sorted(info.keys())
        out["%s_info_keys" % tag] = np.array(keys)
        out["%s_info_vals" % tag] = np.array([info[k] for k in keys], dtype=np.float64)

    # ---- K10: quantile-regression Huber loss (algo/utils.py:5-13) on (B, Q) source / target
    rs = np.random.RandomState(31)
    Bq, Q = 32, 51
    src, tgt = rs.randn(Bq, Q), rs.randn(Bq, Q) * 1.5 + 0.2
    tau = (2 * np.arange(Q) + 1) / (2.0 * Q)
    out.update(qr_source=src, qr_target=tgt, qr_tau=tau,
               qr_loss=np.array(quantile_regression_loss(torch.from_numpy(tau), torch.from_numpy(src),
                                                         torch.from_numpy(tgt)).item()))
    np.savez_compressed(os.path.join(GOLDEN, "hotpath.npz"), **out)
    print("hotpath.npz:", len(out), "arrays")


def _json(obj):
    return np.array(json.dumps(obj))


def _store_infos(out, tag, infos):
    """Logged scalars of each update, in key order (JSON keeps a float64 exactly)."""
    out[tag + "_infos"] = _json([{k: float(v) for k, v in i.items()} for i in infos])


def _store_params(out, tag, params):
    out[tag + "_nparams"] = np.array(len(params))
    for i, p in enumerate(params):
        out["%s_p%d" % (tag, i)] = p


def golden_pins(trl):
    """Outputs of the reference's own classes that tests/test_oracle_vs_reference.py pins the oracle port and the
    product's host-side code against (same seeds, same inputs as the tests draw)."""
    import tempfile
    import torch
    from tests import test_oracle_vs_reference as tv
    out = {}
    tmp = tempfile.mkdtemp()

    # ---- PPO: collector + buffer + agent, two epochs (test_port_reproduces_reference_ppo)
    import torchrl.networks as networks
    import torchrl.policies as policies
    from torchrl.algo import PPO
    from torchrl.collector.on_policy import VecOnPolicyCollector
    from torchrl.env import get_vec_env
    from torchrl.replay_buffers.on_policy import OnPolicyReplayBuffer
    N, T, hidden, rows, oe, seed = tv.PPO_CASE
    for max_frames in tv.PPO_MAX_FRAMES:
        tag = "ppo%d" % max_frames
        params = {"reward_scale": 1, "obs_norm": True}
        env = get_vec_env("SynthHalfCheetah-v0", dict(params), N)
        eval_env = get_vec_env("SynthHalfCheetah-v0", dict(params), N)
        env.seed(seed)
        torch.manual_seed(seed)
        np.random.seed(seed)
        buf = OnPolicyReplayBuffer(env_nums=N, max_replay_buffer_size=T * N, time_limit_filter=True)
        net = dict(hidden_shapes=list(hidden), append_hidden_shapes=[], base_type=networks.MLPBase,
                   activation_func=torch.nn.Tanh)
        pf = policies.GuassianContPolicyBasicBias(input_shape=env.observation_space.shape[0],
                                                  output_shape=env.action_space.shape[0], tanh_action=True, **net)
        vf = networks.Net(input_shape=env.observation_space.shape, output_shape=1, **net)
        col = VecOnPolicyCollector(vf, env=env, eval_env=eval_env, pf=pf, replay_buffer=buf, device="cpu",
                                   train_render=False, epoch_frames=T * N, max_episode_frames=max_frames, eval_episodes=1)
        logger = tv._NullLogger()
        agent = PPO(pf=pf, vf=vf, plr=3e-4, vlr=3e-4, clip_para=0.2, opt_epochs=oe, tau=0.95, shuffle=True,
                    entropy_coeff=0.005, env=env, replay_buffer=buf, collector=col, logger=logger, discount=0.99,
                    num_epochs=488, batch_size=rows * N, gae=True, device="cpu", save_dir=tmp)
        rewards, arrays = [], {}
        for epoch in range(2):
            agent.current_epoch = epoch
            rewards.append(col.train_one_epoch()["train_epoch_reward"])
            for k in tv.PPO_KEYS:
                arrays["e%d_%s" % (epoch, k)] = tv._digest(getattr(buf, "_" + k))
            agent.update_per_epoch()
            arrays["e%d_advs" % epoch] = tv._digest(buf._advs)
            arrays["e%d_rets" % epoch] = tv._digest(buf._estimate_returns)
        out[tag + "_rewards"] = np.array(rewards, dtype=np.float64)
        out[tag + "_arrays"] = _json(arrays)
        out[tag + "_param_keys"] = _json(sorted(tv._param_key(p.detach().numpy())
                                                for p in list(pf.parameters()) + list(vf.parameters())))
        _store_infos(out, tag, logger.infos)
        nrm = env._obs_normalizer
        out[tag + "_norm_mean"], out[tag + "_norm_var"] = nrm._mean.copy(), nrm._var.copy()
        out[tag + "_norm_count"] = np.array(nrm._count)

    # ---- Normalizer and quantile loss (test_numpy_oracle_pieces_against_reference_functions)
    from torchrl.env.base_wrapper import Normalizer
    import torchrl.algo.utils as atu
    rs = np.random.RandomState(0)
    ref = Normalizer((5,))
    filts = []
    for _ in range(4):
        x = rs.randn(9, 5) * 3 + 1
        ref.update_estimate(x)
        filts.append(ref.filt(x))
    out.update(pieces_filt=np.array(filts), pieces_mean=ref._mean.copy(), pieces_var=ref._var.copy())
    tau = (2 * np.arange(7) + 1) / 14.0
    src, tgt = rs.randn(6, 7), rs.randn(6, 7)
    out["pieces_qr"] = np.array(atu.quantile_regression_loss(torch.tensor(tau).view(1, -1), torch.tensor(src),
                                                             torch.tensor(tgt)).item())

    # ---- TwinSAC-Q / TD3 / DDPG updates on explicit batches
    import gym
    from torchrl.algo import TwinSACQ, TD3
    from torchrl.algo.off_policy.ddpg import DDPG
    o, a, hidden, B, seed = tv.OFF_CASE
    batches = tv._offpolicy_batches(o, a, B, 4, seed)

    class FakeEnv:
        action_space = gym.spaces.Box(-np.ones(a), np.ones(a))
        observation_space = gym.spaces.Box(-np.ones(o), np.ones(o))

    class FakeCollector:
        epoch_frames = 1
    common = dict(env=FakeEnv(), replay_buffer=None, collector=FakeCollector(), logger=None, discount=0.99,
                  batch_size=B, device="cpu", save_dir=tmp, tau=0.005, use_soft_update=True)
    for kind in ("sac", "td3", "ddpg"):
        torch.manual_seed(seed)
        net = dict(hidden_shapes=list(hidden), append_hidden_shapes=[], base_type=networks.MLPBase,
                   activation_func=torch.nn.ReLU)
        if kind == "sac":
            pf = policies.GuassianContPolicy(input_shape=o, output_shape=2 * a, tanh_action=True, **net)
        elif kind == "td3":
            pf = policies.FixGuassianContPolicy(input_shape=o, output_shape=a, tanh_action=True, norm_std_explore=0.1,
                                                **net)
        else:
            pf = policies.DetContPolicy(input_shape=o, output_shape=a, tanh_action=True, **net)
        if kind == "ddpg":
            qf = networks.QNet(input_shape=o + a, output_shape=1, **net)
            agent = DDPG(pf=pf, qf=qf, plr=1e-3, qlr=1e-3, **common)
        else:
            qf1 = networks.QNet(input_shape=o + a, output_shape=1, **net)
            qf2 = networks.QNet(input_shape=o + a, output_shape=1, **net)
            if kind == "sac":
                agent = TwinSACQ(pf=pf, qf1=qf1, qf2=qf2, plr=3e-4, qlr=3e-4, policy_std_reg_weight=1e-3,
                                 policy_mean_reg_weight=1e-3, **common)
            else:
                agent = TD3(pf=pf, qf1=qf1, qf2=qf2, plr=1e-3, qlr=1e-3, **common)
            torch.manual_seed(100)
        _store_infos(out, kind, [agent.update(b) for b in batches])
        _store_params(out, kind, [p.detach().numpy().copy() for n_ in agent.networks for p in n_.parameters()])

    # ---- Logger files (test_logger_files_match_reference)
    from torchrl.utils.logger import Logger
    rs = np.random.RandomState(0)
    updates, epochs = tv._logger_inputs(rs)
    lg = Logger("exp", "SynthHalfCheetah-v0", 3, tv._logger_params(), log_dir=os.path.join(tmp, "log"))
    for e in range(3):
        for info in updates[e]:
            lg.add_update_info(info)
        lg.add_epoch_info(e, (e + 1) * 4096, 1.5 * (e + 1), epochs[e])
    lg.finish()
    d = os.path.join(tmp, "log", "exp", "SynthHalfCheetah-v0", "3")
    out["logger_csv"] = np.array(open(os.path.join(d, "log.csv")).read())
    out["logger_params"] = np.array(open(os.path.join(d, "params.json")).read())

    # ---- Networks / policies: parameters and forward outputs (test_networks_and_policies_...)
    import torchrl.networks as rnet
    import torchrl.policies as rpol
    nets = tv._build_nets(rnet, rpol, 7)
    digests = {name: [[k, tv._digest(v.detach().numpy())] for k, v in m.state_dict().items()] for name, m in nets}
    out["nets_state"] = _json(digests)
    for name, y in tv._forward_nets(nets):
        out["nets_out_" + name + "_n"] = np.array(len(y))
        for i, v in enumerate(y):
            out["nets_out_%s_%d" % (name, i)] = v.numpy()

    # ---- RLAlgo.train bookkeeping (test_train_loop_bookkeeping_matches_reference)
    from torchrl.algo.rl_algo import RLAlgo
    col, log = tv._BookCol(), tv._BookLog()
    algo = tv._instrument(RLAlgo)(env=tv._BookEnv(), replay_buffer=None, collector=col, logger=log, num_epochs=7,
                                  batch_size=64, device="cpu", save_interval=3, eval_interval=2,
                                  save_dir=os.path.join(tmp, "r"))
    algo.snaps, algo.updates = [], 0
    algo.train()
    out["train_loop"] = _json({"snaps": algo.snaps, "updates": algo.updates, "evals": col.e, "rows": log.rows,
                               "episode_rewards": [float(x) for x in algo.episode_rewards],
                               "training_episode_rewards": [float(x) for x in algo.training_episode_rewards],
                               "best_eval": float(algo.best_eval)})

    # ---- Command-line flags (test_command_line_flags_match_reference)
    # `cuda` depends on the machine the flags are parsed on: record both answers of torch.cuda.is_available()
    from torchrl.utils.args import get_args
    saved = sys.argv, torch.cuda.is_available
    try:
        for avail in (False, True):
            torch.cuda.is_available = lambda: avail
            flags = []
            for argv in tv.ARGVS:
                sys.argv = ["prog"] + argv
                flags.append(vars(get_args()))
            out["args_cuda%d" % avail] = _json(flags)
    finally:
        sys.argv, torch.cuda.is_available = saved

    # ---- algo/utils.py (test_algo_utils_match_reference)
    torch.manual_seed(0)
    x = torch.randn(64) * 2
    out.update(utils_huber=atu.huber(x).numpy(), utils_huber_03=atu.huber(x, 0.3).numpy())
    for dt in (torch.float32, torch.float64):
        tau = ((2 * torch.arange(9) + 1) / 18.0).to(dt)
        s, t = torch.randn(5, 9, dtype=dt), torch.randn(5, 9, dtype=dt)
        out["utils_qr_" + str(dt)[6:]] = atu.quantile_regression_loss(tau, s, t).numpy()
    src, tgt, _ = tv._utils_nets()
    for _ in range(3):
        atu.soft_update_from_to(src, tgt, 0.005)
    _store_params(out, "utils_soft", [p.detach().numpy().copy() for p in tgt.parameters()])
    opt = torch.optim.Adam(tgt.parameters(), lr=1.0)
    lrs = []
    for epoch in (0, 17, 487):
        atu.update_linear_schedule(opt, epoch, 488, 3e-4)
        lrs.append(opt.param_groups[0]["lr"])
    out["utils_lrs"] = np.array(lrs, dtype=np.float64)

    # ---- epsilon-greedy exploration (test_epsilon_greedy_policy_matches_reference)
    torch.manual_seed(0)
    qf = torch.nn.Linear(5, 4)
    pol = rpol.EpsilonGreedyDQNDiscretePolicy(qf=qf, start_epsilon=1.0, end_epsilon=0.1, decay_frames=20, action_shape=4)
    obs = torch.randn(30, 1, 5)
    np.random.seed(3)
    acts, eps = [], []
    for ob in obs:
        acts.append(np.asarray(pol.explore(ob)["action"]).copy())
        eps.append(pol.epsilon)
    out.update(egreedy_acts=np.array(acts), egreedy_eps=np.array(eps, dtype=np.float64), egreedy_count=np.array(pol.count))

    # ---- host VecEnv over the gym wrapper chain (test_host_vecenv_and_wrapper_chain_match_reference)
    from torchrl.env.get_env import get_single_env
    from torchrl.env.vecenv import VecEnv
    for adt in (np.float32, np.float64):
        tag = "vecenv_" + np.dtype(adt).name
        env = VecEnv(tv.VEC_N, get_single_env, ["SynthHalfCheetah-v0", dict(tv.VEC_PARAM)])
        for e in env.envs:
            tv._shorten(e)
        env.seed(9)
        out[tag + "_reset"] = env.reset()
        rs = np.random.RandomState(1)
        steps = {"obs": [], "rew": [], "done": [], "time_limit": [], "reset_rows": []}
        for t in range(tv.VEC_T):
            o_, r_, d_, i_ = env.step(rs.uniform(-1.4, 1.4, size=(tv.VEC_N, 6)).astype(adt))
            # copies: partial_reset writes the reset rows into the arrays step() returned
            steps["obs"].append(o_.copy()); steps["rew"].append(r_.copy()); steps["done"].append(d_.copy())
            steps["time_limit"].append(np.array(i_["time_limit"]))
            steps["reset_rows"].append(env.partial_reset(d_.squeeze(-1)) if d_.any() else np.zeros_like(o_))
            if t == 8:
                env.eval()
        for k, v in steps.items():
            out["%s_%s" % (tag, k)] = np.array(v)
    np.savez_compressed(os.path.join(GOLDEN, "reference_pins.npz"), **out)
    print("reference_pins.npz:", len(out), "arrays")


def golden_onpolicy(trl):
    """A2C, V-MPO and TRPO updates of the reference agents on explicit batches: initial weights, logged scalars and
    parameters after each update (tests/test_onpolicy_algos.py)."""
    import tempfile
    import torch
    import gym
    import torchrl.networks as networks
    import torchrl.policies as policies
    from torchrl.algo import A2C, TRPO, VMPO
    from tests import test_onpolicy_algos as ta
    out = {}

    class Env:
        action_space = gym.spaces.Box(-np.ones(ta.A), np.ones(ta.A))
        observation_space = gym.spaces.Box(-np.ones(ta.O), np.ones(ta.O))

    def agent(kind):
        torch.manual_seed(3)
        net = dict(hidden_shapes=list(ta.HID), append_hidden_shapes=[], base_type=networks.MLPBase,
                   activation_func=torch.nn.Tanh)
        pf = policies.GuassianContPolicyBasicBias(input_shape=ta.O, output_shape=ta.A, tanh_action=True, **net)
        vf = networks.Net(input_shape=(ta.O,), output_shape=1, **net)
        cls = {"a2c": A2C, "vmpo": VMPO, "trpo": TRPO}[kind]
        ag = cls(pf=pf, vf=vf, env=Env(), replay_buffer=None, collector=ta._Col(), logger=ta._NullLogger(),
                 discount=0.99, num_epochs=10, batch_size=64, gae=True, device="cpu", save_dir=tempfile.mkdtemp(),
                 shuffle=True, tau=0.95, **ta.KW[kind])
        return ag

    def params(tag, ag, names=("pf", "vf")):
        for k, v in ta._params(ag, names).items():
            out["%s_%s" % (tag, k)] = v.astype(np.float32)          # the nets' own dtype: exact

    params("init", agent("a2c"))

    for kind, seed in (("a2c", 0), ("vmpo", 1)):
        ag = agent(kind)
        assert all(np.array_equal(v, out["init_" + k]) for k, v in ta._params(ag).items())
        _store_infos(out, kind, [ag.update(b) for b in ta._batches(4, 64, seed)])
        params(kind + "_final", ag)
        if kind == "vmpo":
            out["vmpo_dual"] = np.array([float(ag.eta), float(ag.alpha)])
    for lead in ta.TRPO_LEADS:
        tag = "trpo_%s" % ("flat" if lead is None else "x".join(map(str, lead)))
        ag = agent("trpo")
        assert all(np.array_equal(v, out["init_" + k]) for k, v in ta._params(ag).items())
        batches = ta._batches(2, 128, 2, lead)
        for i, b in enumerate(batches):          # actions the initial policy could have produced
            with torch.no_grad():
                o = torch.as_tensor(b["obs"], dtype=torch.float32)
                mean, std, _ = ag.pf(o)
                b["acts"] = torch.tanh(mean + std * torch.randn_like(mean)).numpy().astype(np.float64)
            out["%s_acts%d" % (tag, i)] = b["acts"]
        for i, b in enumerate(batches):
            _store_infos(out, "%s_u%d" % (tag, i), [ag.update(b)])
            params("%s_u%d" % (tag, i), ag, ("pf",))
        for i, b in enumerate(batches):
            fb = dict(obs=b["obs"].reshape(-1, ta.O), estimate_returns=b["estimate_returns"].reshape(-1, 1))
            _store_infos(out, "%s_v%d" % (tag, i), [ag.update_vf(fb)])
        params(tag + "_final", ag, ("vf",))
    np.savez_compressed(os.path.join(GOLDEN, "onpolicy_algos.npz"), **out)
    print("onpolicy_algos.npz:", len(out), "arrays")


def main():
    from oracle import reference_loader
    trl = reference_loader.load()
    os.makedirs(GOLDEN, exist_ok=True)
    only = sys.argv[1:]
    for name, fn in sorted(globals().items()):
        if name.startswith("golden_") and callable(fn):
            if only and name[len("golden_"):] not in only:
                continue
            fn(trl)


if __name__ == "__main__":
    main()
