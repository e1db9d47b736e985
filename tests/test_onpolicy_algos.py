"""A2C, V-MPO and TRPO on the device against the reference (torch CPU): the reference's agents were run on the
explicit batches below through `update(batch)` -- the reference's own entry point -- and their initial weights, the
logged scalars of every update and the parameters after the updates are stored in tests/golden/onpolicy_algos.npz
(`python -m oracle.make_golden onpolicy` regenerates it where the reference is importable).  The device agents start
from the stored weights, take the same batches and must reproduce the stored scalars and parameters.  SURVEY.md 8(f).4.

Stated tolerances (fp32 device kernels vs torch-CPU fp32): logged scalars rtol 2e-3 + atol 2e-4 (TRPO policy loss /
KL-driven quantities 5e-3), parameters atol 2e-4 (TRPO: 1e-3 of the step, the conjugate-gradient solve amplifies
rounding).  The device epoch loop (captured graphs) is checked against the eager `update` path of the same agent.
"""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

O, A, HID = 11, 3, (32, 32)
KW = {"a2c": dict(plr=1e-3, vlr=1e-3, entropy_coeff=0.01),
      "vmpo": dict(plr=1e-3, vlr=1e-3, opt_epochs=2, alpha_eps=0.01),
      "trpo": dict(plr=3e-4, vlr=1e-3, max_kl=0.01, cg_damping=0.1, cg_iters=10, residual_tol=1e-10, entropy_coeff=0.01,
                   v_opt_times=2)}
TRPO_LEADS = [None, (8, 16)]


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(os.path.join(golden_dir, "onpolicy_algos.npz"))


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


class _Col:
    epoch_frames = 64


def _batches(n, B, seed, lead=None):
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        shape = (B,) if lead is None else lead
        obs = rs.randn(*shape, O)
        acts = np.tanh(0.4 * rs.randn(*shape, A))
        out.append(dict(obs=obs, acts=acts, advs=rs.randn(*shape, 1), estimate_returns=rs.randn(*shape, 1),
                        values=rs.randn(*shape, 1)))
    return out


def _stored(g, tag, names=("pf", "vf")):
    """{net.key: array} of what _params() returned for the reference agent at `tag`."""
    pre = tag + "_"
    return {k[len(pre):]: g[k].astype(np.float64) for k in g.files
            if k.startswith(pre) and k[len(pre):].split(".")[0] in names}


def _stored_infos(g, tag):
    return json.loads(str(g[tag + "_infos"]))


def _load(net, params, name):
    import torch
    net.load_state_dict({k[len(name) + 1:]: torch.from_numpy(v) for k, v in params.items() if k.startswith(name + ".")})


def _device_agent(kind, init):
    import torch
    import torchrl_b200.networks as networks
    import torchrl_b200.policies as policies
    from torchrl_b200.algo import A2C, TRPO, VMPO
    from torchrl_b200.spaces import Box

    class Env:
        action_space = Box(-np.ones(A), np.ones(A))
        observation_space = Box(-np.ones(O), np.ones(O))
    net = dict(hidden_shapes=list(HID), append_hidden_shapes=[], base_type=networks.MLPBase, activation_func=torch.nn.Tanh)
    pf = policies.GuassianContPolicyBasicBias(input_shape=O, output_shape=A, tanh_action=True, **net)
    vf = networks.Net(input_shape=(O,), output_shape=1, **net)
    _load(pf, init, "pf")
    _load(vf, init, "vf")
    cls = {"a2c": A2C, "vmpo": VMPO, "trpo": TRPO}[kind]
    return cls(pf=pf, vf=vf, env=Env(), replay_buffer=None, collector=_Col(), logger=_NullLogger(), discount=0.99,
               num_epochs=10, batch_size=64, gae=True, device="cuda:0", save_dir=None, shuffle=True, tau=0.95,
               use_cuda_graph=False, **KW[kind])


def _params(agent, names=("pf", "vf")):
    import torch
    out = {}
    for n in names:
        for k, v in getattr(agent, n).state_dict().items():
            out[n + "." + k] = v.detach().cpu().numpy().astype(np.float64)
    return out


def _compare_infos(mine, ref, rtol=2e-3, atol=2e-4, skip=()):
    assert len(mine) == len(ref)
    for u, (m, r) in enumerate(zip(mine, ref)):
        assert set(r.keys()) <= set(m.keys()), (sorted(r.keys()), sorted(m.keys()))
        for k, v in r.items():
            if k in skip:
                continue
            assert abs(m[k] - v) <= rtol * abs(v) + atol, (u, k, m[k], v)


def test_a2c_update_matches_reference(g):
    mine = _device_agent("a2c", _stored(g, "init"))
    batches = _batches(4, 64, 0)
    m_infos = [mine.update(b) for b in batches]
    _compare_infos(m_infos, _stored_infos(g, "a2c"))
    pr, pm = _stored(g, "a2c_final"), _params(mine)
    assert pr.keys() == pm.keys()
    for k in pr:
        np.testing.assert_allclose(pm[k], pr[k], atol=2e-4, err_msg=k)


def test_vmpo_update_matches_reference(g):
    mine = _device_agent("vmpo", _stored(g, "init"))
    batches = _batches(4, 64, 1)
    m_infos = [mine.update(b) for b in batches]
    _compare_infos(m_infos, _stored_infos(g, "vmpo"))
    pr, pm = _stored(g, "vmpo_final"), _params(mine)
    assert pr.keys() == pm.keys()
    for k in pr:
        np.testing.assert_allclose(pm[k], pr[k], atol=2e-4, err_msg=k)
    eta, alpha = g["vmpo_dual"]
    assert abs(float(mine.dual[0]) - eta) < 2e-4 and abs(float(mine.dual[1]) - alpha) < 2e-4


@pytest.mark.parametrize("lead", TRPO_LEADS)
def test_trpo_update_matches_reference(g, lead):
    """Flat (B, .) batches (per-sample KL) and the (T, N, .) whole-rollout form the reference's update_per_epoch
    passes (its KL sums over the env axis: the N / act_dim quirk)."""
    tag = "trpo_%s" % ("flat" if lead is None else "x".join(map(str, lead)))
    mine = _device_agent("trpo", _stored(g, "init"))
    # actions the policy could have produced (log-probs of arbitrary actions underflow exp() in the reference's ratio)
    batches = _batches(2, 128, 2, lead)
    for i, b in enumerate(batches):
        b["acts"] = g["%s_acts%d" % (tag, i)]
    p0 = _stored(g, "init", ("pf",))
    for i, b in enumerate(batches):
        m_info = mine.update(b)
        _compare_infos([m_info], _stored_infos(g, "%s_u%d" % (tag, i)), rtol=5e-3, atol=5e-4)
        pr, pm = _stored(g, "%s_u%d" % (tag, i), ("pf",)), _params(mine, ("pf",))
        assert pr.keys() == pm.keys()
        step = max(np.abs(pr[k] - p0[k]).max() for k in pr)
        assert step > 1e-5, "the reference took no step: the test would be vacuous"
        for k in pr:
            np.testing.assert_allclose(pm[k], pr[k], atol=2e-2 * step + 1e-5, err_msg=k)
        # continue both from the SAME parameters so that one update's rounding does not leak into the next
        _load(mine.pf, pr, "pf")
        p0 = pr
    flat = [dict(obs=b["obs"].reshape(-1, O), estimate_returns=b["estimate_returns"].reshape(-1, 1)) for b in batches]
    for i, b in enumerate(flat):
        m_info = mine.update_vf(b)
        _compare_infos([m_info], _stored_infos(g, "%s_v%d" % (tag, i)))
    pr, pm = _stored(g, tag + "_final", ("vf",)), _params(mine, ("vf",))
    assert pr.keys() == pm.keys()
    for k in pr:
        np.testing.assert_allclose(pm[k], pr[k], atol=2e-4, err_msg=k)


@pytest.mark.parametrize("kind", ["a2c", "vmpo", "trpo"])
def test_epoch_loop_graph_path_equals_eager_path(kind):
    """collector -> update_per_epoch with CUDA graphs == the same with eager launches (buffers, parameters, infos)."""
    import torch
    import torchrl_b200.networks as networks
    import torchrl_b200.policies as policies
    from torchrl_b200.algo import A2C, TRPO, VMPO
    from torchrl_b200.collector import VecOnPolicyCollector
    from torchrl_b200.env import get_vec_env
    from torchrl_b200.replay_buffers import OnPolicyReplayBuffer
    runs = []
    for use_graph in (False, True):
        N, T = 64, 16
        env = get_vec_env("SynthHalfCheetah-v0", {"reward_scale": 1, "obs_norm": True}, N)
        eval_env = get_vec_env("SynthHalfCheetah-v0", {"reward_scale": 1, "obs_norm": True}, N)
        env.seed(5); torch.manual_seed(5); np.random.seed(5)
        buf = OnPolicyReplayBuffer(env_nums=N, max_replay_buffer_size=T * N, time_limit_filter=True)
        net = dict(hidden_shapes=[32, 32], append_hidden_shapes=[], base_type=networks.MLPBase, activation_func=torch.nn.Tanh)
        pf = policies.GuassianContPolicyBasicBias(input_shape=17, output_shape=6, tanh_action=True, **net)
        vf = networks.Net(input_shape=(17,), output_shape=1, **net)
        col = VecOnPolicyCollector(vf, env=env, eval_env=eval_env, pf=pf, replay_buffer=buf, device="cuda:0",
                                   epoch_frames=T * N, max_episode_frames=40, use_cuda_graph=use_graph)
        common = dict(pf=pf, vf=vf, env=env, replay_buffer=buf, collector=col, logger=_NullLogger(), discount=0.99,
                      num_epochs=10, batch_size=4 * N, gae=True, device="cuda:0", save_dir=None, shuffle=True, tau=0.95,
                      use_cuda_graph=use_graph, plr=3e-4, vlr=3e-4)
        if kind == "a2c":
            agent = A2C(entropy_coeff=0.01, **common)
        elif kind == "vmpo":
            agent = VMPO(opt_epochs=3, alpha_eps=0.01, **common)
        else:
            agent = TRPO(max_kl=0.01, cg_damping=0.1, cg_iters=10, residual_tol=1e-10, entropy_coeff=0.01, v_opt_times=3,
                         **common)
        for epoch in range(3):                      # the graphs are captured after three eager minibatches
            agent.current_epoch = epoch
            col.train_one_epoch()
            agent.update_per_epoch()
        runs.append((agent.opt.data.clone(), [dict(i) for i in agent._last_infos]))
        assert all(np.isfinite(v) for i in agent._last_infos for v in i.values())
    (p0, i0), (p1, i1) = runs
    torch.testing.assert_close(p0, p1, rtol=1e-3, atol=2e-5)
    assert len(i0) == len(i1) and len(i0) > 0
    for d0, d1 in zip(i0, i1):
        for k in d0:
            assert abs(d0[k] - d1[k]) <= 2e-3 * max(1.0, abs(d0[k])), (k, d0[k], d1[k])
