"""The REFERENCE'S OWN example scripts, byte-for-byte as oracle/build_ref.py copied them to oracle/_ref/examples,
run end to end on the device path: `import torchrl...` resolves to compat/torchrl (an alias of torchrl_b200), `import gym`
to compat/gym, the JSON configs name a synthetic device env.  This is the drop-in boundary of SURVEY.md 8(b) exercised
the way a user of the reference would: nothing in the script changes, only what `torchrl` means.

Skipped when oracle/_ref is absent (python oracle/build_ref.py creates it where /root/reference is mounted)."""
import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_EXAMPLES = os.path.join(ROOT, "oracle", "_ref", "examples")

needs_ref = pytest.mark.skipif(not os.path.isdir(REF_EXAMPLES), reason="oracle/_ref not built")


def _run_reference_example(script, cfg_name, patch, nenv, tmp_path, extra_check=None):
    path = os.path.join(REF_EXAMPLES, script)
    src_ref = os.path.join("/root/reference/examples", script)
    if os.path.exists(src_ref):                               # where the mount exists: prove the copy is verbatim
        assert hashlib.sha1(open(path, "rb").read()).hexdigest() == hashlib.sha1(open(src_ref, "rb").read()).hexdigest()
    cfg = json.load(open(os.path.join(ROOT, "config", cfg_name)))
    patch(cfg)
    cfg_path = tmp_path / cfg_name
    json.dump(cfg, open(cfg_path, "w"))
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "compat"), ROOT, env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, path, "--config", str(cfg_path), "--vec_env_nums", str(nenv), "--seed", "1",
                        "--log_dir", str(tmp_path / "log"), "--overwrite"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    work = tmp_path / "log" / os.path.splitext(cfg_name)[0] / cfg["env_name"] / "1"
    assert (work / "log.csv").exists() and (work / "params.json").exists(), os.listdir(tmp_path)
    rows = open(work / "log.csv").read().strip().splitlines()
    assert len(rows) >= 2, rows
    return work, rows[0]


def _small_on_policy(c, key, n=64):
    c["replay_buffer"]["size"] = n * 16
    c["collector"].update(epoch_frames=n * 16, max_episode_frames=40)
    c["general_setting"].update(num_epochs=3, batch_size=n * 4, eval_interval=2, save_interval=2)
    c["net"]["hidden_shapes"] = [32, 32]
    c[key].update(c[key])


def _small_off_policy(c, n=32):
    c["replay_buffer"]["size"] = n * 64
    c["collector"].update(epoch_frames=n * 8, max_episode_frames=30)
    c["general_setting"].update(num_epochs=2, batch_size=n * 4, opt_times=5, eval_interval=1, save_interval=1, pretrain_epochs=1)
    c["net"]["hidden_shapes"] = [32, 32]


@pytest.mark.gpu
@needs_ref
def test_reference_ppo_example_runs_unmodified(tmp_path):
    def patch(c):
        _small_on_policy(c, "ppo")
        c["ppo"]["opt_epochs"] = 2
    work, header = _run_reference_example("ppo_continuous_vec.py", "ppo_synth_halfcheetah.json", patch, 64, tmp_path)
    files = set(os.listdir(work / "model"))
    for f in ("model_pf_best.pth", "model_vf_0.pth", "model_pf_finish.pth", "_obs_normalizer_finish.pkl"):
        assert f in files, files
    for key in ("Train_Epoch_Reward", "Training/policy_loss_Mean", "grad_norm/pf_Max", "eval_traj_length"):
        assert key in header, header


@pytest.mark.gpu
@needs_ref
def test_reference_twin_sac_q_example_runs_unmodified(tmp_path):
    work, header = _run_reference_example("twin_sac_q_continuous_vec.py", "twin_sac_q_synth_ant.json", _small_off_policy, 32,
                                           tmp_path)
    files = set(os.listdir(work / "model"))
    assert "model_qf1_finish.pth" in files and "model_pf_best.pth" in files
    assert "Alpha_Mean" in header


@pytest.mark.gpu
@needs_ref
def test_reference_td3_example_runs_unmodified(tmp_path):
    work, header = _run_reference_example("td3_continuous_vec.py", "td3_synth_halfcheetah.json", _small_off_policy, 32,
                                           tmp_path)
    assert "model_qf2_finish.pth" in set(os.listdir(work / "model"))
    assert "Training/qf1_loss_Mean" in header, header


@pytest.mark.gpu
@needs_ref
def test_reference_ddpg_example_runs_unmodified(tmp_path):
    work, header = _run_reference_example("ddpg_continuous_vec.py", "ddpg_synth_halfcheetah.json", _small_off_policy, 32,
                                           tmp_path)
    assert "model_qf_finish.pth" in set(os.listdir(work / "model"))


@pytest.mark.gpu
@needs_ref
def test_reference_a2c_example_runs_unmodified(tmp_path):
    def patch(c):
        _small_on_policy(c, "a2c")
    work, header = _run_reference_example("a2c_continuous_vec.py", "a2c_synth_halfcheetah.json", patch, 64, tmp_path)
    assert "Training/vf_loss_Mean" in header, header


def test_alias_package_resolves_to_the_product(tmp_path):
    """CPU: `import torchrl.<sub>` through compat/ yields the torchrl_b200 module objects themselves."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import torchrl, torchrl_b200, gym\n"
            "import torchrl.policies as p, torchrl.networks as n\n"
            "from torchrl.collector.on_policy import VecOnPolicyCollector\n"
            "from torchrl.replay_buffers.on_policy import OnPolicyReplayBuffer\n"
            "from torchrl.utils import get_args, get_params, Logger\n"
            "from torchrl.algo import PPO, TD3, TwinSACQ, DDPG, A2C\n"
            "from torchrl.env import get_vec_env\n"
            "import torchrl_b200.policies, torchrl_b200.algo\n"
            "assert p is torchrl_b200.policies and PPO is torchrl_b200.algo.PPO\n"
            "assert gym.spaces.Box is __import__('torchrl_b200.spaces', fromlist=['Box']).Box\n"
            "print('alias ok')\n" % (ROOT, os.path.join(ROOT, "compat")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert r.returncode == 0 and "alias ok" in r.stdout, r.stdout + r.stderr
