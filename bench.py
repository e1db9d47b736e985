#!/usr/bin/env python
"""bench.py -- env-steps/sec of the PPO hot path (rollout + GAE + update) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one PPO epoch of BASELINE.json configs[1]: 4096 synthetic HalfCheetah-shaped envs per
GPU (obs 17, act 6), horizon 128, MLP(256,256) policy and value nets, 10 optimisation passes of
32 minibatches (4 time-rows x all envs = 16384 samples per GPU): 524288 env-steps per GPU per step.
With N > 1 every rank owns 4096 envs (weak scaling; configs[4] at N = 8) and the flat pf|vf
gradient is all-reduced over NCCL once per minibatch.

Prints ONE JSON line (rank 0).  `value` = device-timed (CUDA events, max over ranks) throughput
with the host out of the loop (no per-epoch read-backs); `e2e` = the same metric through the
public collector/agent API, wall-clock, including every host->device (minibatch row order,
learning rates) and device->host (per-update logged scalars, episode returns) copy.
`--impl reference` times the reference's own CPU implementation of the same workload on the box's host cores:
the unmodified reference classes from oracle/_ref (oracle/build_ref.py copies them there; git-ignored), whole
epochs timed end to end (oracle/ref_port.py only if no copy of the reference is present).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ENVS_PER_GPU = 4096
HORIZON = 128
HIDDEN = (256, 256)
BATCH_ROWS = 4
OPT_EPOCHS = 10
OBS_DIM, ACT_DIM = 17, 6
ENV_ID = "SynthHalfCheetah-v0"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=N_ENVS_PER_GPU)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true",
                    help="skip the secondary measurements (BASELINE configs[0], [2], [3] and the desynchronised-episode PPO)")
    ap.add_argument("--cpu-procs", type=int, default=0, help="env worker processes of the CPU arm (0 = auto)")
    ap.add_argument("--cpu-budget-s", type=float, default=600.0,
                    help="wall-clock budget of the CPU arm; whole epochs are dropped (never shortened) beyond it")
    ap.add_argument("--matmul", default="tc3", choices=["fp32", "tf32x3", "tc3"],
                    help="MLP GEMM path: tc3 = hand-written tcgen05 3xTF32 kernel on the 256-wide layers (default), fp32 = cuBLAS SIMT everywhere, tf32x3 = 3 cuBLAS TF32 GEMMs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last device-timed step computed (rollout sample, "
                         "advantages, returns, normaliser state, parameters, logged scalars) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clocks and throttle reasons DURING the timed region, sampled through NVML from a thread of this process
    (pynvml: nvmlDeviceGetClockInfo / nvmlDeviceGetCurrentClocksEventReasons, every 100 ms).

    Round 1 polled with an `nvidia-smi -lms` child process; even when started before the warm-up it made the
    device-timed leg bistable -- 88 vs 120-127 ms/step at 2 GPUs in one run out of three, never without the poller
    (gpurun_out/bench_n2_{default,nofork,noclocks,...}.txt, round 2) -- because a stalled launch thread on one rank
    stalls every rank at the next collective.  The in-process NVML queries take microseconds and spawn nothing; the
    child-process poller remains only as a fallback when pynvml is missing."""
    _REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.t0 = self.t1 = None
        self.samples = []                    # (time, sm_mhz, sm_max_mhz, reason mask)
        self._stop = False
        self._thread = None
        self.proc = None
        self.path = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def _loop(self, nv, handle):
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(handle))
                self.samples.append((time.time(), float(sm), float(mx), mask))
            except Exception:                               # noqa: BLE001 -- a failed query is a missing sample
                pass
            time.sleep(0.1)

    def start(self):
        if self.gpu is None:
            return
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            handle = nv.nvmlDeviceGetHandleByIndex(self._physical_index())
            self._thread = threading.Thread(target=self._loop, args=(nv, handle), daemon=True)
            self._thread.start()
            return
        except Exception:                                   # noqa: BLE001
            self._thread = None
        try:
            self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:                                   # noqa: BLE001
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    @staticmethod
    def _stamp(text):
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def _read_child(self):
        """Samples of the fallback nvidia-smi child process -> self.samples."""
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:                                   # noqa: BLE001
            self.proc.kill()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 10:
                    continue
                try:
                    clk, cmax = float(f[2]), float(f[3])
                except ValueError:
                    continue
                mask = 0
                for (bit, _), val in zip(self._REASONS, f[6:10]):
                    if val.lower().startswith("active"):
                        mask |= bit
                self.samples.append((self._stamp(f[0]) or 0.0, clk, cmax, mask))
        except OSError:
            pass
        try:
            os.unlink(self.path)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "how": None}
        if self._thread is not None:
            self._stop = True
            self._thread.join(timeout=2)
            out["how"] = "nvml thread, 100 ms"
        elif self.proc is not None:
            self._read_child()
            out["how"] = "nvidia-smi -lms 200"
        else:
            return out
        inside = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1 + 0.05]
        rows = inside or self.samples                       # no stamped sample inside the region: keep them all
        if rows:
            sm = sorted(x[1] for x in rows)
            mask = 0
            for x in rows:
                mask |= x[3]
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(x[2] for x in rows),
                       reasons=sorted(name for bit, name in self._REASONS if mask & bit), samples=len(rows))
        return out


# ----------------------------------------------------------------------------------------- CPU arm
def workload_string(envs_per_gpu, world):
    """The ONE description of the workload, printed identically by both arms."""
    return ("PPO SynthHalfCheetah-v0 (obs 17, act 6), %d envs/GPU x %d GPU, horizon %d, MLP%s, minibatch %d/GPU, "
            "%d opt epochs (BASELINE.json configs[%d])"
            % (envs_per_gpu, world, HORIZON, list(HIDDEN), BATCH_ROWS * envs_per_gpu, OPT_EPOCHS, 1 if world == 1 else 4))


class _NullLogger:
    def add_update_info(self, info):
        pass

    def add_epoch_info(self, *a, **k):
        pass

    def log(self, *a):
        pass

    def finish(self):
        pass


class CpuPipeline:
    """The reference's own CPU path for this workload, whole epochs at a time:
        collector.train_one_epoch()   T vec-env steps through SubProcVecEnv worker processes (+ NormObs, policy and
                                      value forward per step)                         collector/on_policy.py:90-153
        agent.update_per_epoch()      Python GAE loop + opt_epochs x T/b torch-CPU minibatch updates   ppo.py:27-39
    `kind == "reference"`: the UNMODIFIED reference classes, imported from oracle/_ref (the copy oracle/build_ref.py
    makes; /root/reference in the build container) behind oracle/shims for the absent third-party modules, over the
    synthetic gym env of oracle/synth_env.py.  `kind == "port"`: oracle/ref_port.py (pinned bit-for-bit to the
    reference by tests/test_oracle_vs_reference.py) -- only when no copy of the reference is present."""

    def __init__(self, env_nums, proc_nums, threads, seed=0, horizon=HORIZON):
        import numpy as np
        import torch
        from oracle import reference_loader
        torch.set_num_threads(threads)
        assert horizon % BATCH_ROWS == 0
        self.env_nums, self.proc_nums, self.threads, self.horizon = env_nums, proc_nums, threads, horizon
        self.frames = horizon * env_nums
        if reference_loader.available():
            self.kind = "reference"
            reference_loader.load()
            import torchrl.networks as networks
            import torchrl.policies as policies
            from torchrl.algo import PPO
            from torchrl.collector.on_policy import VecOnPolicyCollector
            from torchrl.env import get_subprocvec_env, get_vec_env
            from torchrl.replay_buffers.on_policy import OnPolicyReplayBuffer
            params = {"reward_scale": 1, "obs_norm": True}
            if proc_nums > 1:
                env = get_subprocvec_env(ENV_ID, dict(params), env_nums, proc_nums)
                eval_env = get_vec_env(ENV_ID, dict(params), 1)     # never stepped here; the collector wants one
            else:
                env = get_vec_env(ENV_ID, dict(params), env_nums)
                eval_env = get_vec_env(ENV_ID, dict(params), 1)
            env.seed(seed)
            torch.manual_seed(seed)
            np.random.seed(seed)
            buf = OnPolicyReplayBuffer(env_nums=env_nums, max_replay_buffer_size=horizon * env_nums, time_limit_filter=True)
            net = dict(hidden_shapes=list(HIDDEN), append_hidden_shapes=[], base_type=networks.MLPBase,
                       activation_func=torch.nn.Tanh)
            pf = policies.GuassianContPolicyBasicBias(input_shape=OBS_DIM, output_shape=ACT_DIM, tanh_action=True, **net)
            vf = networks.Net(input_shape=(OBS_DIM,), output_shape=1, **net)
            col = VecOnPolicyCollector(vf, env=env, eval_env=eval_env, pf=pf, replay_buffer=buf, device="cpu",
                                       train_render=False, epoch_frames=horizon * env_nums, max_episode_frames=999,
                                       eval_episodes=1)
            self._tmp = tempfile.mkdtemp(prefix="bench_ref_")
            agent = PPO(pf=pf, vf=vf, plr=3e-4, vlr=3e-4, clip_para=0.2, opt_epochs=OPT_EPOCHS, tau=0.95, shuffle=True,
                        entropy_coeff=0.005, env=env, replay_buffer=buf, collector=col, logger=_NullLogger(),
                        discount=0.99, num_epochs=488, batch_size=BATCH_ROWS * env_nums, gae=True, device="cpu",
                        save_dir=self._tmp)
            self.env, self.eval_env, self.col, self.agent = env, eval_env, col, agent
        else:
            self.kind = "port"
            from oracle import ref_port
            env, col, agent = ref_port.build_ppo(env_id=ENV_ID, env_nums=env_nums, proc_nums=proc_nums, horizon=horizon,
                                                 hidden=HIDDEN, batch_rows=BATCH_ROWS, opt_epochs=OPT_EPOCHS, seed=seed)
            self.env, self.eval_env, self.col, self.agent = env, None, col, agent
        self.epochs_done = 0

    def epoch(self):
        """One WHOLE epoch, timed for real: returns (seconds, collect seconds, update seconds)."""
        self.agent.current_epoch = self.epochs_done
        t0 = time.perf_counter()
        self.col.train_one_epoch()
        t1 = time.perf_counter()
        self.agent.update_per_epoch()
        t2 = time.perf_counter()
        self.epochs_done += 1
        return t2 - t0, t1 - t0, t2 - t1

    def close(self):
        for e in (self.env, self.eval_env):
            try:
                if e is not None:
                    e.close()
            except Exception:
                pass

    def describe(self):
        s = ("%s: whole epochs timed end to end, each = %d vec-env steps x %d envs over %d env worker processes "
             "(SubProcVecEnv) + Python GAE + %d PPO minibatches of %d samples on %d torch threads"
             % ("unmodified reference classes (oracle/_ref)" if self.kind == "reference" else "oracle/ref_port.py",
                self.horizon, self.env_nums, self.proc_nums, OPT_EPOCHS * (self.horizon // BATCH_ROWS),
                BATCH_ROWS * self.env_nums, self.threads))
        if self.horizon != HORIZON:
            s += ("; BOUNDED SAMPLE: horizon %d instead of %d -- same env count, same minibatch size, same work per "
                  "collector step and per minibatch, %dx fewer of both per epoch, so env-steps/s is unchanged while an "
                  "epoch stays at ~1 GPU's worth of CPU work" % (self.horizon, HORIZON, HORIZON // self.horizon))
        return s


def auto_procs(env_nums, want=0):
    cores = os.cpu_count() or 1
    p = want or min(cores, 64)
    while p > 1 and env_nums % p:
        p -= 1
    return max(p, 1), cores


def best_torch_threads(cores, batch):
    """torch intra-op thread count that makes the CPU arm's PPO minibatch fastest on this host.  More threads is
    not monotonically better (all 128 hyper-threads of the GPU box are ~100x SLOWER than 32 for these GEMM sizes), so
    probe a few counts once and keep the best: the CPU arm gets the most favourable setting, not a pessimised one."""
    import torch
    import torch.nn as nn
    cands = sorted({c for c in (8, 16, 32, 64, cores // 2, cores) if 1 <= c <= cores})
    net = nn.Sequential(nn.Linear(OBS_DIM, HIDDEN[0]), nn.Tanh(), nn.Linear(HIDDEN[0], HIDDEN[1]), nn.Tanh(),
                        nn.Linear(HIDDEN[1], ACT_DIM))
    x = torch.randn(batch, OBS_DIM)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        for _ in range(2):
            net.zero_grad()
            t0 = time.perf_counter()
            net(x).square().mean().backward()
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:          # past the knee: larger counts only get worse
            break
    return best


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation on this box's host cores, same workload as our arm.
    Every step is one whole epoch timed for real (W untimed, then K timed); if the box is so slow that W + K epochs
    would exceed --cpu-budget-s, fewer are run and `steps` / `warmup` report what was actually done."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = max(args.gpus, 1)
    env_nums = args.envs_per_gpu * world                     # our arm's global env count at this N
    procs, cores = auto_procs(env_nums, args.cpu_procs)
    threads = best_torch_threads(cores, BATCH_ROWS * env_nums)
    t_start = time.perf_counter()
    # several GPUs' worth of envs: a whole 128-step epoch of the CPU pipeline would take world x ~35 s, and W + K of them
    # far more than "a few minutes"; the horizon of the timed epochs shrinks with the world size instead (see describe())
    horizon = HORIZON
    while horizon * world > HORIZON and horizon // 2 >= 4 * BATCH_ROWS:
        horizon //= 2
    pipe = CpuPipeline(env_nums, procs, threads, horizon=horizon)
    try:
        warm, timed, parts = 0, [], []
        for i in range(args.warmup):
            dt, _, _ = pipe.epoch()
            warm += 1
            left = args.cpu_budget_s - (time.perf_counter() - t_start)
            if left < dt * (2 + max(0, args.warmup - 1 - i)):      # keep room for >= 2 timed epochs
                break
        for i in range(args.steps):
            dt, tc, tu = pipe.epoch()
            timed.append(dt)
            parts.append((tc, tu))
            if len(timed) >= 2 and (time.perf_counter() - t_start) + dt > args.cpu_budget_s:
                break
    finally:
        pipe.close()
    k = len(timed)
    t_total = sum(timed)
    value = pipe.frames * k / t_total
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": k, "warmup": warm, "ms_per_step": t_total / k * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 nets / f64 buffers",
        "data": "synthetic",
        "config": {"workload": workload_string(args.envs_per_gpu, world), "global_envs": env_nums,
                   "parallelism": "cpu: %d env worker processes, %d torch threads" % (procs, threads)},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": max(procs, threads), "host_logical_cores": cores,
                         "kind": pipe.kind, "sample": pipe.describe() + "; %d warm-up + %d timed epochs" % (warm, k),
                         "detail": {"epoch_s": timed, "collect_s": [p[0] for p in parts], "update_s": [p[1] for p in parts],
                                    "requested_steps": args.steps, "requested_warmup": args.warmup}},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------- our arm
def build_agent(args, ctx, device):
    import numpy as np
    import torch
    import torchrl_b200.networks as networks
    import torchrl_b200.policies as policies
    from torchrl_b200.algo import PPO
    from torchrl_b200.collector import VecOnPolicyCollector
    from torchrl_b200.env import get_vec_env
    from torchrl_b200.replay_buffers import OnPolicyReplayBuffer
    from torchrl_b200.utils import NullLogger
    n_local = args.envs_per_gpu
    n_total = n_local * ctx.world_size
    first = ctx.rank * n_local
    params = {"reward_scale": 1, "obs_norm": True}
    env = get_vec_env(ENV_ID, params, n_local, device=device, first_env=first, total_envs=n_total)
    eval_env = get_vec_env(ENV_ID, params, n_local, device=device, first_env=first, total_envs=n_total)
    env.dist = ctx if ctx.active else None
    env.seed(0)
    torch.manual_seed(0)            # identical nets and identical minibatch row order on every rank
    np.random.seed(0)
    buf = OnPolicyReplayBuffer(env_nums=n_local, max_replay_buffer_size=HORIZON * n_local, time_limit_filter=True)
    net = dict(hidden_shapes=list(HIDDEN), append_hidden_shapes=[], base_type=networks.MLPBase,
               activation_func=torch.nn.Tanh)
    pf = policies.GuassianContPolicyBasicBias(input_shape=OBS_DIM, output_shape=ACT_DIM, tanh_action=True, **net)
    vf = networks.Net(input_shape=(OBS_DIM,), output_shape=1, **net)
    col = VecOnPolicyCollector(vf, env=env, eval_env=eval_env, pf=pf, replay_buffer=buf, device=device,
                               train_render=False, epoch_frames=HORIZON * n_local, max_episode_frames=999,
                               eval_episodes=1, use_cuda_graph=not args.no_graph)
    if ctx.active:
        # decorrelate exploration noise across ranks (different envs, different Philox streams)
        pf._rng_state(device).seed += 7919 * ctx.rank
    agent = PPO(pf=pf, vf=vf, plr=3e-4, vlr=3e-4, clip_para=0.2, opt_epochs=OPT_EPOCHS, tau=0.95, shuffle=True,
                entropy_coeff=0.005, env=env, replay_buffer=buf, collector=col, logger=NullLogger(), discount=0.99,
                num_epochs=488, batch_size=BATCH_ROWS * n_local, gae=True, device=device, save_dir=None,
                use_cuda_graph=not args.no_graph, dist=ctx if ctx.active else None)
    return agent, col, buf, env


def gae_roofline(device, iters=10):
    """GAE scan on an L2-exceeding working set (T=128, N=2^20: 2.4 GB), L2 flushed between launches."""
    import torch
    from torchrl_b200 import ops
    T, N = 128, 1 << 20
    R = torch.randn(T, N, device=device)
    V = torch.randn(T, N, device=device)
    Tm = (torch.rand(T, N, device=device) < 0.01).to(torch.uint8)
    TL = (torch.rand(T, N, device=device) < 0.005).to(torch.uint8)
    LV = torch.randn(N, device=device)
    A, Rt = torch.empty_like(R), torch.empty_like(R)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    for _ in range(3):
        ops.gae_scan(R, V, Tm, TL, LV, 0.99, 0.95, True, A, Rt)
    times = []
    for _ in range(iters):
        flush.fill_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.gae_scan(R, V, Tm, TL, LV, 0.99, 0.95, True, A, Rt)
        e.record()
        torch.cuda.synchronize(device)
        times.append(s.elapsed_time(e) * 1e-3)
    avg = sum(times) / len(times)
    alg_bytes = 18 * T * N + 4 * N
    del R, V, Tm, TL, LV, A, Rt, flush
    torch.cuda.empty_cache()
    return alg_bytes, avg


def gae_in_step_time(agent, buf, iters=20):
    """Duration of the GAE launch at the config's own size (T=128, N=4096: 9.4 MB, L2-resident)."""
    import torch
    with torch.no_grad():
        lv = torch.zeros(buf.env_nums, device=agent.device)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    buf.generalized_advantage_estimation(lv, 0.99, 0.95)
    torch.cuda.synchronize()
    s.record()
    for _ in range(iters):
        buf.generalized_advantage_estimation(lv, 0.99, 0.95)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e-3 / iters


# ----------------------------------------------------------------------------------------- secondary numbers
def _time_epochs(col, agent, epochs, warm=2):
    """(ms collect, ms update) per epoch, CUDA events around whole phases."""
    import torch
    for e in range(warm):
        agent.current_epoch = e
        col.train_one_epoch()
        agent.update_per_epoch()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tc = tu = 0.0
    for _ in range(epochs):
        ev[0].record()
        col.rollout_no_sync()
        ev[1].record()
        agent.update_per_epoch(flush_infos=False)
        ev[2].record()
        torch.cuda.synchronize()
        tc += ev[0].elapsed_time(ev[1])
        tu += ev[1].elapsed_time(ev[2])
    return tc / epochs, tu / epochs


def secondary_measurements(args, device):
    """Driver-visible numbers for the BASELINE configs that are not the headline (each a few seconds):
    configs[0] the reference's own CPU-runnable case (8 envs, 4 worker processes), configs[2] TwinSAC-Q on 1024
    Ant-shaped envs with a 1M-transition ring, configs[3] QR-DQN + prioritised replay on 512 Atari-shaped envs, and
    the headline PPO config on the env variant with desynchronised episodes (bootstrap branch active on every step)."""
    import numpy as np
    import torch
    import torch.nn as nn
    import torchrl_b200.networks as networks
    import torchrl_b200.policies as policies
    from torchrl_b200.algo import PPO, QRDQN, TwinSACQ
    from torchrl_b200.collector import PixelVecCollector, VecCollector, VecOnPolicyCollector
    from torchrl_b200.env import get_vec_env
    from torchrl_b200.replay_buffers import BaseReplayBuffer, OnPolicyReplayBuffer, PrioritizedReplayBuffer
    from torchrl_b200.utils import NullLogger
    out = {}
    # ---- configs[0]: the reference's CPU plumbing at its own size
    try:
        pipe = CpuPipeline(8, 4, min(8, os.cpu_count() or 1))
        try:
            pipe.epoch()
            ts = [pipe.epoch()[0] for _ in range(3)]
        finally:
            pipe.close()
        out["configs[0]"] = {"workload": "PPO SynthHalfCheetah-v0, 8 envs over 4 worker processes, horizon 128, MLP[256, 256], "
                                         "CPU collector + CPU torch update (%s)" % pipe.kind,
                             "env_steps_per_s": 8 * HORIZON * len(ts) / sum(ts), "epoch_s": ts, "kind": pipe.kind}
    except Exception as e:                                          # noqa: BLE001
        out["configs[0]"] = {"error": repr(e)[:200]}
    # ---- headline config on the desynchronised-episode env
    N = args.envs_per_gpu
    env = get_vec_env("SynthHalfCheetahTerm-v0", {"reward_scale": 1, "obs_norm": True}, N, device=device)
    ev_env = get_vec_env("SynthHalfCheetahTerm-v0", {"reward_scale": 1, "obs_norm": True}, N, device=device)
    env.seed(0); torch.manual_seed(0); np.random.seed(0)
    buf = OnPolicyReplayBuffer(env_nums=N, max_replay_buffer_size=HORIZON * N, time_limit_filter=True)
    net = dict(hidden_shapes=list(HIDDEN), append_hidden_shapes=[], base_type=networks.MLPBase, activation_func=nn.Tanh)
    pf = policies.GuassianContPolicyBasicBias(input_shape=OBS_DIM, output_shape=ACT_DIM, tanh_action=True, **net)
    vf = networks.Net(input_shape=(OBS_DIM,), output_shape=1, **net)
    col = VecOnPolicyCollector(vf, env=env, eval_env=ev_env, pf=pf, replay_buffer=buf, device=device,
                               epoch_frames=HORIZON * N, max_episode_frames=999)
    agent = PPO(pf=pf, vf=vf, plr=3e-4, vlr=3e-4, clip_para=0.2, opt_epochs=OPT_EPOCHS, tau=0.95, shuffle=True,
                entropy_coeff=0.005, env=env, replay_buffer=buf, collector=col, logger=NullLogger(), discount=0.99,
                num_epochs=488, batch_size=BATCH_ROWS * N, gae=True, device=device, save_dir=None)
    tc, tu = _time_epochs(col, agent, 3, warm=3)
    out["ppo_desynchronised_episodes"] = {
        "workload": "configs[1] on SynthHalfCheetahTerm-v0 (state-dependent termination, ~5 % of the envs reset per step: "
                    "V(next_obs) bootstrap forward on every collector step)",
        "env_steps_per_s": HORIZON * N / (tc + tu) * 1e3, "ms_rollout": tc, "ms_update": tu}
    del agent, col, buf, env, ev_env
    torch.cuda.empty_cache()
    # ---- configs[2]
    N = 1024
    env = get_vec_env("SynthAnt-v0", {"reward_scale": 1, "obs_norm": False}, N, device=device)
    ev_env = get_vec_env("SynthAnt-v0", {"obs_norm": False}, N, device=device)
    env.seed(0); torch.manual_seed(0); np.random.seed(0)
    buf = BaseReplayBuffer(env_nums=N, max_replay_buffer_size=int(1e6))
    net = dict(hidden_shapes=[256, 256], append_hidden_shapes=[], base_type=networks.MLPBase, activation_func=nn.ReLU)
    pf = policies.GuassianContPolicy(input_shape=111, output_shape=16, tanh_action=True, **net)
    qf1 = networks.QNet(input_shape=119, output_shape=1, **net)
    qf2 = networks.QNet(input_shape=119, output_shape=1, **net)
    col = VecCollector(env=env, eval_env=ev_env, pf=pf, replay_buffer=buf, device=device, epoch_frames=64 * N,
                       max_episode_frames=999)
    agent = TwinSACQ(pf=pf, qf1=qf1, qf2=qf2, plr=3e-4, qlr=3e-4, policy_std_reg_weight=0, policy_mean_reg_weight=0,
                     env=env, replay_buffer=buf, collector=col, logger=NullLogger(), discount=0.99, batch_size=4 * N,
                     device=device, save_dir=None, tau=0.005, opt_times=64, num_epochs=10)
    tc, tu = _time_epochs(col, agent, 3)
    out["configs[2]"] = {"workload": "TwinSAC-Q, 1024 SynthAnt envs (obs 111, act 8), 1M-transition ring, batch 4096, MLP[256, 256]",
                         "collect_env_steps_per_s": 64 * N / tc * 1e3, "updates_per_s": 64 / tu * 1e3,
                         "env_steps_per_s_at_1_update_per_step": 64 * N / (tc + tu) * 1e3}
    del agent, col, buf, env, ev_env
    torch.cuda.empty_cache()
    # ---- configs[3]
    N, Q = 512, 200
    env = get_vec_env("SynthAtari-v0", {}, N, device=device)
    ev_env = get_vec_env("SynthAtari-v0", {}, N, device=device)
    env.seed(0); torch.manual_seed(0); np.random.seed(0)
    buf = PrioritizedReplayBuffer(env_nums=N, max_replay_buffer_size=100 * N)
    qf = networks.Net(input_shape=(4, 84, 84), output_shape=6 * Q,
                      hidden_shapes=[[16, [8, 8], [4, 4], [0, 0]], [32, [4, 4], [2, 2], [0, 0]], [64, [3, 3], [1, 1], [0, 0]]],
                      append_hidden_shapes=[512], base_type=networks.CNNBase, activation_func=nn.ReLU)
    pf = policies.EpsilonGreedyQRDQNDiscretePolicy(quantile_num=Q, qf=qf, start_epsilon=0.1, end_epsilon=0.1,
                                                   decay_frames=1000000, action_shape=6)
    col = PixelVecCollector(env=env, eval_env=ev_env, pf=pf, replay_buffer=buf, device=device, epoch_frames=32 * N,
                            max_episode_frames=50000)
    agent = QRDQN(quantile_num=Q, qf=qf, pf=pf, qlr=5e-5, optimizer_info={"eps": 0.0003125}, env=env, replay_buffer=buf,
                  collector=col, logger=NullLogger(), discount=0.99, batch_size=2 * N, device=device, save_dir=None,
                  opt_times=16, use_soft_update=False, target_hard_update_period=10000, num_epochs=10)
    tc, tu = _time_epochs(col, agent, 3)
    out["configs[3]"] = {"workload": "QR-DQN (200 quantiles) + prioritised replay, 512 SynthAtari envs (4x84x84 uint8), batch 1024",
                         "collect_env_steps_per_s": 32 * N / tc * 1e3, "updates_per_s": 16 / tu * 1e3}
    del agent, col, buf, env, ev_env
    torch.cuda.empty_cache()
    return out


SETTLE_EPOCHS = 30        # untimed epochs between the W warm-up steps and the first timed leg (see run_ours)
DUMP_ENVS = 1024          # envs sampled (fixed seed) for --dump-outputs: ~25 MB whatever --envs-per-gpu is


def dump_outputs(path, agent, buf, env):
    """--dump-outputs: what the last timed epoch computed, as a caller of the collector + PPO update receives it.
    The rollout (T, N, .) arrays, its advantages and returns on a fixed seeded sample of DUMP_ENVS envs (their
    indices in env_sample.npy); the observation normaliser's state; the flat pf|vf parameters after the update; every
    logged scalar of every minibatch update.  Runs before anything else touches the buffer."""
    import re
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    n = buf.env_nums
    cols = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_ENVS), replace=False))
    idx = torch.as_tensor(cols, device=agent.device)
    out = {"env_sample": cols, "params": agent.opt.data}
    for k in ("obs", "next_obs", "acts", "rewards", "values", "terminals", "time_limits", "advs", "estimate_returns"):
        out[k] = getattr(buf, "_" + k).index_select(1, idx)
    nrm = env._obs_normalizer
    out.update(obs_norm_mean=nrm._mean, obs_norm_var=nrm._var, obs_norm_count=nrm._count)
    infos = agent._flush_infos(agent._mb_state["U"])
    for key in infos[0]:
        out["info_" + re.sub(r"[^A-Za-z0-9_.-]", "_", key)] = np.array([i[key] for i in infos], dtype=np.float64)
    for name, v in out.items():
        a = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def run_ours(args):
    import torch
    from torchrl_b200 import _lib
    from torchrl_b200.distributed import DataParallelContext
    ctx = DataParallelContext()
    if ctx.world_size != args.gpus and ctx.world_size > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, ctx.world_size))
    device = ctx.device
    if device.type != "cuda":
        raise SystemExit("bench.py needs a CUDA device (no CPU path in the product)")
    _lib.load()                                           # fail loudly if the native library is missing
    from torchrl_b200.networks import fused
    fused.set_matmul_mode(args.matmul)
    agent, col, buf, env = build_agent(args, ctx, device)
    frames_per_step = HORIZON * args.envs_per_gpu * ctx.world_size

    def epoch(host_io):
        agent.current_epoch = 0
        if host_io:
            col.train_one_epoch()
            agent.update_per_epoch()
        else:
            col.rollout_no_sync()
            # bound the launch queue (no data copied): the public-API leg waits here too (it reads the episode
            # count), and a queue holding the rollout's 128 AND the update's 320 graph launches measured ~8 % slower
            # on B200 than two shorter ones; with several ranks this also aligns them before the collective-bearing
            # update graphs
            torch.cuda.current_stream(device).synchronize()
            agent.update_per_epoch(flush_infos=False)

    # one nvidia-smi poller for the whole job (rank 0's GPU), started now so that its start-up is over before
    # the timed region (see ClockSampler)
    sampler = ClockSampler(ctx.local_rank if (ctx.rank == 0 and os.environ.get("BENCH_NO_CLOCKS") != "1") else None)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        epoch(True)
    # settle: with several ranks the first ~2 s of the job are not steady (whichever leg ran first -- right behind 3
    # warm-up epochs -- came out 10-80 % slow in 1 run of 3, per-step times flat inside the run; the second leg never
    # did).  A fixed number of extra untimed epochs (the same on every rank: they contain collectives) covers it.
    for _ in range(SETTLE_EPOCHS):
        epoch(True)
    torch.cuda.synchronize(device)

    # ---- e2e: public API, wall clock, host copies inside ---------------------------------------
    ctx.barrier()
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    e2e_step_ms = []
    for _ in range(args.steps):
        t1 = time.perf_counter()
        epoch(True)
        e2e_step_ms.append(round((time.perf_counter() - t1) * 1e3, 3))
    torch.cuda.synchronize(device)
    ctx.barrier()
    t_e2e = ctx.max_over_ranks(time.perf_counter() - t0)

    # ---- value: device-timed, host out of the loop ------------------------------------------
    # (second, after its own warm-up epochs: measured first, right behind the job's start-up, this leg was bistable
    # with several ranks -- 1 run in 3 came out 20-50 % slower than the public-API leg that followed it)
    for _ in range(max(args.warmup, 3)):
        epoch(False)
    torch.cuda.synchronize(device)
    launches0 = _lib.launch_count()
    ctx.barrier()
    torch.cuda.synchronize(device)
    sampler.mark_begin()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    marks[0].record()
    for k in range(args.steps):
        epoch(False)
        marks[k + 1].record()
        if os.environ.get("BENCH_VALUE_SYNC", "1") == "1":
            # bound the launch queue: wait (no data copied) until the epoch has drained before queueing
            # the next ~450 graph launches; an unbounded queue measured ~15% slower on B200
            torch.cuda.current_stream(device).synchronize()
    torch.cuda.synchronize(device)
    sampler.mark_end()
    ctx.barrier()
    clocks = sampler.stop()
    t_dev = ctx.max_over_ranks(marks[0].elapsed_time(marks[-1]) * 1e-3)
    step_ms = [round(marks[k].elapsed_time(marks[k + 1]), 3) for k in range(args.steps)]    # this rank's steps
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, agent, buf, env)

    value = frames_per_step * args.steps / t_dev
    e2e_value = frames_per_step * args.steps / t_e2e
    st = agent._mb_state
    h2d = st["perm_host"].numel() * 8 + agent.opt.lr_host.numel() * 4 * 2
    d2h = st["log32"].numel() * 4 + st["log64"].numel() * 8 + 4 + 4 + 8 * args.envs_per_gpu

    roofline = None
    if ctx.rank == 0 and not args.skip_roofline:
        peak, how = measured_peaks()
        alg_bytes, dur = gae_roofline(device)
        t_small = gae_in_step_time(agent, buf)
        traffic = None
        pj = os.path.join(ROOT, "profiles", "gae_scan_ncu_summary.json")
        if os.path.exists(pj):
            traffic = json.load(open(pj)).get("dram_bytes_per_launch")
        roofline = {"kernel": "gae_tma_kernel<GAE> (csrc/gae_tma.cu: persistent, TMA-staged tiles; what trl_gae_scan "
                              "launches at this size)", "bound": "hbm",
                    "workload": "T=128 x N=2^20 rollout (2.42 GB algorithmic), L2 flushed between launches",
                    "achieved": alg_bytes / dur / 1e9, "peak": peak, "peak_source": how, "unit": "GB/s",
                    "frac": alg_bytes / dur / 1e9 / peak, "traffic": traffic,
                    "algorithmic_bytes_per_launch": alg_bytes, "launch_us": dur * 1e6,
                    "in_step": {"workload": "T=128 x N=%d (9.4 MB, L2-resident): latency-bound" % args.envs_per_gpu,
                                "launch_us": t_small * 1e6,
                                "achieved_GBs": (18 * HORIZON * args.envs_per_gpu) / t_small / 1e9}}

    cpu_baseline = None
    if ctx.rank == 0 and args.gpus == 1 and not args.skip_cpu_baseline:
        procs, cores = auto_procs(args.envs_per_gpu, args.cpu_procs)
        threads = best_torch_threads(cores, BATCH_ROWS * args.envs_per_gpu)
        pipe = CpuPipeline(args.envs_per_gpu, procs, threads)
        try:
            dt, tc, tu = pipe.epoch()                       # ONE whole epoch, timed for real (~20-30 s of CPU work)
        finally:
            pipe.close()
        cpu_baseline = {"value": pipe.frames / dt, "unit": "env-steps/s", "cores": max(procs, threads),
                        "host_logical_cores": cores, "kind": pipe.kind,
                        "sample": pipe.describe() + "; 1 epoch, no warm-up epoch (the reference arm, --impl reference, "
                                                    "times warm epochs)",
                        "detail": {"epoch_s": dt, "collect_s": tc, "update_s": tu}}

    secondary = None
    if ctx.rank == 0 and args.gpus == 1 and not args.skip_secondary:
        try:
            secondary = secondary_measurements(args, device)
        except Exception as e:                                      # noqa: BLE001 -- never lose the headline line
            secondary = {"error": repr(e)[:300]}

    if ctx.rank == 0:
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": ctx.world_size,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": t_dev / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.envs_per_gpu, ctx.world_size),
                       "global_envs": args.envs_per_gpu * ctx.world_size,
                       "untimed_epochs": "%d warm-up + %d settling epochs before the first timed leg (e2e), %d more before "
                                         "the device-timed leg" % (max(args.warmup, 3), SETTLE_EPOCHS, max(args.warmup, 3)),
                       "parallelism": "dp%d (env sharding; flat gradient summed by a one-shot all-reduce over NVLink peer memory fused "
                                      "with the gradient norms, csrc/comm.cu)" % ctx.world_size,
                       "matmul": {"fp32": "fp32 cuBLAS SIMT (TF32 off)",
                                  "tf32x3": "3xTF32 error-compensated tensor-core GEMMs (fp32-faithful), cuBLAS",
                                  "tc3": "256-wide layers: hand-written tcgen05 3xTF32 GEMM on CTA pairs (fp32-faithful, "
                                         "csrc/gemm_pair.cu); 17-wide / <=8-wide layers: HBM-bound fp32 kernels (csrc/skinny.cu)"}[args.matmul], "cuda_graphs": not args.no_graph,
                       "l2": "each step rewrites the whole 100 MB rollout working set and all activations "
                             "(> 126 MB L2 per epoch); the GAE roofline launch flushes L2 explicitly"},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": t_e2e / args.steps * 1e3},
            "gpu_launches": launches,
            "step_ms": step_ms,
            "e2e_step_ms": e2e_step_ms,
            "clocks": clocks,
        }
        if roofline is not None:
            line["roofline"] = roofline
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if secondary is not None:
            line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    # teardown: drop the captured graphs (they hold NCCL work) before leaving; with several ranks exit
    # hard after a final barrier -- destroy_process_group() was observed to hang for minutes when
    # CUDA graphs that captured NCCL kernels are still alive
    agent._mb_graph = None
    col._graphs.clear()
    torch.cuda.synchronize(device)
    if ctx.active:
        ctx.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
