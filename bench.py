"""Learner grad-steps/s of the recurrent QMIX update path (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this engine (one process per GPU; torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy (same
                                                             # arguments -> same inputs: compare two builds output for output)

One "step" = sample(B) -> train_policy_on_batch -> soft_target_updates (base_runner.py:259-284) on synthetic
SMAC-shaped replay data.  Prints ONE JSON line (rank 0).
  value    : steps/s with everything resident in HBM -- the whole step (device MT19937 draw, gather, fused learner,
             Adam, Polyak) replayed from one CUDA graph; CUDA-event timed, max over ranks.
  e2e      : same metric through the drop-in Python API with HOST inputs: every step inserts one freshly collected
             episode from pinned host memory (H2D), draws indices on the host with np.random.choice (H2D), trains,
             soft-updates and reads loss/grad_norm/Q_tot back (D2H) -- the runner's per-step sequence.
  roofline : dominant kernel of the step (per-kernel CUDA-event timing on the launch stream).
  cpu_baseline : the oracle port of the reference learner timed on the host cores (bounded sample).
"""
import argparse
import ctypes as C
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "off-policy_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (n_agents, obs, act, state, T, B, per)    -- BASELINE.json configs
    "qmix_3m": (3, 30, 9, 48, 60, 32, False),          # configs[1]: the configuration the metric is quoted on
    "qmix_8m_per": (8, 80, 14, 168, 120, 64, True),    # configs[3]
    "qmix_2s3z": (5, 80, 11, 120, 120, 32, False),     # configs[4]
    # configs[0]: scripts/train_mpe_qmix.sh = recurrent QMIX on MPE simple_spread (obs 18, Discrete(5), state 54, episode_length 25,
    # --use_reward_normalization, no available-action masks) -- the reference's own CPU-runnable case
    "qmix_mpe_spread": (3, 18, 5, 54, 25, 32, False),
}
PROFILE_REPS, PROFILE_INNER, E2E_MIN_STEPS, CPU_STEPS, E2E_WARM = 6, 8, 20, 20, 5     # loop lengths (tests/test_bench_dryrun.py shrinks them)
NO_AVAIL = {"qmix_mpe_spread"}       # MPE passes avail_acts = None (runner/rnn/mpe_runner.py:62) and normalises rewards


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/ncu_traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(path)).get(kernel, {}).get("dram_bytes")
    except Exception:
        return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tflops=1590.0, tflops_sustained=1400.0, src="fallback")


DUMP_BYTES = 64 << 20


def dump_outputs(outdir, arrays):
    """--dump-outputs: what the timed path computed in its last step, one <outdir>/<name>.npy per array (float64 where the engine keeps
    float64 or integers, float32 otherwise), so that two builds run with the same arguments can be compared output for output.  An array
    larger than its share of DUMP_BYTES is cut to a fixed, seeded sample of its elements (the same positions in every run)."""
    os.makedirs(outdir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, a in arrays.items():
        a = np.asarray(a.detach().cpu() if torch.is_tensor(a) else a)
        a = a.astype(np.float64 if a.dtype in (np.float64, np.int64) else np.float32)
        if a.nbytes > share:
            pos = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[pos]
        np.save(os.path.join(outdir, name + ".npy"), a)


def qmix_outputs(tr, rep, B):
    """What the caller of one QMIX / M_QMix step holds afterwards: its train_info, the replay indices it sampled, the new PER priorities
    and importance weights, and the live and target parameters (the policy's networks are views of them)."""
    out = dict(loss=tr._info[0], grad_norm=tr._info[1], Q_tot=tr._info[2], sample_indices=rep.sampled_indices(B), params=tr.theta,
               target_params=tr.theta_tgt)
    if tr.use_per:
        out.update(priorities=tr._prio_view[:B], importance_weights=rep.sampled_weights(B))
    return out


def maddpg_outputs(tr, rep, B):
    """The same for one R-MADDPG / R-MATD3 update; the actor's loss and gradient norm only when that update trained the actor."""
    pol, info = tr.policies["policy_0"], tr._info
    out = dict(critic_loss=info[0], critic_grad_norm=info[1], sample_indices=rep.sampled_indices(B),
               actor_params=pol.actor_vecs[0], target_actor_params=pol.actor_vecs[1], critic_params=pol.critic_vecs[0],
               target_critic_params=pol.critic_vecs[1])
    if (tr.num_updates["policy_0"] - 1) % tr.actor_update_interval == 0:
        out.update(actor_loss=info[4], actor_grad_norm=info[5])
    return out


MADDPG_WORKLOADS = {
    # name: (n_agents, obs, act (Box), state, T, B, td3)    -- BASELINE.json configs[2]: MPE simple_spread shapes, continuous actions
    "rmaddpg_spread": (3, 18, 2, 54, 25, 32, False, False),
    "rmatd3_spread": (3, 18, 2, 54, 25, 32, True, False),
    # the env's real action space, Discrete(5) (envs/mpe/environment.py:62-63): one-hot actions, Gumbel-softmax actors
    "rmaddpg_spread_disc": (3, 18, 5, 54, 25, 32, False, True),
    "rmatd3_spread_disc": (3, 18, 5, 54, 25, 32, True, True),
}


def run_maddpg(args):
    """R-MADDPG / R-MATD3 learner (BASELINE config 3): sample -> shared_train_policy_on_batch -> soft update.  `value`: the
    whole update replayed from captured CUDA graphs; `e2e`: the eager drop-in calls (one C call enqueues the ~40 kernels of an
    update) with a D2H loss read per step; CPU arm = the pinned oracle port."""
    from offpolicy._b200 import capi
    from offpolicy._b200 import factory as mc
    from offpolicy._b200 import factory as rc
    n, o, a, sdim, T, B, td3, disc = MADDPG_WORKLOADS[args.workload]
    cfg = mc.MaddpgLearnerConfig(n_agents=n, obs_dim=o, act_dim=a, state_dim=sdim, td3=td3, actor_update_interval=2 if td3 else 1, gain=1.0, discrete=disc)

    def sample_gumbel(shape, eps=1e-20):        # util.py:127-130: one uniform_ draw from torch's CPU generator
        u = torch.empty(*shape).uniform_()
        return -torch.log(-torch.log(u + eps) + eps)

    def cpu_learner():        # the CPU arm only: the oracle port of the reference learner, same configuration values
        import dataclasses
        from oracle.maddpg import MaddpgConfig, MaddpgLearner
        return MaddpgLearner(MaddpgConfig(**dataclasses.asdict(cfg)), seed=1)
    E = min(args.buffer, 5000)
    rs = np.random.default_rng(0)

    def episodes(k):
        return [rs.standard_normal((T + 1, k, n, o), dtype=np.float32), np.repeat(rs.standard_normal((T + 1, k, 1, sdim), dtype=np.float32), n, 2),
                (np.eye(a, dtype=np.float32)[rs.integers(0, a, (T, k, n))] if disc else rs.uniform(-1, 1, (T, k, n, a)).astype(np.float32)), np.repeat(rs.standard_normal((T, k, 1, 1), dtype=np.float32), n, 2),
                np.zeros((T, k, n, 1), np.float32), np.zeros((T, k, 1), np.float32)]

    def cpu_noise(s):
        """the draws the reference makes per update (util.py:127-130, 217-218)"""
        upd = s % cfg.actor_update_interval == 0
        if disc:
            return (sample_gumbel((T + 1, n * B, a)).numpy() if td3 else None), (sample_gumbel((T, n * B, a)).numpy() if upd else None)
        return (torch.empty(T + 1, n * B, a).normal_(0, cfg.target_noise).numpy() if td3 else None), None

    if args.impl == "reference":
        from oracle.replay import UniformReplay
        th = best_threads = 8
        torch.set_num_threads(th)
        buf = UniformReplay(min(E, 1024), T, n, o, sdim, a, use_avail=False)
        for c in range(0, min(E, 1024), 64):
            buf.insert(64, *episodes(64), None)
        L = cpu_learner()
        np.random.seed(1)
        times = []
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            out, inds = buf.sample(B)
            noise, anoise = cpu_noise(s)
            info, _ = L.step(out, noise, anoise)
            if info["update_actor"]:
                L.soft_update()
            float(info["critic_loss"])
            if s >= args.warmup:
                times.append(time.perf_counter() - t0)
        sps = 1.0 / float(np.median(times))
        emit((dict(metric="learner grad-steps/sec", value=sps, unit="steps/s", impl="reference", n_gpus=args.gpus, steps=args.steps,
                              warmup=args.warmup, ms_per_step=1e3 / sps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                              data="synthetic", config=dict(workload=args.workload, batch=B, episode_len=T, n_agents=n),
                              cpu_baseline=dict(value=sps, unit="steps/s", cores=th, kind="port", sample="%d timed updates" % args.steps),
                              e2e=dict(value=sps, unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)))
        return
    torch.cuda.set_device(0)
    torch.set_num_threads(1)        # tiny host ops (noise draws): the reference's default n_training_threads = 1 (config.py:17-18)
    lib = capi.lib()
    from offpolicy.utils.rec_buffer import RecReplayBuffer
    info = {"policy_0": dict(obs_space=[o], share_obs_space=[sdim], act_space=mc.Discrete(a) if disc else mc.Box(a))}
    buf = RecReplayBuffer(info, {"policy_0": list(range(n))}, E, T, True, False, rng="device", max_batch=128)
    for c in range(0, E, 128):
        k = min(128, E - c)
        buf.insert(k, *[rc.pd(x) for x in episodes(k)], None)
    torch.manual_seed(1)
    with contextlib.redirect_stdout(sys.stderr):        # (the drop-in classes mirror the reference's prints)
        margs, pol, tr = mc.build_maddpg(cfg, B, T)
    buf.seed_device_rng(1)

    def step():
        smp = buf.sample(B)
        info_t, _, _ = tr.shared_train_policy_on_batch("policy_0", smp)
        if info_t["update_actor"]:
            pol.soft_target_updates()
        return info_t

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    from offpolicy._b200.graph import MaddpgStepGraph
    graph = MaddpgStepGraph(buf, tr, B)
    for _ in range(max(args.warmup, 3)):
        graph.launch()
    graph.synchronize()
    l0 = lib.mx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        e0.record(graph.stream)
        for _ in range(args.steps):
            graph.launch()
        e1.record(graph.stream)
        graph.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = int(lib.mx_launch_count() - l0)
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, maddpg_outputs(tr, buf.policy_buffers["policy_0"], B))
    if args.quick:          # tuning sweeps: the device-resident number only (not a bench line)
        emit(dict(quick=True, workload=args.workload, value=1000.0 / ms, ms_per_step=ms, opts=args.opt, kernels_per_step=launches / args.steps))
        return
    for _ in range(10):
        float(step()["critic_loss"])
    torch.cuda.synchronize()
    n_e2e = max(50, min(args.steps, 200))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        float(step()["critic_loss"])
    torch.cuda.synchronize()
    e2e = n_e2e / (time.perf_counter() - t0)
    torch.set_num_threads(8)
    L = cpu_learner()
    from oracle.maddpg import synth_batch_cont, synth_batch_disc
    tms = []
    for s in range(8):
        batch = (synth_batch_disc if disc else synth_batch_cont)(cfg, B, T, seed=s) + (None, None)
        t0 = time.perf_counter()
        noise, anoise = cpu_noise(s)
        i2, _ = L.step(batch, noise, anoise)
        if i2["update_actor"]:
            L.soft_update()
        if s >= 2:
            tms.append(time.perf_counter() - t0)
    cpu = 1.0 / float(np.median(tms))
    emit(dict(metric="learner grad-steps/sec", value=1000.0 / ms, unit="steps/s", n_gpus=1, steps=args.steps, warmup=max(args.warmup, 3),
                          ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                          config=dict(workload=args.workload, batch=B, episode_len=T, n_agents=n, obs_dim=o, act_dim=a, state_dim=sdim,
                                      buffer_episodes=E, step="CUDA graphs (one per update_actor variant): device MT19937 sample + mx_maddpg_step (+ soft update when the actor was updated); "
                                           "noise drawn on the host from torch's CPU RNG like the reference and copied H2D per update"),
                          e2e=dict(value=e2e, unit="steps/s", h2d_bytes_per_step=((T + 1) * n * B * a * 4 if td3 else 0) + ((T + 1) * n * B * a * 4 // cfg.actor_update_interval if disc else 0),
                                   d2h_bytes_per_step=4,
                                   path="RecReplayBuffer.sample + R_MADDPG.shared_train_policy_on_batch + soft_target_updates + D2H critic_loss"),
                          gpu_launches=launches, kernels_per_step=launches / args.steps,
                          roofline=dict(bound="tensor", kernel="(many small launches)", achieved=None, peak=peaks()["tflops_sustained"], unit="TFLOP/s",
                                        frac=None, traffic=None, note="launch/latency bound at B=32, T=25; see DESIGN.md"),
                          cpu_baseline=dict(value=cpu, unit="steps/s", cores=8, kind="port", sample="6 timed updates of the same workload (oracle port)"),
                          clocks=clocks.summary()))


def make_cfg(w):
    from offpolicy._b200.factory import LearnerConfig
    n, o, a, s, T, B, per = WORKLOADS[w]
    return LearnerConfig(n_agents=n, obs_dim=o, act_dim=a, state_dim=s, use_per=per, gain=1.0), T, B


def workload_config(args, cfg, T, B, world):
    """The `config` object of the JSON line: a function of the command line only, so both arms (--impl engine / reference) print the
    same thing for the same workload.  Arm-specific detail goes to the `notes` key."""
    E = args.buffer            # weak scaling: every GPU keeps a full-size replay shard (larger than L2) and its own batch
    return dict(workload=args.workload, batch_per_gpu=B, episode_len=T, n_agents=cfg.n_agents, obs_dim=cfg.obs_dim, act_dim=cfg.act_dim,
                state_dim=cfg.state_dim, buffer_episodes_per_gpu=E, parallelism="dp%d" % world if world > 1 else "single",
                l2="inputs gathered from a replay larger than L2; the per-step working set is L2-resident by design")


def oracle_cfg(cfg):
    """The CPU arm's view of the same workload: the oracle's config dataclass (same field names)."""
    import dataclasses
    from oracle.qmix import QmixConfig
    return QmixConfig(**dataclasses.asdict(cfg))


def synth_episodes(cfg, T, n, rs, avail=True):
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    f = [rs.standard_normal((T + 1, n, N, O), dtype=np.float32), np.repeat(rs.standard_normal((T + 1, n, 1, S), dtype=np.float32), N, 2),
         np.eye(A, dtype=np.float32)[rs.integers(0, A, (T, n, N))], np.repeat(rs.standard_normal((T, n, 1, 1), dtype=np.float32), N, 2),
         np.zeros((T, n, N, 1), np.float32), np.zeros((T, n, 1), np.float32), np.ones((T + 1, n, N, A), np.float32) if avail else None]
    return f


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.samples, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) >= 6 and s[2 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(self.samples))


# ---------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference learner on the host cores
# ---------------------------------------------------------------------------------------------------------
def best_cpu_threads(cfg, T, B, E, avail=True):
    """The reference sets torch.set_num_threads(n_training_threads); on a many-core host more threads are SLOWER for
    these tiny ops, so the baseline uses the fastest of a few thread counts (probed with 3 timed steps each)."""
    cores = os.cpu_count() or 1
    best, best_sps = 1, 0.0
    for th in sorted({1, 4, 8, 16, min(32, cores)}):
        if th > cores:
            continue
        sps, _ = cpu_learner_steps_per_s(cfg, T, B, E, 3, 1, th, avail)
        if sps > best_sps:
            best, best_sps = th, sps
    return best


def cpu_learner_steps_per_s(cfg, T, B, E, steps, warmup, threads, avail=True):
    from oracle.qmix import QmixLearner
    from oracle.replay import UniformReplay, PrioritizedReplay
    cfg = oracle_cfg(cfg)
    torch.set_num_threads(threads)
    rs = np.random.default_rng(0)
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    buf = (PrioritizedReplay(0.6, E, T, N, O, S, A) if cfg.use_per else UniformReplay(E, T, N, O, S, A, use_avail=avail, reward_norm=not avail))
    for c in range(0, E, 64):
        n = min(64, E - c)
        buf.insert(n, *synth_episodes(cfg, T, n, rs, avail))
    torch.manual_seed(1)
    np.random.seed(1)
    L = QmixLearner(cfg, seed=1)
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        if cfg.use_per:
            out, inds = buf.sample(B, 0.4)
        else:
            out, inds = buf.sample(B)
        info, prio, _ = L.step(out)
        if cfg.use_per:
            buf.update_priorities(inds, prio)
        L.soft_update()
        float(info["loss"])
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    return 1.0 / float(np.median(times)), float(np.median(times)) * 1e3


def torch_eager_gpu_steps_per_s(cfg, T, B, E, steps, warmup, avail=True):
    """Secondary baseline (SURVEY.md section 8(d)): the reference learner's own eager PyTorch ops on the SAME B200 (what
    `--cuda` gives the reference): the oracle port with its networks on cuda:0, batches sampled by the NumPy replay on the host and
    copied up per step like the reference's to_torch(...).to(device).  ~10^4 small ATen launches per step."""
    from oracle.qmix import QmixLearner
    from oracle.replay import UniformReplay, PrioritizedReplay
    cfg = oracle_cfg(cfg)
    rs = np.random.default_rng(0)
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    buf = (PrioritizedReplay(0.6, E, T, N, O, S, A) if cfg.use_per else UniformReplay(E, T, N, O, S, A, use_avail=avail, reward_norm=not avail))
    for c in range(0, E, 64):
        n = min(64, E - c)
        buf.insert(n, *synth_episodes(cfg, T, n, rs, avail))
    torch.manual_seed(1)
    np.random.seed(1)
    L = QmixLearner(cfg, seed=1, device="cuda")
    times = []
    for s in range(warmup + steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out, inds = buf.sample(B, 0.4) if cfg.use_per else buf.sample(B)
        info, prio, _ = L.step(out)
        if cfg.use_per:
            buf.update_priorities(inds, prio)
        L.soft_update()
        float(info["loss"])
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    return 1.0 / float(np.median(times))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, T, B = make_cfg(args.workload)
    world = max(1, args.gpus)
    E = args.buffer         # one rank's shard: the CPU arm is one learner on the host cores
    avail = args.workload not in NO_AVAIL
    cores = best_cpu_threads(cfg, T, B, min(E, 256), avail)         # (thread-count probe on a small replay: the learner dominates)
    sps, ms = cpu_learner_steps_per_s(cfg, T, B, E, args.steps, args.warmup, cores, avail)
    line = dict(metric="learner grad-steps/sec", value=sps, unit="steps/s", impl="reference", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=workload_config(args, cfg, T, B, world),
                cpu_baseline=dict(value=sps, unit="steps/s", cores=cores, host_cores=os.cpu_count(), kind="port",
                                  sample="%d timed learner steps (sample+train+soft update) of the same workload, replay of %d episodes" % (args.steps, E)),
                e2e=dict(value=sps, unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


# ---------------------------------------------------------------------------------------------------------
# algorithmic work per kernel (DESIGN.md "roofline"), H=64
# ---------------------------------------------------------------------------------------------------------
def kernel_work(cfg, T, B, P):
    N, O, A, S, H, ME, HY = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim, 64, cfg.mixer_hidden, cfg.hyper_hidden
    M, E = B * (T + 1) * N, B * T
    mix = (S * HY + HY * N * ME) + (S * HY + HY * ME) + S * ME + (S * HY + HY) + N * ME + ME
    fl = {
        "k_front_fwd": 2 * 2.0 * M * (O * H + H * H + 3 * H * H),
        "k_gru_fwd": 2 * 2.0 * M * 3 * H * H,
        "k_qhead": 2 * 2.0 * M * H * A,
        "k_mixer": 2.0 * E * mix * 4,                    # target fwd + live fwd + live bwd (dgrad + wgrad)
        "k_mix_hyper_fwd": 2.0 * E * (mix - N * ME - ME) * 2,         # split pipeline: hypernet layers of the live + target mixers
        "k_mix_core": 2.0 * E * (N * ME + ME) * 4,                    # q-dependent part: both forwards + backward
        "k_mid": 2.0 * E * (N * ME + ME) * 4 + 2.0 * E * N * H * A * 3 + 2.0 * E * N * 3 * H,    # 3 head evaluations per row + core + head backward
        "k_mix_hyper_bwd": 2.0 * E * (mix - N * ME - ME) * 2,         # dgrad + wgrad of the live hypernets
        "k_qhead_bwd": 2.0 * M * 3 * H,
        "k_gru_bwd": 2.0 * M * 3 * H * H,
        "k_front_bwd": 2.0 * M * (2 * 3 * H * H * 2 + 3 * H * H + 2 * H * H + H * H + 2 * O * H + O * H) / 1.0,
        "k_gru_wgrad": 2.0 * M * (2 * 3 * H * H),      # dW_ih + dW_hh when they run as their own kernel (option gru_wgrad_split): taken off k_front_bwd below
        # tensor-core variants (options front_tc_wide / wgrad_tc): same algorithmic work as the kernels they replace, split in two for the backward
        "k_front_fwd_tc": 2 * 2.0 * M * (O * H + H * H + 3 * H * H),
        "k_front_fwd_tc_wide": 2 * 2.0 * M * (O * H + H * H + 3 * H * H),
        "k_front_bwd_tc": 2.0 * M * (3 * H * H + H * H + O * H),                      # dx2 = dgi.W_ih, dx1 = da2.W2, dx0 = da1.W1
        "k_wgrad_tc": 2.0 * M * (2 * 3 * H * H + H * H + O * H),                     # dW_ih, dW_hh, dW2, dW1
    }
    fields = 4.0 * B * (N * (T + 1) * O + (T + 1) * S + N * T * A + N * (T + 1) * A + 3 * N * T + T)
    by = {"k_gather": 2 * fields, "k_adam": 4.0 * P * 7, "k_polyak": 4.0 * P * 3, "k_grad_reduce": 4.0 * P * 2,
          "k_optim_fused": 4.0 * P * (7 + 3)}            # Adam + fused Polyak (the per-CTA partials it also sums are an implementation cost)
    return fl, by


def run_engine(args):
    from offpolicy._b200 import capi, factory
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    torch.cuda.set_device(local)
    torch.set_num_threads(1)        # host side of the engine arm: the reference's own default (config.py n_training_threads = 1)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = capi.lib()
    dev = capi.device()
    cfg, T, B = make_cfg(args.workload)
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    E = args.buffer            # one full-size replay shard per rank (weak scaling: per-GPU batch AND per-GPU replay fixed; the shard stays larger than L2 at every N)
    rs = np.random.default_rng(rank)
    avail = args.workload not in NO_AVAIL
    buf = factory.make_rec_buffers(N, O, A, S, T, E, per_alpha=0.6 if cfg.use_per else None, norm=not avail, rng="device", max_batch=max(B, 128), avail=avail)

    def wrap(ep):
        return [factory.pd(x) if x is not None else None for x in ep]
    for c in range(0, E, 128):
        n = min(128, E - c)
        buf.insert(n, *wrap(synth_episodes(cfg, T, n, rs, avail)))
    torch.manual_seed(1)
    np.random.seed(1)
    with contextlib.redirect_stdout(sys.stderr):        # the drop-in QMix mirrors the reference's "double Q learning will be used" print
        args_ns, pol, tr = factory.build_qmix(cfg, B, T, debug=False)      # product configuration: no debug outputs, k_mid
    pb = buf.policy_buffers["policy_0"]
    buf.seed_device_rng(1 + rank)
    stream = torch.cuda.current_stream()
    sp = capi.stream_ptr

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident loop ----------------
    graph = None
    tgraph = None
    run_stream = torch.cuda.current_stream()
    p2p = world > 1 and bool(getattr(tr, "_p2p", False))      # gradient exchange over NVLink peer memory inside the step (no NCCL)
    if world == 1 or p2p:
        from offpolicy._b200.graph import StepGraph
        torch.cuda.synchronize()
        graph = StepGraph(buf, tr, B, beta=0.4)
        kernels_per_step = graph.num_kernels
        run_stream = graph.stream
        step = graph.launch
    else:
        def eager():
            if cfg.use_per:
                smp = buf.sample(B, 0.4, "policy_0")
            else:
                smp = buf.sample(B)
            info, prio, idx = tr.train_policy_on_batch(smp)
            if cfg.use_per:
                buf.update_priorities(idx, prio, "policy_0")
            tr.soft_target_updates()
        for _ in range(3):
            eager()
        torch.cuda.synchronize()
        c0 = lib.mx_launch_count()
        eager()
        kernels_per_step = int(lib.mx_launch_count() - c0)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        try:
            with torch.cuda.stream(side):
                eager()
                tgraph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(tgraph, stream=side):
                    eager()
            torch.cuda.current_stream().wait_stream(side)
            step = tgraph.replay
        except Exception as ex:       # NCCL capture unavailable: stay eager
            sys.stderr.write("graph capture of the data-parallel step failed (%s); running eager\n" % ex)
            tgraph = None
            step = eager

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    if p2p:
        tr.ws_view("xstat").zero_()          # exchange breakdown accumulated by the optimiser kernel over the timed steps
        torch.cuda.synchronize()
    launches0 = lib.mx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record(run_stream)
        for _ in range(args.steps):
            step()
        e1.record(run_stream)
        barrier()
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms_total, op=torch.distributed.ReduceOp.MAX)
    ms_step = float(ms_total) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, qmix_outputs(tr, pb, B))
    exchange = None
    if p2p:
        # per rank: mean us per step spent pushing the gradient to the peers (+ system fence), waiting for the last peer's flag (rank skew +
        # NVLink latency), adding the slots; and the longest single wait
        x = tr.ws_view("xstat").clone()
        n = max(float(x[3]), 1.0)
        mine = torch.tensor([float(x[0]) / n / 1e3, float(x[1]) / n / 1e3, float(x[2]) / n / 1e3, float(x[4]) / 1e3], device=dev)
        allx = [torch.zeros_like(mine) for _ in range(world)]
        torch.distributed.all_gather(allx, mine)
        exchange = dict(per_rank_us=[dict(push=round(float(v[0]), 2), wait=round(float(v[1]), 2), sum=round(float(v[2]), 2), max_wait=round(float(v[3]), 1)) for v in allx],
                        note="stamped by the thread that owns the four scalar columns: push = its stores to the peers, wait = until every peer's lines for those columns have arrived and are summed (flag-in-data lines; option p2p_ll=0: push + fence, wait for the last peer's flag, local sum)")
    launches = int(lib.mx_launch_count() - launches0)
    if tgraph is not None:
        launches = kernels_per_step * args.steps

    if args.quick:          # tuning sweeps: the device-resident number only (not a bench line)
        if rank == 0:
            emit(dict(quick=True, workload=args.workload, value=world * 1000.0 / ms_step, ms_per_step=ms_step, opts=args.opt,
                      kernels_per_step=kernels_per_step, n_gpus=world, exchange=exchange))
            sys.stdout.flush()
        if graph is not None:
            graph.close()
        if world > 1:
            torch.distributed.barrier()
            os._exit(0)
        return

    # ---------------- e2e: host inputs through the drop-in API ----------------
    fresh = [synth_episodes(cfg, T, 1, rs, avail) for _ in range(8)]
    h2d = sum(x.nbytes for x in fresh[0] if x is not None)
    d2h = 4

    def e2e_step(i):
        buf.insert(1, *wrap(fresh[i % 8]))
        if cfg.use_per:
            smp = buf.sample(B, 0.4, "policy_0")
        else:
            smp = buf.sample(B)
        info, prio, idx = tr.train_policy_on_batch(smp)
        if cfg.use_per:
            buf.update_priorities(idx, prio, "policy_0")
        tr.soft_target_updates()
        return float(info["loss"])                                                    # D2H read of the step's result (syncs)

    def e2e_run(n):
        for i in range(E2E_WARM):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(n):
            e2e_step(i)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
        return world * n / float(dt)

    n_e2e = max(E2E_MIN_STEPS, min(args.steps, 200))
    # (1) indices drawn per call from NumPy's process-global stream on the host, as the reference does (one extra H2D of B int64)
    buf.rng = "numpy"
    e2e_host_rng_sps = e2e_run(n_e2e)
    # (2) the same NumPy stream continued ON THE DEVICE (RecReplayBuffer.adopt_numpy_rng(): bit-identical indices as long as nothing else
    #     draws from np.random between two samples, which holds here; no index upload, no host draw) -- the headline e2e number
    buf.adopt_numpy_rng()
    e2e_sps = e2e_run(n_e2e)

    # same loop with the loss read lagging ONE step (copied to pinned memory asynchronously, read after the next step has been
    # enqueued): what a runner that logs train_info asynchronously sees.  Reported beside, not instead of, the synchronous number.
    pins = [torch.zeros(4, dtype=torch.float32).pin_memory() for _ in range(2)]
    evts = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_step_lagged(i):
        buf.insert(1, *wrap(fresh[i % 8]))
        smp = buf.sample(B, 0.4, "policy_0") if cfg.use_per else buf.sample(B)
        info, prio, idx = tr.train_policy_on_batch(smp)
        if cfg.use_per:
            buf.update_priorities(idx, prio, "policy_0")
        tr.soft_target_updates()
        k = i & 1
        pins[k].copy_(tr._info[:4], non_blocking=True)
        evts[k].record()
        evts[k ^ 1].synchronize()
        return float(pins[k ^ 1][0])                                                  # D2H result of the PREVIOUS step

    evts[1].record()
    for i in range(min(4, E2E_WARM)):
        e2e_step_lagged(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(n_e2e):
        e2e_step_lagged(i)
    barrier()
    lag_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        torch.distributed.all_reduce(lag_s, op=torch.distributed.ReduceOp.MAX)
    e2e_lagged_sps = world * n_e2e / float(lag_s)

    # ---------------- per-kernel timing (eager, CUDA events on the launch stream) ----------------
    # every rank runs this loop: the eager step contains the all-reduce, so the collective counts must match on all ranks
    buf.rng = "device"
    tr.use_step_graph = False       # individual launches (with event marks between them), not the captured graph
    kern = {}
    reps, inner = PROFILE_REPS, PROFILE_INNER
    for rep in range(reps + 1):
        # `inner` eager steps are queued back to back (no host sync) so the GPU never waits for a launch: the
        # event-to-event intervals are then kernel durations, not host launch gaps; the first step of each burst is dropped
        lib.mx_profile_begin(sp())
        for _ in range(inner):
            if cfg.use_per:
                smp = buf.sample(B, 0.4, "policy_0")
            else:
                smp = buf.sample(B)
            info, prio, idx = tr.train_policy_on_batch(smp)
            if cfg.use_per:
                buf.update_priorities(idx, prio, "policy_0")
            tr.soft_target_updates()
        names = C.create_string_buffer(16384)
        ms = (C.c_float * 512)()
        n = lib.mx_profile_end(sp(), names, 16384, ms, 512)
        if rep >= 1:
            per = n // inner
            for k, (nm, t) in enumerate(zip(names.value.decode().split(";"), list(ms)[:n])):
                if k >= per:
                    kern.setdefault(nm, []).append(t)
    barrier()
    if rank != 0:
        # stay alive until rank 0 has printed its line, then leave without tearing NCCL down (destroy_process_group after
        # CUDA graphs that captured collectives can block at exit)
        torch.distributed.barrier()
        sys.stdout.flush()
        os._exit(0)
    kavg = {k: float(np.median(v)) for k, v in kern.items()}
    ksum = sum(kavg.values())
    fl, by = kernel_work(cfg, T, B, tr.P)
    if "k_gru_wgrad" in kavg:
        fl["k_front_bwd"] -= fl["k_gru_wgrad"]
    top = max(kavg, key=kavg.get)
    pk = peaks()
    if top in fl:
        ach = fl[top] / (kavg[top] * 1e-3) / 1e12
        roof = dict(bound="tensor", kernel=top, achieved=ach, peak=pk["tflops_sustained"], unit="TFLOP/s", frac=ach / pk["tflops_sustained"],
                    traffic=ncu_traffic(top), peak_source=pk["src"] + " bf16 sustained (kernel timed inside the step)",
                    note="FP32 FFMA kernel (1e-4 parity budget); serial-recurrence / latency bound at these sizes, see DESIGN.md")
    else:
        ach = by.get(top, 0.0) / (kavg[top] * 1e-3) / 1e9
        roof = dict(bound="hbm", kernel=top, achieved=ach, peak=pk["hbm"], unit="GB/s", frac=ach / pk["hbm"], traffic=ncu_traffic(top), peak_source=pk["src"])
    # latency model of the serial recurrences (SURVEY.md 8(d): "give the latency model alongside the roofline fraction"): the step
    # contains (T+1) dependent GRU steps forward (live and target nets side by side) and T backward; `floor` = the dependency chain of
    # one step counted from the SASS (LDS -> 4 FFMA2 -> 2 shuffles -> sigmoid -> tanh -> blend -> STS -> barrier; DESIGN.md section 4)
    csum = clocks.summary()
    sm_hz = 1e6 * float(csum.get("sm_mhz") or csum.get("sm_max_mhz") or 1965.0)
    t_f, t_b = kavg.get("k_gru_fwd"), kavg.get("k_gru_bwd")
    if t_f and t_b:
        FLOOR_F, FLOOR_B = 330.0, 230.0
        cyc_f, cyc_b = t_f * 1e-3 * sm_hz / (T + 1), t_b * 1e-3 * sm_hz / T
        floor_ms = ((T + 1) * FLOOR_F + T * FLOOR_B) / sm_hz * 1e3
        roof["latency_model"] = dict(serial_steps=2 * T + 1, t_step_cycles=dict(fwd=round(cyc_f, 1), bwd=round(cyc_b, 1)),
                                     floor_cycles=dict(fwd=FLOOR_F, bwd=FLOOR_B), chain_ms=round(t_f + t_b, 5), floor_ms=round(floor_ms, 5),
                                     frac=round(floor_ms / (t_f + t_b), 4), share_of_step=round((t_f + t_b) / ms_step, 4),
                                     sm_mhz=round(sm_hz / 1e6, 1))
    gather_gbs = by["k_gather"] / (kavg.get("k_gather", 1e9) * 1e-3) / 1e9
    breakdown = {k: dict(ms=round(v, 5), share=round(v / ksum, 4)) for k, v in sorted(kavg.items(), key=lambda kv: -kv[1])}

    # ---------------- CPU baseline (bounded sample) ----------------
    Ecpu = min(args.buffer, 1024)
    n_cpu = min(CPU_STEPS, 20 if args.workload == "qmix_3m" else 5)
    cores = best_cpu_threads(cfg, T, B, Ecpu, avail)
    sps_all, ms_all = cpu_learner_steps_per_s(cfg, T, B, Ecpu, n_cpu, 2, cores, avail)
    sps_one, ms_one = (sps_all, ms_all) if cores == 1 else cpu_learner_steps_per_s(cfg, T, B, Ecpu, n_cpu, 2, 1, avail)
    best = max(sps_all, sps_one)
    eager_gpu = None
    try:        # never let the secondary baseline break the bench line
        torch.set_num_threads(1)
        eager_gpu = torch_eager_gpu_steps_per_s(cfg, T, B, Ecpu, 10, 3, avail)
    except Exception as ex:
        sys.stderr.write("torch eager GPU baseline skipped: %r\n" % (ex,))

    value = world * 1000.0 / ms_step
    line = dict(
        metric="learner grad-steps/sec", value=value, unit="steps/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
        ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
        config=workload_config(args, cfg, T, B, world),
        notes=dict(grad_exchange=("all-reduce over NVLink peer memory INSIDE the optimiser kernel (k_optim_fused: {value, step} lines pushed to every peer, rank-ordered sum as they arrive)" if p2p
                                  else "NCCL all-reduce of the flat gradient buffer") if world > 1 else None,
                   value_definition="batch-%d grad-steps/s summed over ranks (each rank samples its own shard; one flat all-reduce)" % B,
                   replay_mb=round(pb.L.total_bytes / 1e6, 1),
                   step="CUDA graph: device MT19937 draw + gather + fused QMIX learner + one-launch reduce/clip/Adam/Polyak; state-only kernels (weight images, "
                        "mixer hypernets) on a forked graph branch beside the agent-net kernels" if (graph or tgraph) else "eager"),
        e2e=dict(value=e2e_sps, unit="steps/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h), steps=n_e2e,
                 host_rng_value=e2e_host_rng_sps,       # same loop with np.random drawn on the host per call (+ B*8 bytes H2D): the reference's own mode
                 lagged_read_value=e2e_lagged_sps,      # same loop, each step's loss read one step late (asynchronous logging)
                 path="RecReplayBuffer.insert(1 episode, pinned host memory -> H2D) + sample (NumPy's MT19937 stream continued on the device after "
                      "adopt_numpy_rng()) + QMix.train_policy_on_batch + soft_target_updates + D2H read of the loss, every step"),
        gpu_launches=launches, kernels_per_step=kernels_per_step,
        roofline=roof, kernels=breakdown, kernel_sum_ms=round(ksum, 5),        # > ms_per_step when branches of the step graph overlap
        gather_gbs=gather_gbs,
        cpu_baseline=dict(value=best, unit="steps/s", cores=cores if sps_all >= sps_one else 1, host_cores=os.cpu_count(), kind="port",
                          best_threads_steps_per_s=sps_all, one_thread_steps_per_s=sps_one,
                          sample="%d timed steps (sample+train+soft update) of the same workload on a %d-episode replay, oracle port of the reference learner" % (n_cpu, Ecpu)),
        torch_eager_gpu_baseline=dict(value=eager_gpu, unit="steps/s", kind="port",
                                      sample="10 timed steps of the oracle port of the reference learner with its networks on cuda:0 (eager PyTorch, "
                                             "host-side NumPy replay + H2D per step): the reference's own `--cuda` mode on this GPU"),
        clocks=clocks.summary())
    if exchange is not None:
        line["exchange"] = exchange
    emit(line)
    sys.stdout.flush()
    if graph is not None:
        graph.close()
    if world > 1:
        torch.distributed.barrier()
        os._exit(0)


# ---------------------------------------------------------------------------------------------------------
# MLP (transition-level) QMIX: SURVEY.md section 8(f).4 -- batches of single transitions from a large transition replay
# ---------------------------------------------------------------------------------------------------------
MLP_WORKLOADS = {
    # name: (n_agents, obs, act, state, B, transitions): MPE simple_spread shapes at the MLP scripts' batch / buffer sizes
    # (scripts/train_mpe_maddpg.sh:14: batch 1000, buffer 500 000; there is no recurrence, a transition is one replay row)
    "mqmix_mpe_spread": (3, 18, 5, 54, 1000, 500000),
}


def mlp_cfg(w):
    from offpolicy._b200.factory import LearnerConfig
    n, o, a, s, B, E = MLP_WORKLOADS[w]
    return LearnerConfig(n_agents=n, obs_dim=o, act_dim=a, state_dim=s, gain=1.0), B, E


def synth_steps(cfg, n, rs):
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    f32 = np.float32
    return [rs.standard_normal((n, N, O), dtype=f32), rs.standard_normal((n, S), dtype=f32), np.eye(A, dtype=f32)[rs.integers(0, A, (n, N))],
            np.repeat(rs.standard_normal((n, 1, 1), dtype=f32), N, 1), rs.standard_normal((n, N, O), dtype=f32), rs.standard_normal((n, S), dtype=f32),
            np.zeros((n, N, 1), f32), (rs.random((n, 1)) < 0.04).astype(f32), np.ones((n, N, 1), f32), None, None]


def mlp_cpu_steps_per_s(cfg, B, E, steps, warmup, threads):
    from oracle.mqmix import MqmixLearner, TransitionReplay
    cfg = oracle_cfg(cfg)
    torch.set_num_threads(threads)
    rs = np.random.default_rng(0)
    buf = TransitionReplay(E, cfg.n_agents, cfg.obs_dim, cfg.state_dim, cfg.act_dim, use_avail=False, reward_norm=False)
    for c in range(0, E, 8192):
        n = min(8192, E - c)
        buf.insert(n, *synth_steps(cfg, n, rs))
    torch.manual_seed(1)
    np.random.seed(1)
    L = MqmixLearner(cfg, seed=1)
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        out, inds = buf.sample(B)
        info, prio, _ = L.step(out)
        L.soft_update()
        float(info["loss"])
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    return 1.0 / float(np.median(times)), float(np.median(times)) * 1e3


def mlp_best_threads(cfg, B, E):
    cores = os.cpu_count() or 1
    best, best_sps = 1, 0.0
    for th in sorted({1, 4, 8, 16, min(32, cores)}):
        if th <= cores:
            sps, _ = mlp_cpu_steps_per_s(cfg, B, E, 5, 2, th)
            if sps > best_sps:
                best, best_sps = th, sps
    return best


def run_mlp(args):
    """M_QMix learner: sample(B transitions) -> train_policy_on_batch -> soft_target_updates (runner/mlp/base_runner.py batch_train)."""
    cfg, B, E_full = mlp_cfg(args.workload)
    N, O, A, S = cfg.n_agents, cfg.obs_dim, cfg.act_dim, cfg.state_dim
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if args.impl == "reference":
        E = min(E_full, 65536)
        cores = mlp_best_threads(cfg, B, E)
        sps, ms = mlp_cpu_steps_per_s(cfg, B, E, args.steps, args.warmup, cores)
        emit(dict(metric="learner grad-steps/sec", value=sps, unit="steps/s", impl="reference", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                  ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                  config=dict(workload=args.workload, batch=B, n_agents=N, obs_dim=O, act_dim=A, state_dim=S, buffer_transitions=E),
                  cpu_baseline=dict(value=sps, unit="steps/s", cores=cores, host_cores=os.cpu_count(), kind="port",
                                    sample="%d timed learner steps (sample+train+soft update), transition replay of %d" % (args.steps, E)),
                  e2e=dict(value=sps, unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0))
        return
    from offpolicy._b200 import capi
    from offpolicy._b200.graph import StepGraph
    from offpolicy.utils.mlp_buffer import MlpReplayBuffer
    from offpolicy._b200 import factory as mc
    torch.cuda.set_device(0)
    torch.set_num_threads(1)
    lib, dev = capi.lib(), capi.device()
    E = min(E_full, args.buffer * 100) if args.buffer != 5000 else E_full          # --buffer N (non-default) = N*100 transitions for quick runs
    info = {"policy_0": dict(obs_space=[O], share_obs_space=[S], act_space=mc.Discrete(A))}
    buf = MlpReplayBuffer(info, {"policy_0": list(range(N))}, E, True, False, max_batch=1024)        # the replay's batch limit (B = 1000 fits)
    rs = np.random.default_rng(0)
    d = lambda x: {"policy_0": x}
    for c in range(0, E, 1024):
        n = min(1024, E - c)
        buf.insert(n, *[d(x) for x in synth_steps(cfg, n, rs)])
    torch.manual_seed(1)
    np.random.seed(1)
    with contextlib.redirect_stdout(sys.stderr):
        margs, pol, tr = mc.build_mqmix(cfg, B, debug=False)
    rep = buf.policy_buffers["policy_0"].rep
    buf.seed_device_rng(1)
    sp = capi.stream_ptr
    torch.cuda.synchronize()
    graph = StepGraph(buf, tr, B)
    for _ in range(max(args.warmup, 3)):
        graph.launch()
    graph.synchronize()
    launches0 = lib.mx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        e0.record(graph.stream)
        for _ in range(args.steps):
            graph.launch()
        e1.record(graph.stream)
        torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / args.steps
    launches = int(lib.mx_launch_count() - launches0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, qmix_outputs(tr, rep, B))
    if args.quick:
        emit(dict(quick=True, workload=args.workload, value=1000.0 / ms_step, ms_per_step=ms_step, opts=args.opt, kernels_per_step=graph.num_kernels))
        graph.close()
        return

    # e2e: the runner's per-step sequence with host inputs: one freshly collected transition inserted (H2D), indices drawn on the host
    # (np.random.randint == np.random.choice, H2D), train, soft update, loss read back (D2H)
    buf.rng = "numpy"
    fresh = [synth_steps(cfg, 1, rs) for _ in range(8)]
    h2d = sum(x.nbytes for x in fresh[0] if x is not None) + B * 8

    def e2e_step(i):
        buf.insert(1, *[d(x) for x in fresh[i % 8]])
        info_t, _, _ = tr.train_policy_on_batch(buf.sample(B), True)
        tr.soft_target_updates()
        return float(info_t["loss"])

    for i in range(E2E_WARM):
        e2e_step(i)
    torch.cuda.synchronize()
    n_e2e = max(E2E_MIN_STEPS, min(args.steps, 200))
    t0 = time.perf_counter()
    for i in range(n_e2e):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_sps = n_e2e / (time.perf_counter() - t0)

    # per-kernel timing (eager launches, CUDA events on the launch stream)
    buf.seed_device_rng(2)
    tr.use_step_graph = False
    kern, reps, inner = {}, PROFILE_REPS, PROFILE_INNER
    for rep_i in range(reps + 1):
        lib.mx_profile_begin(sp())
        for _ in range(inner):
            tr.train_policy_on_batch(buf.sample(B), True)
            tr.soft_target_updates()
        names = C.create_string_buffer(16384)
        ms = (C.c_float * 512)()
        n = lib.mx_profile_end(sp(), names, 16384, ms, 512)
        if rep_i >= 1:
            per = n // inner
            for k, (nm, t) in enumerate(zip(names.value.decode().split(";"), list(ms)[:n])):
                if k >= per:
                    kern.setdefault(nm, []).append(t)
    kavg = {k: float(np.median(v)) for k, v in kern.items()}
    ksum = sum(kavg.values())
    H, ME, HY = 64, cfg.mixer_hidden, cfg.hyper_hidden
    M = 2 * B * N                                         # agent-net rows: obs and next obs of every agent
    mix = (S * HY + HY * N * ME) + (S * HY + HY * ME) + S * ME + (S * HY + HY) + N * ME + ME
    fl = {"k_front_fwd": 2 * 2.0 * M * (O * H + H * H + H * A), "k_front_fwd_tc": 2 * 2.0 * M * (O * H + H * H + H * A),
          "k_front_bwd": 2.0 * M * (2 * H * A + 3 * H * H + 3 * O * H) / 2, "k_mixer": 2.0 * B * mix * 4,
          "k_mix_hyper_fwd": 2.0 * B * (mix - N * ME - ME) * 2, "k_mix_hyper_bwd": 2.0 * B * (mix - N * ME - ME) * 2, "k_mix_core": 2.0 * B * (N * ME + ME) * 4}
    fields = 4.0 * B * (N * 2 * O + 2 * S + N * A + 3 * N + 1)
    by = {"k_gather": 2 * fields, "k_adam": 4.0 * tr.P * 7, "k_polyak": 4.0 * tr.P * 3, "k_grad_reduce": 4.0 * tr.P * 2}
    top = max(kavg, key=kavg.get)
    pk = peaks()
    if top in by:
        ach = by[top] / (kavg[top] * 1e-3) / 1e9
        roof = dict(bound="hbm", kernel=top, achieved=ach, peak=pk["hbm"], unit="GB/s", frac=ach / pk["hbm"], traffic=None, peak_source=pk["src"])
    else:
        ach = fl.get(top, 0.0) / (kavg[top] * 1e-3) / 1e12
        roof = dict(bound="tensor", kernel=top, achieved=ach, peak=pk["tflops_sustained"], unit="TFLOP/s", frac=ach / pk["tflops_sustained"], traffic=None,
                    peak_source=pk["src"] + " bf16 sustained (kernel timed inside the step)",
                    note="FP32 kernel (1e-4 parity budget); ~6000 agent-net rows per step: latency / occupancy bound, see DESIGN.md")
    Ecpu = min(E, 65536)
    cores = mlp_best_threads(cfg, B, Ecpu)
    sps_cpu, _ = mlp_cpu_steps_per_s(cfg, B, Ecpu, CPU_STEPS, 3, cores)
    emit(dict(metric="learner grad-steps/sec", value=1000.0 / ms_step, unit="steps/s", n_gpus=1, steps=args.steps, warmup=max(args.warmup, 3),
              ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
              config=dict(workload=args.workload, batch_transitions=B, n_agents=N, obs_dim=O, act_dim=A, state_dim=S, buffer_transitions=E,
                          l2="transitions gathered from a replay of %.0f MB (> L2)" % (rep.L.total_bytes / 1e6),
                          step="CUDA graph: device MT19937 draw + gather + fused MLP-QMIX learner + Adam + Polyak"),
              e2e=dict(value=e2e_sps, unit="steps/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=4, steps=n_e2e,
                       path="MlpReplayBuffer.insert(1 transition) + sample(np.random.choice) + M_QMix.train_policy_on_batch + soft_target_updates + D2H loss"),
              gpu_launches=launches, kernels_per_step=graph.num_kernels, roofline=roof,
              kernels={k: dict(ms=round(v, 5), share=round(v / ksum, 4)) for k, v in sorted(kavg.items(), key=lambda kv: -kv[1])}, kernel_sum_ms=round(ksum, 5),
              gather_gbs=by["k_gather"] / (kavg.get("k_gather", 1e9) * 1e-3) / 1e9,
              cpu_baseline=dict(value=sps_cpu, unit="steps/s", cores=cores, host_cores=os.cpu_count(), kind="port",
                                sample="%d timed steps (sample+train+soft update) on a %d-transition replay, oracle port of the reference M_QMix learner" % (CPU_STEPS, Ecpu)),
              clocks=clocks.summary()))
    graph.close()


_REAL_STDOUT = None


def emit(line):
    """The bench contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner on communicator
    creation, the drop-in classes' reference-style prints), so main() points fd 1 at stderr and the result goes to the saved fd."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="qmix_3m", choices=sorted(WORKLOADS) + sorted(MADDPG_WORKLOADS) + sorted(MLP_WORKLOADS))
    ap.add_argument("--buffer", type=int, default=5000, help="replay episodes (scripts/train_smac_qmix.sh default 5000)")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only (tuning sweeps; not the bench contract line)")
    ap.add_argument("--opt", action="append", default=[], help="engine option name=int (mx_set_option), e.g. --opt pdl=0 --opt front_tc=0")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the engine's outputs; the reference arm has none")
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl != "reference" and a.opt:
        from offpolicy._b200 import capi
        for kv in a.opt:
            k, v = kv.split("=")
            capi.check(capi.lib().mx_set_option(k.encode(), int(v)))
    if a.workload in MADDPG_WORKLOADS:
        if int(os.environ.get("RANK", "0")) == 0:
            run_maddpg(a)
        return
    if a.workload in MLP_WORKLOADS:
        run_mlp(a)
        return
    if a.impl == "reference":
        run_reference(a)
    else:
        run_engine(a)


if __name__ == "__main__":
    main()
