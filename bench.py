#!/usr/bin/env python
"""Benchmark of the learner hot paths named by BASELINE.json.

  python bench.py [--gpus N --steps K --warmup W] [--config cfg2|cfg3|cfg4] [--impl reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...       (one rank per GPU, NCCL; env-sharded, weak scaling)

Configs (BASELINE.json `configs`):
  cfg2 (default, the headline): ppo2 NatureCNN, synthetic 84x84x4 uint8, 4096 envs x 128 steps
  cfg3: ppo2 mlp, obs_dim 376 (Humanoid shape), 17-d Gaussian policy, value_network='copy', 16384 envs x 512 steps
  cfg4: deepq NatureCNN + dueling streams, prioritized replay of 1M transitions (tree capacity 2^20), batch 512

A PPO2 "step" is ONE full update: T+1 batched policy forwards over N envs, the GAE scan, and noptepochs x nminibatches
fused train steps (gather + forward + loss + backward + clip + Adam).  A deepq "step" is one train iteration: stratified
PER sample of 512 + IS weights, double-Q train step gathering from the resident replay, priority write-back.

Prints ONE JSON line (rank 0).  `value` times the step with inputs resident in HBM; `e2e` times the same metric
through the public host-facing path (host VecEnv: pinned obs -> H2D every env step, actions D2H every env step, loss
statistics D2H every update).  The default run also measures cfg3 and cfg4 briefly (`other_configs`) so that every
BASELINE config has a driver-visible number; `roofline_all` lists every kernel with its useful flops / bytes.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFGS = {
    "cfg2": dict(kind="ppo2", key="cfg2",
                 name="ppo2 NatureCNN synthetic 84x84x4 uint8, 4096 envs x 128 nsteps (BASELINE configs[1])",
                 network="cnn", ob_shape=(84, 84, 4), ob_dtype="uint8", n_actions=6, act_dim=None, nenvs=4096,
                 nsteps=128, nminibatches=4, noptepochs=4, lr=2.5e-4, cliprange=0.1, ent_coef=0.01, vf_coef=0.5,
                 max_grad_norm=0.5, gamma=0.99, lam=0.95, value_network=None, train_chunk=None,
                 flop_fwd=18.693e6, ref_envs=16, steps=3, warmup=3),
    "cfg3": dict(kind="ppo2", key="cfg3",
                 name="ppo2 mlp synthetic obs_dim=376 (Humanoid shape), 17-d Gaussian, value_network=copy, "
                      "16384 envs x 512 nsteps (BASELINE configs[2])",
                 network="mlp", ob_shape=(376,), ob_dtype="float32", n_actions=None, act_dim=17, nenvs=16384,
                 nsteps=512, nminibatches=32, noptepochs=10, lr=3e-4, cliprange=0.2, ent_coef=0.0, vf_coef=0.5,
                 max_grad_norm=0.5, gamma=0.99, lam=0.95, value_network="copy", train_chunk=262144,
                 flop_fwd=114944.0, ref_envs=64, steps=2, warmup=3),
    "cfg4": dict(kind="deepq", key="cfg4",
                 name="deepq NatureCNN + dueling, prioritized replay 1M transitions (tree 2^20) of 84x84x4 uint8, "
                      "batch 512 (BASELINE configs[3])",
                 network="cnn", ob_shape=(84, 84, 4), n_actions=6, buffer_size=1000000, batch=512, alpha=0.6, beta=0.4,
                 lr=1e-4, gamma=0.99, train_freq=4, steps=200, warmup=20),
}


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = []
        for i, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(s[3 + i].lower().startswith("active") for s in self.samples):
                reasons.append(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks.update(json.load(open(pk)))
        peaks["src"] = "measured"
    return peaks


# ---------------------------------------------------------------------------------------------- CPU reference arms
def cpu_reference_update(cfg, nenvs_sample, threads=None, steps=1, warmup=0):
    """The reference's CPU path for one PPO2 update (TF1 unavailable -> oracle port, torch-CPU fp32), with the
    reference's structure: T+1 batched forwards (runner.py:26-50), numpy GAE (:53-65), host shuffle + minibatch
    loop (ppo2.py:157-166) with per-minibatch normalisation, clip, Adam.  Per-sample work identical to cfg;
    only the env count is reduced (bounded sample)."""
    import torch
    from oracle import nets
    from oracle.gae import gae_reference_order, sf01
    if threads:
        torch.set_num_threads(threads)
    T, n = cfg["nsteps"], nenvs_sample
    rng = np.random.RandomState(0)
    np.random.seed(0)
    discrete = cfg["act_dim"] is None
    nA = cfg["n_actions"] if discrete else cfg["act_dim"]
    params = nets.init_policy_params(cfg["network"], cfg["ob_shape"], "discrete" if discrete else "box", nA,
                                     value_network=cfg["value_network"])
    oracle = nets.PPO2Oracle(params, cfg["network"], cfg["ent_coef"], cfg["vf_coef"], cfg["max_grad_norm"],
                             value_network=cfg["value_network"])
    if cfg["ob_dtype"] == "uint8":
        pool = [rng.randint(0, 256, (n,) + tuple(cfg["ob_shape"])).astype(np.uint8) for _ in range(8)]
    else:
        pool = [np.clip(rng.randn(n, *cfg["ob_shape"]), -10, 10).astype(np.float32) for _ in range(8)]
    rews = rng.randn(64, n).astype(np.float32)
    dones = rng.rand(64, n) < 0.01
    nmb = cfg["nminibatches"]
    while (n * T) % nmb or (n * T) // nmb < 1:
        nmb //= 2
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        mb_obs, mb_act, mb_val, mb_nlp, mb_done, mb_rew = [], [], [], [], [], []
        d = np.zeros(n, bool)
        for t in range(T):
            obs = pool[t % 8]
            noise = (rng.rand(n, nA).astype(np.float32) * 0.998 + 0.001) if discrete else rng.randn(n, nA).astype(np.float32)
            a, v, nlp, _ = oracle.step(obs, noise)
            mb_obs.append(obs.copy()); mb_act.append(a); mb_val.append(v); mb_nlp.append(nlp); mb_done.append(d)
            d = dones[t % 64]
            mb_rew.append(rews[t % 64])
        last_v = oracle.value(pool[T % 8])
        mb_obs, mb_rew, mb_val = np.asarray(mb_obs), np.asarray(mb_rew, np.float32), np.asarray(mb_val, np.float32)
        adv, ret = gae_reference_order(mb_rew, mb_val, np.asarray(mb_done), last_v, d, cfg["gamma"], cfg["lam"])
        obs_f, ret_f, act_f, val_f, nlp_f = map(sf01, (mb_obs, ret, np.asarray(mb_act), mb_val, np.asarray(mb_nlp, np.float32)))
        nbatch = n * T
        nbt = nbatch // nmb
        inds = np.arange(nbatch)
        for _ in range(cfg["noptepochs"]):
            np.random.shuffle(inds)
            for s in range(0, nbatch, nbt):
                mb = inds[s:s + nbt]
                oracle.train(cfg["lr"], cfg["cliprange"], obs_f[mb], ret_f[mb], None, act_f[mb], val_f[mb], nlp_f[mb])
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return n * T, times


def cpu_reference_deepq(cfg, threads=None, steps=2, warmup=1, cap=1 << 16):
    """The reference's CPU path for one deepq train iteration (deepq.py:292-303): python PrioritizedReplayBuffer
    sample (oracle port of replay_buffer.py:107-167 on a tree of `cap` leaves -- the python descent costs log2(cap)
    per sample, 16 vs 20 levels), observation gather, the TF graph of build_graph.py:388-430 (oracle port, torch-CPU
    fp32: three forwards + backward at batch 512), update_priorities."""
    import random
    import torch
    from oracle import nets
    from oracle.segment_tree import PrioritizedSampler
    if threads:
        torch.set_num_threads(threads)
    B, nA = cfg["batch"], cfg["n_actions"]
    rng = np.random.RandomState(0)
    qp = nets.init_q_params(cfg["network"], cfg["ob_shape"], nA, hiddens=(256,), dueling=True, seed=0)
    oracle = nets.DQNOracle(qp, cfg["network"], cfg["gamma"], n_hidden=1, dueling=True, grad_norm_clipping=10.0)
    pool = rng.randint(0, 256, (2048,) + tuple(cfg["ob_shape"])).astype(np.uint8)
    ps = PrioritizedSampler(cap, cfg["alpha"])
    for _ in range(cap):
        ps.add()
    ps.update_priorities(list(range(0, cap, 7)), list(np.abs(rng.randn(len(range(0, cap, 7)))) + 1e-6))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        idx = ps.sample_idx([random.random() for _ in range(B)])
        w = ps.weights(idx, cfg["beta"]).astype(np.float32)
        ii = np.asarray(idx) % 2048
        o_t, o_1 = pool[ii], pool[(ii + 1) % 2048]
        act = rng.randint(0, nA, B)
        td = oracle.train(cfg["lr"], o_t, act, rng.randn(B).astype(np.float32), o_1, np.zeros(B, np.float32), w)
        ps.update_priorities(idx, list(np.abs(td) + 1e-6))
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return B, times


def pick_cpu_threads():
    """All the host threads the CPU path can USE: torch intra-op threads beyond the physical cores this
    process may run on only add contention (128 threads were 100x slower than 8 on the first box), so probe a
    small conv workload over candidate counts <= the affinity mask and keep the fastest."""
    import torch
    import torch.nn.functional as F
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (4, 8, 16, 32, 64, avail) if c <= avail}) or [1]
    x = torch.randn(64, 4, 84, 84)
    w = torch.randn(32, 4, 8, 8)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        F.conv2d(x, w, stride=4)
        t0 = time.perf_counter()
        for _ in range(3):
            F.conv2d(x, w, stride=4)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def metric_of(cfg):
    if cfg["kind"] == "deepq":
        return "deepq learner transitions/sec (PER sample + double-Q train step + priority update, batch 512)", "transitions/s"
    return "PPO2 learner env-steps/sec", "env-steps/s"


def run_reference(args, cfg):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = pick_cpu_threads()
    metric, unit = metric_of(cfg)
    if cfg["kind"] == "deepq":
        nb, times = cpu_reference_deepq(cfg, threads=threads, steps=max(1, min(args.steps, 5)), warmup=1)
        sample = "one train iteration at batch 512 per step (python PER port on a 2^16-leaf tree + torch-CPU fp32 oracle " \
                 "port of the TF1 graph)"
    else:
        n = args.ref_envs or cfg["ref_envs"]
        nb, times = cpu_reference_update(cfg, n, threads=threads, steps=args.steps, warmup=min(args.warmup, 1))
        sample = f"{n} envs x {cfg['nsteps']} steps per update (same per-sample work as {cfg['nenvs']} envs), " \
                 f"torch-CPU fp32 oracle port"
    ms = 1000.0 * float(np.mean(times))
    val = nb / (ms / 1000.0)
    out = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": min(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": cfg["name"], "sample": sample},
           "cpu_baseline": {"value": val, "unit": unit, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
           "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------- rooflines
def summarize_profile(prof, steps):
    """prof: {label: [ms, calls, flops, bytes]} accumulated over the timed region."""
    out = {}
    for label, (ms, calls, flops, nbytes) in prof.items():
        out[label] = {"ms_per_step": ms / steps, "launches_per_step": calls / steps,
                      "flops_per_step": flops / steps, "bytes_per_step": nbytes / steps}
        if flops:
            out[label]["tflops"] = flops / (ms / 1e3) / 1e12 if ms else None
        if nbytes:
            out[label]["gbs"] = nbytes / (ms / 1e3) / 1e9 if ms else None
    return out


# bench label -> kernel template instance (conv_shift.cu dispatch for the NatureCNN layers): <BN,KH,DACT,U8,KX> for the
# forward / dgrad kernel, <BN,KH,U8,KX> for the wgrad kernel
TRAFFIC_KERNEL = {
    "convs.fwd.pi/c1": "conv_shift_fwd_kernel<32, 1, 0, 1, 1>", "convs.fwd.pi/c2": "conv_shift_fwd_kernel<64, 2, 0, 0, 1>",
    "convs.fwd.pi/c3": "conv_shift_fwd_kernel<64, 1, 0, 0, 1>", "convs.dgrad.pi/c3": "conv_shift_fwd_kernel<64, 1, 1, 0, 1>",
    "convs.dgrad.pi/c2": "conv_shift_fwd_kernel<128, 1, 1, 0, 1>", "convs.wgrad.pi/c1": "conv_shift_wgrad_kernel<32, 1, 1, 2>",
    "convs.wgrad.pi/c2": "conv_shift_wgrad_kernel<64, 2, 0, 2>", "convs.wgrad.pi/c3": "conv_shift_wgrad_kernel<64, 1, 0, 3>",
}


def load_traffic():
    """DRAM bytes per SAMPLE of each conv kernel instance from the committed `ncu --set full` capture
    (profiles/r2_traffic.json, written by `tools/summarize_ncu.py traffic <rep> ... <samples>` from the .ncu-rep raw
    page: dram__bytes_read.sum + dram__bytes_write.sum of one launch / the samples that launch processed).  bench
    multiplies by the samples one of ITS launches processes; every launch here and in the capture is >> L2."""
    tj = os.path.join(ROOT, "profiles", "r2_traffic.json")
    return json.load(open(tj)) if os.path.exists(tj) else {}


def kernel_roofline(name, k, peaks, traffic=None):
    n_launch = max(1.0, k["launches_per_step"])
    f_tensor = f_hbm = 0.0
    if k.get("flops_per_step"):
        f_tensor = k["flops_per_step"] / (k["ms_per_step"] / 1e3) / 1e12 / peaks["bf16_tflops_sustained"]
    if k.get("bytes_per_step"):
        f_hbm = k["bytes_per_step"] / (k["ms_per_step"] / 1e3) / 1e9 / peaks["hbm_gbs"]
    if f_tensor >= f_hbm:
        r = {"kernel": name, "bound": "tensor", "achieved": f_tensor * peaks["bf16_tflops_sustained"],
             "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": f_tensor,
             "peak_src": peaks["src"] + " (sustained cuBLAS bf16: kernel timed inside a long step)"}
    else:
        r = {"kernel": name, "bound": "hbm", "achieved": f_hbm * peaks["hbm_gbs"], "peak": peaks["hbm_gbs"],
             "unit": "GB/s", "frac": f_hbm, "peak_src": peaks["src"] + " (copy bandwidth)"}
    t = (traffic or {}).get(TRAFFIC_KERNEL.get(name.split("@")[0], ""))
    samples = k.get("samples_per_launch")
    r.update({"traffic": t["dram_bytes_per_sample"] * samples if t and samples else None,
              "traffic_src": (t.get("src") + f", {t['capture_samples']} samples/launch, scaled per sample") if t else None,
              "algorithmic_bytes_per_launch": k.get("bytes_per_step", 0.0) / n_launch,
              "algorithmic_flops_per_launch": k.get("flops_per_step", 0.0) / n_launch,
              "flops_are": "useful (valid conv outputs only)", "frac_tensor": f_tensor, "frac_hbm": f_hbm,
              "ms_per_launch": k["ms_per_step"] / n_launch, "launches_per_step": n_launch, "share_of_step": k.get("share")})
    return r


# ---------------------------------------------------------------------------------------------- --dump-outputs
DUMP_ROWS = 1 << 19          # rollout rows written per array: all of cfg2's 524288, a fixed sample of cfg3's 8.4 M
DUMP_LIMIT = 64 << 20        # bytes over all files


def sample_rows(n, device):
    """Rows of an n-row rollout array that --dump-outputs writes: all of them, or a seeded sample of DUMP_ROWS that is
    the same in every run, so that two builds can be compared row for row."""
    import torch
    if n <= DUMP_ROWS:
        return slice(None)
    return torch.from_numpy(np.sort(np.random.RandomState(0).choice(n, DUMP_ROWS, replace=False))).to(device)


def seeded_state_restorer(tensors, opt, refresh):
    """-> a callable that puts the learner back into its state of now (the seeded start): `tensors` (parameters, Adam
    moments, for deepq the priority trees) get their current values again, the Adam step count goes back, and
    `refresh` rebuilds what is derived from the parameters.  The gradient, norm and loss reductions of a train step
    use float atomics, so the state after an update differs in the last bits from run to run, and later updates turn
    those bits into different sampled actions or replay indices.  --dump-outputs calls it before the last timed step:
    that step's inputs are then the same in every run, and its outputs differ at most by the rounding of its own
    reductions."""
    saved, t = [x.clone() for x in tensors], opt.t

    def restore():
        for x, s in zip(tensors, saved):
            x.copy_(s)
        opt.t = t
        refresh()
    return restore


def dump_outputs(out_dir, arrays):
    """Write {name: tensor or ndarray} as out_dir/<name>.npy.  float64 stays float64, everything else is written as
    float32 (the integer outputs -- actions, replay indices -- are below 2^24 and stay exact)."""
    import torch
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        out[name.replace("/", ".").replace(":", "_")] = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- PPO2 arm
def run_ppo2(cfg, args, steps, warmup, with_profile, with_e2e, dist_ctx, dump_dir=None):
    import torch
    import torch.distributed as dist
    from baselines_b200 import _lib
    from baselines_b200.common.policies import build_policy
    from baselines_b200.common.vec_env import DeviceSyntheticVecEnv, SyntheticVecEnv
    from baselines_b200.ppo2.model import Model
    from baselines_b200.ppo2.ppo2 import run_epochs
    from baselines_b200.ppo2.runner import Runner
    rank, local_rank, world = dist_ctx
    N, T = cfg["nenvs"], cfg["nsteps"]
    nbatch = N * T
    nbatch_train = nbatch // cfg["nminibatches"]
    dev = torch.device("cuda", local_rank)
    np.random.seed(0)
    ob_dtype = np.dtype(cfg["ob_dtype"])
    env_kw = dict(n_actions=cfg["n_actions"] or 6, act_dim=cfg["act_dim"])

    def make(env):
        policy = build_policy(env, cfg["network"], value_network=cfg["value_network"])
        model = Model(policy=policy, ob_space=env.observation_space, ac_space=env.action_space, nbatch_act=N,
                      nbatch_train=nbatch_train, nsteps=T, ent_coef=cfg["ent_coef"], vf_coef=cfg["vf_coef"],
                      max_grad_norm=cfg["max_grad_norm"], comm=None if world > 1 else False,
                      train_chunk=cfg["train_chunk"])
        return model, Runner(env=env, model=model, nsteps=T, gamma=cfg["gamma"], lam=cfg["lam"])

    last = {}

    def update(model, runner):
        ro, _ = runner.run_device()
        st = run_epochs(model, ro, cfg["lr"], cfg["cliprange"], nbatch, nbatch_train, cfg["noptepochs"], dev,
                        shuffle=args.shuffle)
        last["stats"] = st
        return torch.stack(st).mean(dim=0)

    def timed(model, runner, steps, warmup, read_back, profile=False, before_last=None):
        for _ in range(warmup):
            update(model, runner)
        torch.cuda.synchronize()
        if profile:
            _lib.profile_begin()                                 # per-call events: graphs.py falls back to eager launches
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms, launches = 0.0, 0
        for i, n in enumerate([steps] if before_last is None else [steps - 1, 1]):
            if i == 1:                                           # between the two timed windows
                before_last()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = _lib.LAUNCHES
            e0.record()
            for _ in range(n):
                st = update(model, runner)
                if read_back:
                    st.cpu()                                     # the loss statistics a user reads each update
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
            launches += _lib.LAUNCHES - l0
        if world > 1:
            dist.barrier()
        ms = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, launches / steps

    # ---- device-resident value: first un-instrumented (the headline), then once more with per-call CUDA events
    env_d = DeviceSyntheticVecEnv(N, cfg["ob_shape"], ob_dtype, seed=rank, device=dev, **env_kw)
    model, runner = make(env_d)
    reseed = None
    if dump_dir:
        store = model.net.store
        reseed = seeded_state_restorer([store.params, store.m, store.v], model.opt, model.net.refresh)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step, launches = timed(model, runner, steps, warmup, read_back=False, before_last=reseed)
    clocks = sampler.stop() if rank == 0 else None
    if dump_dir and rank == 0:
        st = torch.stack(last["stats"])
        out = {"loss_stats": st.mean(dim=0), "loss_stats_per_minibatch": st,
               "last_values": runner.rollout.last_values}
        rows = sample_rows(nbatch, dev)
        for name in ("actions", "values", "neglogpacs", "advs", "returns"):
            out["rollout_" + name] = runner.rollout.flat(name)[rows]
        out.update(("params." + k, v) for k, v in model.get_params().items())
        dump_outputs(dump_dir, out)
    prof = None
    ms_prof = None
    if with_profile:
        ms_prof, _ = timed(model, runner, max(1, min(steps, 2)), 0, read_back=False, profile=True)
        prof = (_lib.profile_end(), max(1, min(steps, 2)))
    value = world * nbatch / (ms_step / 1000.0)
    # every rank's own kernel-time sum (eager profile pass): with 16 synchronising all-reduces per update the job runs at
    # the pace of the slowest GPU, so a per-GPU spread shows up 1:1 in the N-GPU step time
    per_rank_kernel_ms = None
    if prof is not None and world > 1:
        mine = torch.tensor([sum(v[0] for v in prof[0].values()) / prof[1]], device=dev)
        allk = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allk, mine)
        per_rank_kernel_ms = [round(float(t.item()), 2) for t in allk]

    # ---- e2e through the host VecEnv
    e2e = None
    if with_e2e:
        del runner, env_d
        torch.cuda.empty_cache()
        ob_bytes = int(np.prod(cfg["ob_shape"])) * ob_dtype.itemsize
        act_bytes = 8 if cfg["act_dim"] is None else 4 * cfg["act_dim"]
        common_h2d = T * N * 5 + cfg["noptepochs"] * nbatch * 8          # rewards + dones + minibatch permutations
        d2h = T * N * act_bytes + 40
        unit = "env-steps/s"
        if cfg["network"] == "cnn" and cfg["ob_shape"][-1] == 4:
            # (a) the reference's Atari pipeline (run.py build_env): VecFrameStack(venv, 4).  The env produces ONE new
            #     84x84x1 frame per step; our VecFrameStack keeps the stack in HBM, so only new frames cross PCIe.
            from baselines_b200.common.vec_env import VecFrameStack
            frame_shape = tuple(cfg["ob_shape"][:-1]) + (1,)
            env_f = VecFrameStack(SyntheticVecEnv(N, frame_shape, np.uint8, seed=rank, **env_kw), 4)
            runner_f = Runner(env=env_f, model=model, nsteps=T, gamma=cfg["gamma"], lam=cfg["lam"])
            ms_f, _ = timed(model, runner_f, max(1, steps), 3, read_back=True)   # eager pass, capture pass, replay pass
            e2e = {"value": world * nbatch / (ms_f / 1000.0), "unit": unit, "ms_per_step": ms_f,
                   "h2d_bytes_per_step": T * N * (ob_bytes // 4 + 1) + common_h2d, "d2h_bytes_per_step": d2h,
                   "input": "VecFrameStack(host VecEnv of 84x84x1 frames, 4): new frames uploaded, stack kept in HBM"}
            del runner_f, env_f
            torch.cuda.empty_cache()
        # (b) a host VecEnv that hands out full observations: every one of them is uploaded
        env_h = SyntheticVecEnv(N, cfg["ob_shape"], ob_dtype, seed=rank, **env_kw)
        runner_h = Runner(env=env_h, model=model, nsteps=T, gamma=cfg["gamma"], lam=cfg["lam"])
        ms_e2e, _ = timed(model, runner_h, max(1, steps), 3, read_back=True)
        full = {"value": world * nbatch / (ms_e2e / 1000.0), "unit": unit, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": (T + 1) * N * ob_bytes + common_h2d, "d2h_bytes_per_step": d2h,
                "input": "host VecEnv handing out full observations: all of them uploaded"}
        if e2e is None:
            e2e = full
        else:
            e2e["stacked_upload"] = full
        del runner_h, env_h
    res = dict(value=value, ms_step=ms_step, launches=launches, clocks=clocks, e2e=e2e, prof=prof, ms_prof=ms_prof,
               chunk=model.chunk, nbatch=nbatch, per_rank_kernel_ms=per_rank_kernel_ms)
    del model
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------- deepq arm
def run_deepq(cfg, args, steps, warmup, with_profile, with_e2e, dist_ctx, dump_dir=None):
    import random
    import torch
    from baselines_b200 import _lib
    from baselines_b200.common import spaces
    from baselines_b200.common.vec_env import SyntheticVecEnv
    from baselines_b200.deepq.build_graph import DQNModel
    from baselines_b200.deepq.replay_buffer import PrioritizedReplayBuffer
    rank, local_rank, world = dist_ctx
    dev = torch.device("cuda", local_rank)
    B, nA = cfg["batch"], cfg["n_actions"]
    np.random.seed(0)
    random.seed(0)
    model = DQNModel(spaces.Box(0, 255, cfg["ob_shape"], np.uint8), nA, cfg["network"], lr=cfg["lr"], gamma=cfg["gamma"],
                     grad_norm_clipping=10, batch_cap=B, seed=0, hiddens=(256,), dueling=True)
    rb = PrioritizedReplayBuffer(cfg["buffer_size"], cfg["alpha"], device=dev)
    g = torch.Generator(device=dev).manual_seed(rank)
    n_fill, blk = cfg["buffer_size"], 32768
    for s in range(0, n_fill, blk):                              # synthetic transitions generated on the device
        k = min(blk, n_fill - s)
        o = torch.randint(0, 256, (k,) + tuple(cfg["ob_shape"]), dtype=torch.uint8, device=dev, generator=g)
        rb.add_batch(o, torch.randint(0, nA, (k,), device=dev, generator=g), torch.randn(k, device=dev, generator=g),
                     o.flip(0), (torch.rand(k, device=dev, generator=g) < 0.01).float())
    pr = (torch.randn(n_fill, device=dev, generator=g).abs().double() + 1e-6) ** cfg["alpha"]   # |N(0,1)| + 1e-6 (SURVEY 8d)
    rb._set_priorities(torch.arange(n_fill, device=dev), pr)
    torch.cuda.synchronize()

    last = {}

    def step():
        idx, w32, _ = rb.sample_device(B, beta=cfg["beta"])
        td = model.train_device(rb._obs_t, rb._obs_tp1, rb._actions, rb._rewards, rb._dones, w32, idx, B)
        rb.update_priorities_device(idx, td, 1e-6)
        last.update(sample_idx=idx, sample_weights=w32, td_errors=td)

    def timed(fn, steps, warmup, profile=False, before_last=None):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if profile:
            _lib.profile_begin()
        ms, launches = 0.0, 0
        for i, n in enumerate([steps] if before_last is None else [steps - 1, 1]):
            if i == 1:                                           # between the two timed windows
                before_last()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = _lib.LAUNCHES
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
            launches += _lib.LAUNCHES - l0
        return ms / steps, launches / steps

    reseed = None
    if dump_dir:
        q = model.q.store
        reseed = seeded_state_restorer([q.params, q.m, q.v, rb._it_sum, rb._it_min, rb._maxp_dev], model.opt,
                                       model.q.refresh)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step, launches = timed(step, steps, warmup, before_last=reseed)
    clocks = sampler.stop() if rank == 0 else None
    if dump_dir and rank == 0:
        out = dict(last)
        out["priorities"] = rb._it_sum[rb._cap + last["sample_idx"]]          # the leaves the step rewrote
        out.update(("params." + k, v) for k, v in model.q.store.export_tf("params").items())
        dump_outputs(dump_dir, out)
    prof = None
    if with_profile:
        timed(step, 20, 0, profile=True)
        prof = (_lib.profile_end(), 20)
    value = world * B / (ms_step / 1000.0)
    e2e = None
    if with_e2e:
        # the deepq.learn loop body (deepq.py:259-307) on a host env: act on one observation (uploaded), step the env,
        # replay.add (pinned staging), and every train_freq-th step the train iteration above
        from baselines_b200.deepq.build_graph import build_act
        act = build_act(model)
        env = SyntheticVecEnv(1, cfg["ob_shape"], np.uint8, n_actions=nA, seed=rank)
        obs = env.reset()[0]
        tf = cfg["train_freq"]
        state = {"obs": obs, "t": 0}

        def env_steps():                                      # train_freq env steps + one train iteration
            for _ in range(tf):
                a = act(state["obs"][None], update_eps=0.1)[0]
                o1, r, d, _ = env.step(np.array([a]))
                rb.add(state["obs"], a, float(r[0]), o1[0], float(d[0]))
                state["obs"] = o1[0]
            step()
        ms_g, _ = timed(env_steps, max(10, steps // 4), 5)
        ob_bytes = int(np.prod(cfg["ob_shape"]))
        e2e = {"value": world * B / (ms_g / 1000.0), "unit": "transitions/s", "ms_per_step": ms_g,
               "env_steps_per_s": world * tf / (ms_g / 1000.0),
               "h2d_bytes_per_step": tf * (3 * ob_bytes + 16) + B * 8, "d2h_bytes_per_step": tf * 8 + 8,
               "input": f"deepq.learn loop body on a host env: {tf} x (act on 1 uploaded obs, env.step, replay.add) + 1 train "
                        f"iteration; train_freq={tf}"}
    res = dict(value=value, ms_step=ms_step, launches=launches, clocks=clocks, e2e=e2e, prof=prof, ms_prof=None,
               chunk=None, nbatch=B)
    del model, rb
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------- main
def main():
    # some images export NCCL_DEBUG=VERSION, which prints a banner on stdout next to the JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CFGS))
    ap.add_argument("--nenvs", type=int, default=None, help="envs per GPU (default: the BASELINE config)")
    ap.add_argument("--ref-envs", type=int, default=None, help="envs in the bounded CPU-reference sample")
    ap.add_argument("--shuffle", default="device", choices=["device", "host"],
                    help="minibatch permutation: keyed bijection kernel (default) or the reference's host np.random.shuffle")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel CUDA-event profile pass")
    ap.add_argument("--no-targets", action="store_true", help="skip the stand-alone GAE / fc1 / PER microbenchmarks")
    ap.add_argument("--no-others", action="store_true", help="default config only: skip the short cfg3 / cfg4 measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MB); that step starts from "
                         "the learner's seeded state, so its inputs are the same in every run")
    args = ap.parse_args()
    cfg = dict(CFGS[args.config])
    if args.nenvs and cfg["kind"] == "ppo2":
        cfg["nenvs"] = args.nenvs
    if args.steps is None:
        args.steps = cfg["steps"]
    if args.warmup is None:
        args.warmup = cfg["warmup"]
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    ctx = (rank, local_rank, world)
    runner_fn = run_deepq if cfg["kind"] == "deepq" else run_ppo2
    res = runner_fn(cfg, args, args.steps, args.warmup, not args.no_profile, not args.no_e2e, ctx, args.dump_outputs)

    # short, driver-visible measurements of the other BASELINE configs (N = 1 only: they are single-GPU configs)
    others = None
    if args.config == "cfg2" and world == 1 and not args.no_others and not args.nenvs:
        others = {}
        for key in ("cfg3", "cfg4"):
            oc = dict(CFGS[key])
            try:
                fn = run_deepq if oc["kind"] == "deepq" else run_ppo2
                r = fn(oc, args, oc["steps"], oc["warmup"], True, True, ctx)
                m, u = metric_of(oc)
                others[key] = {"metric": m, "unit": u, "workload": oc["name"], "value": r["value"],
                               "ms_per_step": r["ms_step"], "steps": oc["steps"], "warmup": oc["warmup"],
                               "gpu_launches_per_step": r["launches"], "e2e": r["e2e"], "train_chunk": r["chunk"],
                               "kernels": _kernels_of(r)}
            except Exception as ex:                              # never lose the headline line to an extra
                others[key] = {"error": repr(ex)}
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    traffic = load_traffic()
    kernels = _kernels_of(res)
    roofline, roofline_all = None, []
    if kernels and cfg["kind"] == "ppo2":
        per = {"train": min(res.get("chunk") or 1 << 62, cfg["nenvs"] * cfg["nsteps"] // cfg["nminibatches"]),
               "act": cfg["nenvs"]}
        for name, k in kernels.items():
            k["samples_per_launch"] = per.get(name.split("@")[-1])
    if kernels:
        for name, k in sorted(kernels.items(), key=lambda kv: -kv[1]["ms_per_step"]):
            if k.get("flops_per_step") or k.get("bytes_per_step"):
                roofline_all.append(kernel_roofline(name, k, peaks, traffic))
        if roofline_all:
            roofline = roofline_all[0]

    metric, unit = metric_of(cfg)
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:              # rank 0 at N=1 only (contract)
        th = pick_cpu_threads()
        if cfg["kind"] == "deepq":
            nb, times = cpu_reference_deepq(cfg, threads=th, steps=2, warmup=1)
            sample = "2 train iterations at batch 512 (python PER port on a 2^16-leaf tree + torch-CPU fp32 oracle port)"
        else:
            n = args.ref_envs or cfg["ref_envs"]
            nb, times = cpu_reference_update(cfg, n, threads=th, steps=1, warmup=0)
            sample = f"one PPO2 update on {n} envs x {cfg['nsteps']} steps (same per-sample work), torch-CPU fp32 " \
                     f"oracle port of the TF1 graph"
        cpu_baseline = {"value": nb / float(np.mean(times)), "unit": unit, "cores": torch.get_num_threads(),
                        "kind": "port", "sample": sample}

    targets = None
    try:
        if args.no_targets or world > 1:
            raise RuntimeError("skipped (--no-targets or N > 1: stand-alone kernels are a 1-GPU measurement)")
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import microbench
        mb = microbench.run(quick=True)
        targets = {"gae": mb.get("gae"), "fc1": mb.get("fc1"), "gae_cpu_numpy": mb.get("gae_cpu"),
                   "per_cfg4": mb.get("per"), "replay_gather_cfg4": mb.get("replay_gather"), "dqn_cfg4": mb.get("dqn"),
                   "how": mb["l2_flush"] + "; CUDA events per launch, median of 10 after 3 warm-ups"}
        # the stand-alone targets as roofline entries (burst peaks: kernels timed alone)
        for gcase in mb.get("gae") or []:
            if isinstance(gcase, dict) and "gbs" in gcase:
                roofline_all.append({"kernel": f"gae_scan T={gcase['T']} N={gcase['N']} ({gcase['bytes'] / 1e6:.0f} MB, "
                                               f"variant {gcase['variant']})", "bound": "hbm", "achieved": gcase["gbs"],
                                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gcase["gbs"] / peaks["hbm_gbs"],
                                     "ms_per_launch": gcase["ms"], "algorithmic_bytes_per_launch": gcase["bytes"],
                                     "traffic": (traffic.get(f"gae_scan_{gcase['T']}x{gcase['N']}") or {}).get("dram_bytes_per_launch"),
                                     "stand_alone": True, "target": 0.6})
        for c in mb.get("fc1") or []:
            if isinstance(c, dict) and "tflops" in c:
                roofline_all.append({"kernel": f"fc1 {c['kind']} M={c['M']} K={c['K']} N={c['N']}", "bound": "tensor",
                                     "achieved": c["tflops"], "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                                     "frac": c["tflops"] / peaks["bf16_tflops"], "ms_per_launch": c["ms"],
                                     "algorithmic_flops_per_launch": c["flops"], "stand_alone": True, "target": 0.5})
        rg = mb.get("replay_gather")
        if isinstance(rg, dict) and "gbs" in rg:
            roofline_all.append({"kernel": "replay obs gather (512 x 2 x 28224 B, uint8 -> fp16)", "bound": "hbm",
                                 "achieved": rg["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": rg["gbs"] / peaks["hbm_gbs"], "ms_per_launch": rg["ms"], "stand_alone": True})
    except Exception as ex:                                    # never lose the headline line to an extra
        targets = {"error": repr(ex)}

    if cfg["kind"] == "ppo2":
        N, T = cfg["nenvs"], cfg["nsteps"]
        tf_step = (T + 1) * N * cfg["flop_fwd"] + cfg["noptepochs"] * N * T * 3 * cfg["flop_fwd"]
        config = {"workload": cfg["name"], "envs_per_gpu": N, "nsteps": T, "nminibatches": cfg["nminibatches"],
                  "noptepochs": cfg["noptepochs"], "parallelism": f"dp{world} (env-sharded, grad allreduce)",
                  "l2": "inputs larger than L2 (rollout observations %.1f GB, every minibatch streams %.2f GB)" %
                        (N * T * np.prod(cfg["ob_shape"]) * (1 if cfg["ob_dtype"] == "uint8" else 4) / 1e9,
                         N * T * np.prod(cfg["ob_shape"]) * (1 if cfg["ob_dtype"] == "uint8" else 4) / cfg["nminibatches"] / 1e9),
                  "train_chunk": res["chunk"],
                  "shuffle": args.shuffle + (" (keyed Feistel bijection evaluated on the device, ops.shuffle_indices)"
                                             if args.shuffle == "device" else " (np.random.shuffle, indices uploaded)")}
        dtype = "f16 operands / f32 accumulate (GAE f64 carry)"
    else:
        tf_step = None
        config = {"workload": cfg["name"], "batch": cfg["batch"], "buffer_transitions": cfg["buffer_size"],
                  "parallelism": f"replicas x{world} (the reference's deepq is single-env; no sharding)",
                  "l2": "replay storage 56 GB: the 512 x 2 gathered observations come from DRAM"}
        dtype = "f16 operands / f32 accumulate (PER trees f64)"
    out = {"metric": metric, "value": res["value"], "unit": unit, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": res["ms_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config,
           "tflops_per_step": tf_step / 1e12 if tf_step else None,
           "mfu_vs_sustained_bf16": (tf_step / (res["ms_step"] / 1e3) / 1e12 / peaks["bf16_tflops_sustained"]) if tf_step else None,
           "gpu_launches": int(round(res["launches"] * args.steps)), "gpu_launches_per_step": res["launches"],
           "timing": "value: un-instrumented timed region; kernels / roofline: a second pass with per-call CUDA events"
                     + (f" ({res['ms_prof']:.1f} ms per step with the events)" if res.get("ms_prof") else ""),
           "per_rank_kernel_ms": res.get("per_rank_kernel_ms"),
           "clocks": res["clocks"], "e2e": res["e2e"], "roofline": roofline, "roofline_all": roofline_all,
           "cpu_baseline": cpu_baseline, "other_configs": others, "targets": targets, "kernels": kernels}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _kernels_of(res):
    if not res.get("prof"):
        return None
    prof, steps = res["prof"]
    kernels = summarize_profile(prof, steps)
    tot = sum(k["ms_per_step"] for k in kernels.values())
    for k in kernels.values():
        k["share"] = k["ms_per_step"] / tot if tot else 0.0
    return kernels


if __name__ == "__main__":
    main()
