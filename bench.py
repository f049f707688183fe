#!/usr/bin/env python
"""bench.py - QMIX learner episodes/sec (+ MAC agent-steps/sec) on SMAC-shaped synthetic episodes: BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 27m_vs_30m] [--impl reference] [--dump-outputs DIR]

One "step" is one QLearner.train call over one batch (both agent unrolls, double-Q targets, both mixers, masked TD loss,
backward, clip, RMSprop, target-sync bookkeeping).  Default workload = BASELINE config 4: QMIX on 27m_vs_30m shapes,
GLOBAL batch 4096, T = 180.  At N GPUs the 4096 episodes are sharded (strong scaling, `"scaling": "strong"`), every rank
trains on its 4096/N episodes and ONE NCCL all-reduce per step carries the gradients and the loss sums; the weak-scaling
figure (4096 episodes per GPU) rides along as `weak`.  Rank 0 prints ONE JSON line:

value         whole-job episodes/s, batch resident in HBM when the timed region starts (CUDA events, max over ranks)
e2e           the same metric through the public API with the batch in pinned HOST memory: the H2D copy of every field
              the step reads and a D2H read of the loss are inside the timed region
roofline      dominant kernel of the step: algorithmic bytes (or FLOPs) / its CUDA-event time averaged over the TIMED
              steps (events recorded between the launches, same stream, same clocks as `value`), vs MEASURED_PEAKS.json
step_roofline SURVEY.md section 8d whole-step bound / measured step
cpu_baseline  the reference's own QLearner.train(use_cuda=False) (staged copy under oracle/_ref, kind "reference"; the
              numpy oracle port when that is absent, kind "port") on this box's host cores, bounded sample
select_actions  BASELINE config 5 (BasicMAC.select_actions, 16384 envs x 27 agents) as a sub-record with its own
              roofline / cpu_baseline / e2e / clocks
configs       BASELINE configs 1-3 (3m/32, 2s3z/1024, MMM2 VDN + IQL/2048) on the same tier, CUDA-graphed step (N = 1 only)
dp_equal      N > 1: a sharded step over N ranks reproduces the 1-GPU step (loss, grad_norm, parameter update)
--impl reference   times the CPU reference alone (rank 0; the other ranks exit 0)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm must see all host cores (set before numpy / torch load)
    for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

from pymarl_b200.synthetic import BASELINE_CONFIGS, SMAC_SHAPES, default_args  # noqa: E402

METRIC = "qmix_learner_episodes_per_sec"
UNIT = "episodes/s"
RO_METRIC, RO_UNIT = "mac_agent_steps_per_sec", "agent-steps/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
H, E = 64, 32


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["source"] = "fallback"
    return d


# ------------------------------------------------------------------------------------------
# algorithmic work per phase (DESIGN.md section 4): (FLOPs, HBM bytes) of one launch
# ------------------------------------------------------------------------------------------
def phase_work(name, B, T, N, O, S, A, mixer):
    """(FLOPs, HBM bytes) one launch of a phase has to do (DESIGN.md section 4).  bf16-tier phases end in _tc:
    their activations are bf16 tile images (128 B per row of 64 columns)."""
    rows = B * T * N
    M = B * (T - 1)
    BT = B * T
    C = (N + 3) * E
    f4 = 4
    ko = -(-O // 64) * 64                      # obs image width (padded to 64-column chunks)
    ks = -(-(S + 1) // 64) * 64                # state image width
    kc = -(-(N + 3) // 2) * 64                 # raw (hypernet output) image width
    if name == "fc1_fwd_both_tc":              # obs fp32 in; obs image, x of both nets, relu mask out
        return 2.0 * rows * O * 2 * H, rows * (O * f4 + ko * 2 + 2 * 128 + 8)
    if name == "gru_unroll_fwd_online_tc":     # x in; h + 4 gate tiles out
        return 2.0 * rows * H * 6 * H, rows * (128 + 128 + 512)
    if name == "gru_unroll_fwd_target_tc":
        return 2.0 * rows * H * 6 * H, rows * (128 + 128)
    if name == "gru_unroll_fwd_both_tc":       # the two recurrences side by side (small batches: forked onto two streams)
        return 2 * 2.0 * rows * H * 6 * H, rows * (128 + 128 + 512 + 128 + 128)
    if name == "gru_fwd_target_select_tc":     # x + online h in; target h never leaves the SM; avail / actions in
        return 2.0 * rows * H * (6 * H + 2 * A), rows * (128 + 128 + A * f4 + 8 + 8)
    if name == "q_select_tc":                  # h of both nets, avail, actions in; chosen / tmax out
        return 2.0 * rows * H * 2 * A, rows * (2 * 128 + A * f4 + 8 + 8)
    if name == "state_to_images":
        return 0.0, BT * (S * f4 + ks * 2)
    if name == "mixer_fwd_target_tc":
        return 2.0 * BT * ks * C, BT * (ks * 2 + N * f4 + f4)
    if name == "mixer_fwd_online_tc":
        return 2.0 * BT * ks * C, BT * (ks * 2 + kc * 2 + N * f4 + f4)
    if name == "mixer_bwd" and mixer == "qmix":   # mix backward on the raw images + weight-gradient GEMM over both images
        return 2.0 * BT * ks * C, BT * (2 * kc * 2 + kc * 2 + ks * 2 + 2 * N * f4)
    if name == "gru_unroll_bwd_tc":            # 4 gate tiles + h + x in; dpre1 out; all rnn.* gradients in TMEM
        return 2.0 * rows * H * (6 * H + 8 * H), rows * (640 + 128 + 128 + 8)
    if name == "dW_rnn_tc":                    # reduction of the per-tile partials
        return 0.0, -(-(B * N) // 128) * (2 * 192 * 64 + 256) * f4
    if name == "dW_fc1_fc2_tc":
        return 2.0 * rows * H * (ko + H + 2 * H), rows * (128 + 128 + ko * 2 + 16)
    if name.startswith("fc1_fwd"):
        return 2.0 * rows * O * H, rows * (O + H) * f4
    if name == "gru_unroll_fwd_online":
        return 2.0 * rows * H * (6 * H + A), rows * (H + H + 4 * H + A) * f4
    if name == "gru_unroll_fwd_target":
        return 2.0 * rows * H * (6 * H + A), rows * (H + A) * f4
    if name == "target_select":
        return 0.0, M * N * (3 * A * f4 + 8 + 8)
    if name.startswith("mixer_fwd"):
        if mixer != "qmix":
            return 0.0, M * (N + 1) * f4
        return 2.0 * M * S * C, M * (S + 2 * C + N + 1) * f4
    if name == "td_loss":
        return 0.0, M * 5 * f4
    if name == "mixer_bwd":
        if mixer != "qmix":
            return 0.0, M * (N + 1) * f4
        return 2.0 * M * S * C, M * (S + 3 * C + 2 * N) * f4
    if name == "gru_unroll_bwd":
        return 2.0 * rows * H * 6 * H, rows * (4 * H * 2 + 3 * H + H) * f4
    if name == "dW_rnn_gemm_atb":
        return 2.0 * rows * H * 6 * H, rows * (2 * 4 * H + 2 * H) * f4
    if name == "dW_fc1_gemm_atb":
        return 2.0 * rows * H * O, rows * (H + O) * f4
    if name == "agent_scatter_grads":
        return 0.0, rows * (2 * H) * f4
    return 0.0, 0.0


def measured_traffic(name, rows):
    """DRAM bytes per launch of a phase's dominant kernel from the committed ncu capture (profiles/traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum per (b, t, n) row), scaled to this run's rows; None if not captured."""
    p = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p)).get("bytes_per_row", {})
    return d[name] * rows if name in d else None


def step_roofline(B, T, N, O, S, A, mixer, peaks):
    """SURVEY.md section 8d: algorithmic FLOPs and HBM bytes of one whole step."""
    d_in = O + A + N
    f_row = 2 * H * (d_in + 6 * H + A)
    f_agent = T * N * (4 * f_row - 2 * d_in * H)
    f_mix = (T - 1) * (3 * 2 * S * E * (N + 3) + 4 * (2 * E + 2 * N * E + 2 * E)) if mixer == "qmix" else 0
    flops = B * (f_agent + f_mix)
    byts = B * (2 * T * N * O * 4 + (2 * T * S * 4 if mixer == "qmix" else 0) + T * N * A * 4 + T * N * 8 + T * 13
                + 2 * T * N * H * 4)
    t_hbm = byts / (peaks["hbm_gbs"] * 1e9)
    t_tensor = flops / (peaks["bf16_tflops_sustained"] * 1e12)
    return flops, byts, max(t_hbm, t_tensor), ("hbm" if t_hbm >= t_tensor else "tensor")


def kernel_roofline(name, ms, B, T, N, O, S, A, mixer, peaks):
    """Achieved vs peak of ONE phase from its algorithmic work and measured time (ms)."""
    fl, by = phase_work(name, B, T, N, O, S, A, mixer)
    if ms <= 0 or (fl <= 0 and by <= 0):
        return None
    tsec = ms * 1e-3
    t_h = by / (peaks["hbm_gbs"] * 1e9)
    t_t = fl / (peaks["bf16_tflops_sustained"] * 1e12)
    if t_t >= t_h:
        ach, peak, unit, bound = fl / tsec / 1e12, peaks["bf16_tflops_sustained"], "TFLOP/s", "tensor"
    else:
        ach, peak, unit, bound = by / tsec / 1e9, peaks["hbm_gbs"], "GB/s", "hbm"
    return {"kernel": name, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
            "algorithmic_bytes": by, "algorithmic_flops": fl, "kernel_ms": ms}


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during a timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def n_samples(self):
        return len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def _finish_sampling(th, sampler, step_fn, ms_per_step, collective=False, min_samples=3, max_seconds=3.0):
    """Short timed regions end before nvidia-smi delivers its first line: keep the GPU busy with the same step (outside
    the timed region) until a few samples exist, so the clocks record describes this workload under load.
    collective=True: the step contains a collective (data-parallel learner), so EVERY rank must run the same number of
    extra steps - a fixed count derived from the (max-over-ranks, hence identical) step time instead of a rank-local
    "until nvidia-smi answered" loop, which would desynchronise the ranks and dead-lock the next all-reduce."""
    if collective:
        n = int(min(4000, max(1, 450.0 / max(ms_per_step, 1e-3))))
        for i in range(n):
            step_fn(i)
            if i % 8 == 7:
                th.cuda.synchronize()
    else:
        t0, i = time.perf_counter(), 0
        while sampler.n_samples() < min_samples and time.perf_counter() - t0 < max_seconds:
            step_fn(i)
            i += 1
            if i % 8 == 0:
                th.cuda.synchronize()
    th.cuda.synchronize()
    return sampler.stop()


# ------------------------------------------------------------------------------------------
# CPU legs: the reference itself (oracle/_ref) or, when it was not staged, the numpy oracle port
# ------------------------------------------------------------------------------------------
def cpu_learner(cfg, batch, steps, warmup):
    """-> cpu_baseline dict for one QLearner.train step on `batch` full-length episodes of the config's shapes."""
    from oracle import ref_harness
    shape = SMAC_SHAPES[cfg["shape"]]
    args = default_args(shape, mixer=cfg["mixer"])
    if ref_harness.available():
        val, ms, cores = ref_harness.time_learner(shape, args, batch, cfg["T"], steps, warmup)
        kind, what = "reference", "reference QLearner.train, torch %s CPU" % __import__("torch").__version__
    else:
        val, ms = _cpu_port_learner(cfg, batch, steps, warmup)
        kind, what, cores = "port", "numpy oracle port (oracle/_ref not staged)", os.cpu_count()
    return {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_step": ms,
            "sample": "%d episodes x T=%d per step, %d steps after %d warm-up (%s)" % (batch, cfg["T"], steps, warmup, what)}


def _cpu_port_learner(cfg, batch, steps, warmup):
    import copy
    import numpy as np
    from oracle import qlearner_oracle as orc
    from pymarl_b200.synthetic import numpy_episode_fields
    shape = SMAC_SHAPES[cfg["shape"]]
    args = default_args(shape, mixer=cfg["mixer"])
    rng = np.random.default_rng(7)
    d_in = shape.obs_dim + shape.n_actions + shape.n_agents
    agent = orc.init_params(orc.agent_param_shapes(d_in, 64, shape.n_actions), rng)
    mixer = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, 32), rng) if cfg["mixer"] == "qmix" else {}
    olr = orc.OracleQLearner(agent, mixer, copy.copy(args))
    fields = numpy_episode_fields(shape, batch, cfg["T"], seed=0, ragged=False)
    for _ in range(warmup):
        olr.train(fields, 0, 0)
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        olr.train(fields, i, 0)
        times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    return batch / mean, mean * 1e3


def cpu_rollout(envs, steps, warmup):
    """-> cpu_baseline dict for one BasicMAC.select_actions step over `envs` envs x 27 agents."""
    from oracle import ref_harness
    shape = SMAC_SHAPES["27m_vs_30m"]
    if ref_harness.available():
        val, ms, cores = ref_harness.time_select_actions(shape, default_args(shape, mixer="qmix"), envs, steps, warmup)
        kind, what = "reference", "reference BasicMAC.select_actions, torch CPU"
    else:
        import numpy as np
        from oracle import qlearner_oracle as orc
        from pymarl_b200.synthetic import numpy_episode_fields
        N, O, A = shape.n_agents, shape.obs_dim, shape.n_actions
        rng = np.random.default_rng(7)
        agent = orc.init_params(orc.agent_param_shapes(O + A + N, H, A), rng)
        fields = numpy_episode_fields(shape, envs, 4, seed=0, ragged=False)
        hstate = np.zeros((envs * N, H), np.float32)
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            u = rng.random((envs, N), dtype=np.float32)
            e = rng.exponential(size=(envs, N, A)).astype(np.float32)
            _, _, hstate = orc.mac_select_actions(agent, fields, 1 + i % 3, hstate, 0.5, u, e)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        ms = 1e3 * sum(times) / len(times)
        val, kind, what, cores = envs * N / (ms * 1e-3), "port", "numpy oracle port (oracle/_ref not staged)", os.cpu_count()
    return {"value": val, "unit": RO_UNIT, "cores": cores, "kind": kind, "ms_per_step": ms,
            "sample": "%d envs x %d agents per step, %d steps after %d warm-up (%s)" % (envs, shape.n_agents, steps, warmup, what)}


def reference_arm(a, cfg):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    shape = SMAC_SHAPES[cfg["shape"]]
    batch = a.cpu_batch or (32 if shape.n_agents > 5 else min(cfg["batch"], 64))
    cb = cpu_learner(cfg, batch, a.steps, a.warmup)
    ro = cpu_rollout(a.cpu_envs, a.steps, a.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload_name(cfg), "name": a.config, "shape": cfg["shape"], "T": cfg["T"], "mixer": cfg["mixer"],
                   "batch": batch, "note": "CPU reference on the host cores; each step a bounded sample of the workload"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "select_actions": {"metric": RO_METRIC, "value": ro["value"], "unit": RO_UNIT, "steps": a.steps, "warmup": a.warmup,
                           "ms_per_step": ro["ms_per_step"], "cpu_baseline": ro},
    }
    print(json.dumps(line), flush=True)


def _workload_name(cfg):
    return ("QMIX learner step, %s shapes" % cfg["shape"]) if cfg["mixer"] == "qmix" else \
        "%s learner step, %s shapes" % ((cfg["mixer"] or "iql").upper(), cfg["shape"])


# ------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide state of the GPU arm."""

    def __init__(self):
        import torch as th
        import torch.distributed as dist
        self.th, self.dist = th, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        th.cuda.set_device(self.local_rank)
        self.dev = th.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.th.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.th.tensor([v], dtype=self.th.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


class _DictBatch:
    """Minimal EpisodeBatch stand-in (QLearner.train / BasicMAC only read batch[key], batch_size, max_seq_length)."""

    def __init__(self, fields, batch_size, max_seq_length):
        self.fields, self.batch_size, self.max_seq_length = fields, batch_size, max_seq_length
        self.device = next(iter(fields.values())).device

    def __getitem__(self, k):
        return self.fields[k]


def build_learner(ctx, cfg, precision, **over):
    th = ctx.th
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from cuda_utils import Logger
    from pymarl_b200 import le_REGISTRY, mac_REGISTRY
    from pymarl_b200.synthetic import make_scheme
    shape = SMAC_SHAPES[cfg["shape"]]
    args = default_args(shape, mixer=cfg["mixer"], device="cuda", use_cuda=True, learner_log_interval=10 ** 12,
                        precision=precision, **over)
    th.manual_seed(7)                                   # identical parameters on every rank
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    learner = le_REGISTRY["q_learner"](mac, scheme, Logger(), args)
    learner.cuda()
    return learner


def learner_outputs(learner):
    """What QLearner.train hands its caller after a step: the updated online parameters and the step's statistics."""
    import numpy as np
    out = {}
    for tag, mod in (("agent", learner.mac.agent), ("mixer", learner.mixer)):
        if mod is not None:
            for k, v in mod.state_dict().items():
                out[tag + "." + k] = v.detach().float().cpu().numpy()
    st = learner.stats()
    for k in ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean"):
        out[k] = np.array([st[k]], dtype=np.float64)
    return out


def rollout_outputs(actions, hidden, n_envs, max_envs=4096):
    """What BasicMAC.select_actions hands its caller after a step: the chosen actions and the hidden state carried into the
    next step, for a fixed, seeded sample of at most `max_envs` envs (the hidden state of 16384 envs is 113 MB).  With
    the default epsilon schedule most actions are random draws; the hidden state carries the network's arithmetic."""
    import numpy as np
    import torch as th
    envs = np.arange(n_envs) if n_envs <= max_envs else np.sort(np.random.default_rng(0).choice(n_envs, max_envs, replace=False))
    idx = th.from_numpy(envs).to(actions.device)
    return {"actions": actions[idx].float().cpu().numpy(),
            "hidden_states": hidden.reshape(n_envs, -1, hidden.shape[-1])[idx].float().cpu().numpy()}


def write_outputs(outputs, out_dir):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def time_learner(ctx, learner, batch, steps, warmup, profile, after_timed=None):
    """W untimed + K timed steps (barrier + synchronize on both sides, CUDA events on the launch stream, max over ranks).
    profile=True arms the library's per-phase events for the TIMED steps themselves, so the per-kernel times see the
    clocks `ms_per_step` sees.  after_timed() runs right after the last timed step, before the untimed steps that keep
    the GPU busy for the clock sampler.  -> (ms per step, phases_ms averaged per step, launches per step, clocks)."""
    th = ctx.th
    from pymarl_b200 import _lib
    l0 = _lib.lib().pmb_launch_count()
    learner.train(batch, 0, 0)
    launches = _lib.lib().pmb_launch_count() - l0      # counted on an eager step (a graph replay launches the same kernels)
    for i in range(1, warmup):
        learner.train(batch, i, 0)
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank).start()
    ev0, ev1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    ctx.barrier()
    if profile:
        _lib.profile_begin()
    ev0.record()
    for i in range(steps):
        learner.train(batch, warmup + i, 0)
    ev1.record()
    ctx.barrier()
    phases = _lib.profile_end(max_phases=1024) if profile else []
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1) / steps)
    if after_timed is not None:
        after_timed()
    clocks = _finish_sampling(th, sampler, lambda i: learner.train(batch, i, 0), ms, collective=ctx.world > 1)
    phase_ms = {}
    for name, pms in phases:
        phase_ms[name] = phase_ms.get(name, 0.0) + pms / steps
    if "end" in phase_ms:                               # from a step's last launch to the next step's first phase mark
        phase_ms["inter_step"] = phase_ms.pop("end")
    return ms, phase_ms, int(launches), clocks


def profile_pass(learner, batch, steps):
    """Per-kernel times of `steps` eager steps (used where the timed region replays a CUDA graph)."""
    from pymarl_b200 import _lib
    saved = getattr(learner.args, "cuda_graph", False)
    learner.args.cuda_graph = False
    learner.train(batch, 0, 0)
    _lib.profile_begin()
    for i in range(steps):
        learner.train(batch, i, 0)
    phases = _lib.profile_end(max_phases=1024)
    learner.args.cuda_graph = saved
    out = {}
    for name, pms in phases:
        out[name] = out.get(name, 0.0) + pms / steps
    if "end" in out:
        out["inter_step"] = out.pop("end")
    return out


def learner_record(ctx, cfg, B_local, ms, phase_ms, launches, clocks, precision):
    """The JSON pieces every learner measurement shares."""
    shape = SMAC_SHAPES[cfg["shape"]]
    N, O, S, A, T = shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, cfg["T"]
    kern = {k: v for k, v in phase_ms.items() if k != "inter_step"}
    top = max(kern, key=kern.get) if kern else None
    roofline = None
    if top:
        roofline = kernel_roofline(top, kern[top], B_local, T, N, O, S, A, cfg["mixer"], ctx.peaks)
        if roofline:
            roofline.update(traffic=measured_traffic(top, B_local * T * N), peak_source=ctx.peaks["source"],
                            share_of_step=kern[top] / max(sum(phase_ms.values()), 1e-9),
                            timed="CUDA events between the launches of the timed steps (same clocks as ms_per_step)")
    fracs = {}
    for k, v in kern.items():
        r = kernel_roofline(k, v, B_local, T, N, O, S, A, cfg["mixer"], ctx.peaks)
        if r:
            fracs[k] = {"ms": round(v, 4), "bound": r["bound"], "frac": round(r["frac"], 3)}
    fl_s, by_s, t_roof, bound_s = step_roofline(B_local, T, N, O, S, A, cfg["mixer"], ctx.peaks)
    return {"ms_per_step": ms, "roofline": roofline,
            "step_roofline": {"flops": fl_s, "bytes": by_s, "t_roof_ms": t_roof * 1e3, "bound": bound_s,
                              "frac": t_roof * 1e3 / ms},
            "phases_ms": phase_ms, "kernels": fracs, "clocks": clocks, "gpu_launches": launches,
            "dtype": "f32" if precision == "fp32" else "bf16 (fp32 accumulate)"}


def e2e_learner(ctx, learner, fields, B_local, T, mixer, steps):
    """Host-resident batch through the public API: H2D of every field the step reads + D2H read of the loss, timed
    by wall clock around synchronised steps (max over ranks)."""
    th = ctx.th
    # Every rank must take the same path (the steps below contain a collective): pin first, then agree.
    host, err = None, None
    try:
        import psutil
        input_bytes = sum(v.numel() * v.element_size() for v in fields.values())
        need = ctx.world * input_bytes
        avail = psutil.virtual_memory().available
        if avail < 1.25 * need:
            raise MemoryError("host has %.0f GB available, the pinned batches of %d ranks need %.0f GB"
                              % (avail / 1e9, ctx.world, need / 1e9))
        host = {k: th.empty(v.shape, dtype=v.dtype, pin_memory=True).copy_(v) for k, v in fields.items()}
    except Exception as ex:                              # e.g. the pod cannot pin 30 GB
        err = repr(ex)[:200]
    if ctx.max_over_ranks(0.0 if err is None else 1.0) > 0:
        return {"value": None, "unit": UNIT, "error": err or "another rank could not pin its batch"}
    try:
        hb = _DictBatch(host, B_local, T)
        learner.train(hb, 0, 0)                          # warm-up (allocates the device copies)
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            learner.train(hb, i, 0)
            loss = learner.last_stats[6].item()          # D2H read of the step's loss
        ctx.barrier()
        dt = ctx.max_over_ranks((time.perf_counter() - t0) / steps)
        h2d = sum(v.numel() * v.element_size() for k, v in host.items()
                  if k in ("obs", "state", "actions", "avail_actions", "reward", "terminated", "filled")
                  and (k != "state" or mixer == "qmix"))
        return {"value": ctx.world * B_local / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                "ms_per_step": dt * 1e3, "steps": steps, "loss": loss,
                "note": "per rank: pinned host batch of %d episodes -> H2D -> train -> loss.item()%s" % (
                    B_local, " (QLearner.train streams the host batch in %d-episode chunks: copy of chunk i+1 under the "
                    "compute of chunk i, one update)" % learner._hs["bufs"][0]["obs"].shape[0]
                    if getattr(learner, "_hs", None) else "")}
    except Exception as ex:
        if ctx.world > 1:
            raise                                        # a rank-local failure inside collective steps cannot be skipped safely
        return {"value": None, "unit": UNIT, "error": repr(ex)[:200]}


# ------------------------------------------------------------------------------------------
def dp_self_check(ctx):
    """N > 1: a step on a batch sharded over the N ranks (train() slices, ONE all-reduce, replicated update) against the
    same step computed by ONE GPU on the whole batch: loss, grad_norm and the parameter update, both tiers.
    Tolerances: loss, grad_norm and every post-update parameter tensor (max|a-b| / max|a|) 1e-6 on the fp32 tier, 1e-3 on the
    bf16 tier; the update p' - p as a flat vector in the relative L2 norm 1e-4 / 1e-2; and the replicated parameters must be
    bit-identical across the ranks.  Every rank computes both sides; rank 0 reports."""
    th = ctx.th
    from pymarl_b200.synthetic import torch_episode_fields
    cfg = dict(shape="27m_vs_30m", T=24, batch=40, mixer="qmix")
    shape = SMAC_SHAPES[cfg["shape"]]
    out = {"ok": True, "world": ctx.world, "batch": cfg["batch"], "T": cfg["T"]}
    fields = torch_episode_fields(shape, cfg["batch"], cfg["T"], seed=4242, ragged=True, device=ctx.dev, with_onehot=False)
    batch = _DictBatch(fields, cfg["batch"], cfg["T"])
    for prec, tol_s, tol_p, exch in (("fp32", 1e-6, 1e-4, "peer"), ("bf16", 1e-3, 1e-2, "peer"), ("bf16", 1e-3, 1e-2, "nccl")):
        res = []
        for dp in (False, True):
            lr = build_learner(ctx, cfg, prec, data_parallel=dp, dp_exchange=exch)
            lr._flat["sq"].fill_(1e-2)
            p0 = lr._flat["p"].clone()
            lr.train(batch, 0, 0)
            st = lr.stats()
            res.append((st["loss"], st["grad_norm"], (lr._flat["p"] - p0).double(), lr._flat["layout"], lr._flat["p"].double().clone()))
        (l1, g1, u1, lay, p1), (l2, g2, u2, _, p2) = res
        e_loss, e_gn = abs(l1 - l2) / max(abs(l1), 1e-30), abs(g1 - g2) / max(abs(g1), 1e-30)
        # post-update parameters per tensor (max|a-b| / max|a|), and the UPDATE as one flat vector in the relative L2 norm
        # (per-tensor relative errors of the update are dominated by tensors whose gradient is a cancelling sum, e.g. the
        # single element of V.2.bias: fp32 summation order alone moves those by 1e-4 of their own size)
        e_par, worst = 0.0, None
        for i in range(len(lay.numel)):
            o, n = lay.offset[i], lay.numel[i]
            if n:
                e = float((p1[o:o + n] - p2[o:o + n]).abs().max() / p1[o:o + n].abs().max().clamp_min(1e-30))
                if e > e_par:
                    e_par, worst = e, i
        nt = lay.n_total
        e_upd = float((u1[:nt] - u2[:nt]).norm() / u1[:nt].norm().clamp_min(1e-30))
        ok = e_loss <= tol_s and e_gn <= tol_s and e_par <= tol_s and e_upd <= tol_p
        # the replicated parameters must be BIT-identical on every rank after the update
        ref = lr._flat["p"].clone()
        ctx.dist.broadcast(ref, src=0)
        same = bool(th.equal(ref, lr._flat["p"]))
        flag = th.tensor([int(ok and same)], device=ctx.dev)
        ctx.dist.all_reduce(flag, op=ctx.dist.ReduceOp.MIN)
        fused = lr._px is not None
        if fused:
            same = same and lr._px.error_word() == 0
            flag2 = th.tensor([int(same)], device=ctx.dev)
            ctx.dist.all_reduce(flag2, op=ctx.dist.ReduceOp.MIN)
            out["ok"] = out["ok"] and bool(flag2.item())
        out[prec + "_" + exch] = {"loss_rel": e_loss, "grad_norm_rel": e_gn, "params_rel": e_par, "worst_tensor": worst,
                                  "update_rel_l2": e_upd, "replicas_bit_identical": same, "tol": [tol_s, tol_p],
                                  "exchange": "fused peer-memory kernel" if fused else "nccl all-reduce"}
        out["ok"] = out["ok"] and bool(flag.item())
        del lr
    return out


# ------------------------------------------------------------------------------------------
def rollout_record(ctx, a, envs, precision, steps, warmup, e2e_steps, with_cpu, outputs=None):
    """BASELINE config 5: one BasicMAC.select_actions step (fc1 -> GRUCell -> fc2 -> avail mask -> epsilon-greedy) over
    `envs` synthetic envs x 27 agents per GPU; agent-steps/s.  The obs of 4 timesteps live in HBM and the step index
    cycles over them (2 GB, larger than L2).  A dict passed as `outputs` receives rollout_outputs() of the last timed step."""
    th = ctx.th
    from pymarl_b200 import mac_REGISTRY, _lib
    from pymarl_b200.synthetic import make_scheme, torch_episode_fields
    shape = SMAC_SHAPES["27m_vs_30m"]
    N, O, A = shape.n_agents, shape.obs_dim, shape.n_actions
    # action_rng="philox": the epsilon-greedy draws come from the kernel's own Philox stream (one fused call per step);
    # "torch" replays the reference's generator order for bit-identical actions (two torch RNG launches + 190 MB extra)
    args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, precision=precision, action_rng=a.action_rng)
    th.manual_seed(7)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (A,), "dtype": th.float32, "group": "agents"}
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    Tb = 4
    fields = torch_episode_fields(shape, envs, Tb, seed=1000 + ctx.rank, ragged=False, device=ctx.dev, with_onehot=False)
    batch = _DictBatch(fields, envs, Tb)
    mac.init_hidden(envs)
    for i in range(warmup):
        mac.select_actions(batch, 1 + i % 3, 1000 * i)
    ctx.barrier()
    sampler = ClockSampler(ctx.local_rank).start()
    launches0 = _lib.lib().pmb_launch_count()
    ev0, ev1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    ctx.barrier()
    ev0.record()
    for i in range(steps):
        acts = mac.select_actions(batch, 1 + i % 3, 1000 * i)
    ev1.record()
    ctx.barrier()
    launches = (_lib.lib().pmb_launch_count() - launches0) // max(1, steps)
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1) / steps)
    if outputs is not None:
        outputs.update(rollout_outputs(acts, mac.hidden_states, envs))
    clocks = _finish_sampling(th, sampler, lambda i: mac.select_actions(batch, 1 + i % 3, 0), ms)     # no collective in this step
    value = ctx.world * envs * N / (ms * 1e-3)
    rows = envs * N
    algo_bytes = rows * (O * 4 + 2 * H * 4 + A * 4 + 8 + 8)          # SURVEY.md section 8d
    ach = algo_bytes / (ms * 1e-3) / 1e9
    # e2e: obs / avail of the step start in pinned host memory, the chosen actions are read back (what a runner does)
    e2e = None
    if e2e_steps > 0:
        host = {k: th.empty(v.shape, dtype=v.dtype, pin_memory=True).copy_(v) for k, v in fields.items()}
        hb = _DictBatch(host, envs, Tb)
        out = th.empty(envs, N, dtype=th.int64, pin_memory=True)
        mac.select_actions(hb, 1, 0)
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            acts = mac.select_actions(hb, 1 + i % 3, 1000 * i)
            out.copy_(acts, non_blocking=True)
            th.cuda.synchronize()
        dt = ctx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
        # obs / avail_actions: the step itself; actions / filled: the step and the one before (last-action input)
        h2d = sum(host[k][:, :1].numel() * host[k].element_size() for k in ("obs", "avail_actions")) + \
            sum(host[k][:, :2].numel() * host[k].element_size() for k in ("actions", "filled"))
        e2e = {"value": ctx.world * envs * N / dt, "unit": RO_UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": envs * N * 8, "ms_per_step": dt * 1e3, "steps": e2e_steps}
    cpu = cpu_rollout(a.cpu_envs, 10, 2) if with_cpu else None
    return {"metric": RO_METRIC, "value": value, "unit": RO_UNIT, "n_gpus": ctx.world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "dtype": "f32" if precision == "fp32" else "bf16 (fp32 accumulate)", "data": "synthetic",
            "config": {"workload": "BasicMAC.select_actions step, 27m_vs_30m shapes", "envs_per_gpu": envs, "n_agents": N,
                       "obs": O, "n_actions": A, "parallelism": "dp%d (envs sharded, no collective)" % ctx.world,
                       "action_rng": a.action_rng,
                       "l2_policy": "obs of 4 timesteps (%.1f GB) cycled, larger than L2" % (fields["obs"].numel() * 4 / 1e9)},
            "roofline": {"kernel": "select_actions_step (all launches of a step)", "bound": "hbm", "achieved": ach,
                         "peak": ctx.peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / ctx.peaks["hbm_gbs"], "traffic": None,
                         "algorithmic_bytes": algo_bytes, "peak_source": ctx.peaks["source"]},
            "cpu_baseline": cpu, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches)}


def rollout_loop_record(ctx, precision, n_envs=4096, episode_limit=60, runs=3):
    """SURVEY.md section 8f-3: whole rollouts through pymarl_b200.runners.VectorRunner - `n_envs` SMAC-shaped synthetic envs
    (27m_vs_30m shapes) stepped on the device until every episode ended (time limit `episode_limit`), each timestep =
    fused select_actions + three pmb_batch_update launches (actions + one-hot, reward / terminated, next state / avail /
    obs + filled) + the env's own device ops.  agent-steps/s over env steps actually taken, wall clock around
    synchronised runs (the loop syncs once per timestep for the live-env count)."""
    th = ctx.th
    from pymarl_b200 import mac_REGISTRY
    from pymarl_b200.runners import VectorRunner, SyntheticVectorEnv
    from pymarl_b200.synthetic import make_scheme
    shape = SMAC_SHAPES["27m_vs_30m"]
    args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, precision=precision, action_rng="philox",
                        batch_size_run=n_envs)
    th.manual_seed(7)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    mac = mac_REGISTRY["basic_mac"](scheme, groups, args)
    mac.cuda()
    env = SyntheticVectorEnv(n_envs, shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions,
                             episode_limit=episode_limit, seed=11 + ctx.rank, p_end=0.01, device=ctx.dev)
    runner = VectorRunner(args, env)
    runner.setup(mac)
    runner.run()                                          # warm-up
    th.cuda.synchronize()
    t_env0, t0 = runner.t_env, time.perf_counter()
    for _ in range(runs):
        runner.run()
    th.cuda.synchronize()
    dt = time.perf_counter() - t0
    steps = runner.t_env - t_env0
    return {"metric": "rollout_loop_agent_steps_per_sec", "value": steps * shape.n_agents / dt, "unit": RO_UNIT,
            "env_steps": steps, "seconds": dt, "runs": runs,
            "config": {"workload": "VectorRunner.run: select_actions + EpisodeBatch.update per timestep, synthetic device envs",
                       "envs": n_envs, "n_agents": shape.n_agents, "episode_limit": episode_limit}}


COMA_KW = dict(agent_output_type="pi_logits", action_selector="multinomial", learner="coma_learner", critic_lr=5e-4,
               td_lambda=0.8, mask_before_softmax=True, epsilon_start=0.5, epsilon_finish=0.01, epsilon_anneal_time=100000,
               test_greedy=True)


def coma_record(ctx, shape_name="2s3z", B=8, T=120, steps=20, warmup=3):
    """SURVEY.md section 8f rank 4: one COMALearner.train step (target critic, td-lambda targets, T-1 critic optimiser steps,
    agent unroll, policy gradient, two RMSprop updates) on SMAC-shaped synthetic episodes at the reference's on-policy batch
    size (coma_smac.yaml: 8 episodes), replayed as one CUDA graph; the reference's COMALearner on the host cores beside it.
    fp32 (CUDA-core) tier; the step is a chain of ~14 small launches per timestep, i.e. latency- not bandwidth-bound."""
    th = ctx.th
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import copy
    from cuda_utils import Logger
    from pymarl_b200 import le_REGISTRY, mac_REGISTRY, _lib
    from pymarl_b200.synthetic import make_scheme, torch_episode_fields
    shape = SMAC_SHAPES[shape_name]
    args = default_args(shape, mixer=None, device="cuda", use_cuda=True, learner_log_interval=10 ** 12, cuda_graph=True, **COMA_KW)
    th.manual_seed(7)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    mac = mac_REGISTRY["basic_mac"](copy.deepcopy(scheme), groups, args)
    learner = le_REGISTRY["coma_learner"](mac, scheme, Logger(), args)
    learner.cuda()
    fields = torch_episode_fields(shape, B, T, seed=3000, ragged=False, device=ctx.dev, with_onehot=False)
    batch = _DictBatch(fields, B, T)
    l0 = _lib.lib().pmb_launch_count()
    learner.train(batch, 0, 0)
    launches = _lib.lib().pmb_launch_count() - l0
    for i in range(1, warmup):
        learner.train(batch, i, 0)
    th.cuda.synchronize()
    ev0, ev1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        learner.train(batch, warmup + i, 0)
    ev1.record()
    th.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    rec = {"metric": "coma_learner_episodes_per_sec", "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
           "gpu_launches": int(launches), "cuda_graph": any(isinstance(v, tuple) for v in learner._graphs.values()),
           "dtype": "f32", "workload": "COMA learner step, %s shapes" % shape_name, "batch": B, "T": T,
           "note": "includes the one D2H read of the per-step statistics every step (the reference syncs per timestep)"}
    try:
        from oracle import ref_harness
        if ref_harness.available():
            cargs = default_args(shape, mixer=None, **COMA_KW)
            val, cms, cores = ref_harness.time_coma_learner(shape, cargs, B, T, 3, 1)
            rec["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "reference", "ms_per_step": cms,
                                   "sample": "%d episodes x T=%d per step, 3 steps after 1 warm-up (reference COMALearner.train, torch CPU)" % (B, T)}
    except Exception as ex:
        rec["cpu_baseline"] = {"value": None, "error": repr(ex)[:200]}
    return rec


def small_config_record(ctx, name, precision, steps, warmup):
    """BASELINE configs 1-3 on one GPU: the whole step replayed as ONE CUDA graph (args.cuda_graph); per-kernel times
    from a separate eager pass; the reference on the host cores next to it."""
    from pymarl_b200.synthetic import torch_episode_fields
    th = ctx.th
    cfg = dict(BASELINE_CONFIGS[name])
    shape = SMAC_SHAPES[cfg["shape"]]
    B, T = cfg["batch"], cfg["T"]
    learner = build_learner(ctx, cfg, precision, cuda_graph=True)
    fields = torch_episode_fields(shape, B, T, seed=2000, ragged=False, device=ctx.dev, with_onehot=False)
    batch = _DictBatch(fields, B, T)
    ms, _, launches, clocks = time_learner(ctx, learner, batch, steps, max(warmup, 3), profile=False)
    graphed = any(isinstance(v, tuple) for v in learner._graphs.values())
    # the same step launched eagerly: at a few ms per step the graph no longer pays (and the forked recurrences of a
    # graph are not ordered the way the eager launches are); the faster of the two is reported
    learner.args.cuda_graph = False
    ms_eager, _, _, clocks_eager = time_learner(ctx, learner, batch, steps, 3, profile=False)
    ms_graph = ms
    if ms_eager < ms:
        ms, clocks, graphed = ms_eager, clocks_eager, False
    phase_ms = profile_pass(learner, batch, 5)
    rec = learner_record(ctx, cfg, B, ms, phase_ms, launches, clocks, precision)
    rec.update(value=B / (ms * 1e-3), unit=UNIT, cuda_graph=graphed, workload=_workload_name(cfg), batch=B, T=T,
               graph_ms_per_step=ms_graph, eager_ms_per_step=ms_eager,
               l2_policy="inputs %.2f GB" % (sum(v.numel() * v.element_size() for v in fields.values()) / 1e9))
    cb = 32 if shape.n_agents > 5 else min(B, 64)
    rec["cpu_baseline"] = cpu_learner(cfg, cb, 3, 1)
    del learner, fields, batch
    th.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="27m_vs_30m", choices=sorted(BASELINE_CONFIGS) + ["select_actions"],
                    help="select_actions = BASELINE config 5 alone: BasicMAC.select_actions over 16384 envs x 27 agents")
    ap.add_argument("--batch", type=int, default=0, help="GLOBAL batch in episodes (default: the BASELINE batch); "
                    "select_actions: envs per GPU")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the global batch is sharded over the GPUs (BASELINE config 4); weak: that batch PER GPU")
    ap.add_argument("--ragged", action="store_true", help="variable-length episodes instead of full-length")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the select_actions / configs 1-3 / weak / dp_equal sub-records")
    ap.add_argument("--cpu-batch", type=int, default=0)
    ap.add_argument("--cpu-envs", type=int, default=256)
    ap.add_argument("--hang-timeout", type=int, default=600,
                    help="multi-rank runs only: seconds after which a stuck job dumps its stacks and exits")
    ap.add_argument("--cuda-graph", action="store_true", help="replay the main config's step as a CUDA graph too")
    ap.add_argument("--dp-exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: fused exchange + update kernel over NVLink peer memory (falls back to nccl when unavailable) or NCCL")
    ap.add_argument("--action-rng", default="philox", choices=["philox", "torch"],
                    help="select_actions: where the epsilon-greedy draws come from")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="bf16 = tcgen05 tensor-core tier (fp32 accumulate, parity 1e-2); fp32 = CUDA-core tier (parity 1e-5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy, to compare two builds: the updated "
                    "agent / mixer parameters (float32) and the loss statistics (float64) of a learner step; the chosen "
                    "actions and the carried hidden state (float32) of a select_actions step")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs compares builds of this project; the reference arm has nothing to dump")
    if a.config == "select_actions":
        if a.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                ro = cpu_rollout(a.cpu_envs, a.steps, a.warmup)
                print(json.dumps({"impl": "reference", "metric": RO_METRIC, "value": ro["value"], "unit": RO_UNIT,
                                  "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ro["ms_per_step"],
                                  "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                                  "data": "synthetic", "config": {"workload": "BasicMAC.select_actions step, 27m_vs_30m shapes",
                                                                   "envs": a.cpu_envs},
                                  "cpu_baseline": ro, "e2e": {"value": ro["value"], "unit": RO_UNIT, "h2d_bytes_per_step": 0,
                                                              "d2h_bytes_per_step": 0}}), flush=True)
            return
        ctx = Ctx()
        outputs = {} if a.dump_outputs else None
        rec = rollout_record(ctx, a, a.batch or 16384, a.precision, a.steps, a.warmup, 0 if a.no_e2e else a.e2e_steps,
                             with_cpu=(ctx.rank == 0 and ctx.world == 1 and not a.no_cpu_baseline), outputs=outputs)
        rec["vs_baseline"] = None
        if ctx.rank == 0:
            if outputs is not None:
                write_outputs(outputs, a.dump_outputs)
            print(json.dumps(rec), flush=True)
        if ctx.world > 1:
            ctx.dist.destroy_process_group()
        return

    cfg = dict(BASELINE_CONFIGS[a.config])
    if a.batch:
        cfg["batch"] = a.batch
    if a.impl == "reference":
        return reference_arm(a, cfg)

    # a multi-rank job that stops making progress (a rank died, a collective mismatched) must not sit in NCCL's 10-minute
    # watchdog: dump the stacks and exit after a generous bound
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import faulthandler
        faulthandler.dump_traceback_later(a.hang_timeout, exit=True)
    ctx = Ctx()
    th = ctx.th
    from pymarl_b200.data_parallel import shard_slice
    from pymarl_b200.synthetic import torch_episode_fields
    shape = SMAC_SHAPES[cfg["shape"]]
    Bg, T = cfg["batch"], cfg["T"]
    N, O, S, A = shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions
    strong = a.scaling == "strong"
    lo, hi = shard_slice(Bg, ctx.rank, ctx.world) if strong else (0, Bg)
    B_local = hi - lo
    extras = not a.no_extras

    dp_equal = dp_self_check(ctx) if (ctx.world > 1 and extras) else None

    # rank-local episodes (dp_shard_batch=False: train() must not slice again); in a weak-scaling side run every rank
    # needs the full batch, so generate that once and let the strong run use its first B_local episodes
    want_weak = strong and ctx.world > 1 and extras
    B_gen = Bg if want_weak else B_local
    learner = build_learner(ctx, cfg, a.precision, dp_shard_batch=False, cuda_graph=a.cuda_graph, dp_exchange=a.dp_exchange)
    fields_all = torch_episode_fields(shape, B_gen, T, seed=1000 + ctx.rank, ragged=a.ragged, device=ctx.dev, with_onehot=False)
    weak = None
    if want_weak:
        wb = _DictBatch(fields_all, B_gen, T)
        wms, _, _, _ = time_learner(ctx, learner, wb, a.steps, a.warmup, profile=False)
        weak = {"value": ctx.world * B_gen / (wms * 1e-3), "unit": UNIT, "ms_per_step": wms, "steps": a.steps, "batch_per_gpu": B_gen,
                "global_batch": ctx.world * B_gen, "scaling": "weak"}
        del wb
    fields = {k: v[:B_local] for k, v in fields_all.items()} if B_gen != B_local else fields_all
    if B_gen != B_local:
        fields = {k: v.contiguous() for k, v in fields.items()}
        del fields_all
        learner._workspace = None
        th.cuda.empty_cache()
    batch = _DictBatch(fields, B_local, T)
    input_bytes = sum(v.numel() * v.element_size() for v in fields.values())

    exchange_desc = "single GPU" if ctx.world == 1 else (
        "exchange + clip + RMSprop fused in one kernel over NVLink peer memory" if getattr(learner, "_px", None) is not None
        else "one NCCL all-reduce of [grads | loss sums] per step")
    outputs = {}
    ms, phase_ms, launches, clocks = time_learner(
        ctx, learner, batch, a.steps, a.warmup, profile=not a.cuda_graph,
        after_timed=(lambda: outputs.update(learner_outputs(learner))) if a.dump_outputs else None)
    if a.dump_outputs and ctx.rank == 0:
        write_outputs(outputs, a.dump_outputs)
    if a.cuda_graph:
        phase_ms = profile_pass(learner, batch, 3)
    rec = learner_record(ctx, cfg, B_local, ms, phase_ms, launches, clocks, a.precision)
    value = (Bg if strong else ctx.world * Bg) / (ms * 1e-3)          # whole-job episodes per second

    e2e = None
    if not a.no_e2e:
        del batch
        e2e = e2e_learner(ctx, learner, fields, B_local, T, cfg["mixer"], a.e2e_steps)
    del fields, learner
    th.cuda.empty_cache()

    cpu = None
    if ctx.rank == 0 and ctx.world == 1 and not a.no_cpu_baseline:
        cb = a.cpu_batch or (32 if N > 5 else min(Bg, 64))
        cpu = cpu_learner(cfg, cb, 5, 1)

    select_actions, configs = None, None
    if extras:
        select_actions = rollout_record(ctx, a, 16384, a.precision, 200, 20, 0 if a.no_e2e else 10,
                                        with_cpu=(ctx.rank == 0 and ctx.world == 1 and not a.no_cpu_baseline))
        if ctx.world == 1 and a.config == "27m_vs_30m":
            try:
                select_actions["rollout_loop"] = rollout_loop_record(ctx, a.precision)
            except Exception as ex:
                select_actions["rollout_loop"] = {"error": repr(ex)[:300]}
            th.cuda.empty_cache()
            configs = {}
            for name in ("3m", "2s3z", "MMM2_vdn", "MMM2_iql"):
                try:
                    configs[name] = small_config_record(ctx, name, a.precision, 50, 5)
                except Exception as ex:
                    configs[name] = {"error": repr(ex)[:300]}
            try:
                configs["coma_2s3z"] = coma_record(ctx)
            except Exception as ex:
                configs["coma_2s3z"] = {"error": repr(ex)[:300]}

    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": rec["dtype"], "data": "synthetic",
            "config": {"workload": _workload_name(cfg), "name": a.config, "n_agents": N, "obs": O, "state": S, "n_actions": A,
                       "T": T, "global_batch": Bg if strong else ctx.world * Bg, "batch_per_gpu": B_local, "mixer": cfg["mixer"],
                       "episodes": "ragged" if a.ragged else "full-length",
                       "parallelism": "dp%d: episodes sharded; %s" % (ctx.world, exchange_desc),
                       "cuda_graph": bool(a.cuda_graph),
                       "l2_policy": "inputs (%.1f GB per GPU) exceed L2" % (input_bytes / 1e9)},
            "roofline": rec["roofline"], "step_roofline": rec["step_roofline"], "phases_ms": rec["phases_ms"],
            "kernels": rec["kernels"], "cpu_baseline": cpu, "clocks": rec["clocks"], "e2e": e2e,
            "gpu_launches": rec["gpu_launches"],
        }
        if weak:
            line["weak"] = weak
        if dp_equal is not None:
            line["dp_equal"] = dp_equal["ok"]
            line["dp_check"] = dp_equal
        if select_actions:
            line["select_actions"] = select_actions
        if configs:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
