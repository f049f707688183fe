"""A/B of padded-step skipping (args.skip_padded_steps) on the learner step.

Workload: BASELINE config 4 (QMIX, 27m_vs_30m, B = 4096, T = 180, bf16 tier), once with the bench's ragged episode
generator (torch_episode_fields(..., ragged=True)) and once with full-length episodes.  ONE learner (one workspace of
~52 GB) is toggled between the arms; per workload the arms alternate off / on --rounds times, each with its own warm-up.

Printed as one JSON line: the median ms / step of each arm (CUDA events around --steps steps), the per-phase times of
one profiled step per arm (pmb_profile_begin / end; the schedule's own launches are the phase "skip_schedule"), the live
(t, tile) item fraction of the skipping arm, an output check (full-length: bit-identical updated parameters and loss
sums; ragged: relative differences) and the card name, power limit and SM clock read in the same run.

    python tools/ragged_bench.py [--steps 20] [--warmup 3] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


class _DictBatch:
    def __init__(self, fields, batch_size, max_seq_length):
        self.fields, self.batch_size, self.max_seq_length = fields, batch_size, max_seq_length
        self.device = next(iter(fields.values())).device

    def __getitem__(self, k):
        return self.fields[k]


def _gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(q.split(","), out))
    except Exception as ex:                      # reported, not fatal
        return {"error": repr(ex)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--T", type=int, default=180)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch as th
    if not th.cuda.is_available():
        raise SystemExit("ragged_bench: no CUDA device (timings are only meaningful on the GPU)")
    from cuda_utils import Logger
    from pymarl_b200 import _lib, le_REGISTRY, mac_REGISTRY
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, torch_episode_fields

    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T = a.batch, a.T
    args = default_args(shape, mixer="qmix", device="cuda", use_cuda=True, learner_log_interval=10 ** 12, precision="bf16")
    th.manual_seed(7)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    learner = le_REGISTRY["q_learner"](mac_REGISTRY["basic_mac"](scheme, groups, args), scheme, Logger(), args)
    learner.cuda()
    p0 = {k: learner._ensure_flat()[k].clone() for k in ("p", "sq", "target")}

    def restore():
        for k, v in p0.items():
            learner._flat[k].copy_(v)

    def run(batch, skip, n):
        args.skip_padded_steps = skip
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            learner.train(batch, i, 0)
        e1.record()
        th.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def profiled(batch, skip):
        args.skip_padded_steps = skip
        th.cuda.synchronize()
        _lib.profile_begin()
        learner.train(batch, 0, 0)
        phases = _lib.profile_end(max_phases=64)
        out = {}
        for name, ms in phases:
            out[name] = round(out.get(name, 0.0) + ms, 4)
        return out

    def outputs(batch, skip):
        restore()
        args.skip_padded_steps = skip
        learner.train(batch, 0, 0)
        th.cuda.synchronize()
        return learner._flat["p"].clone(), learner.last_stats.clone()

    rec = {"config": "27m_vs_30m qmix bf16", "B": B, "T": T, "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
           "gpu": _gpu_info(), "workloads": {}}
    agent_phases = ("fc1_fwd_both_tc", "gru_unroll_fwd_both_tc", "gru_unroll_fwd_online_tc", "gru_unroll_fwd_target_tc",
                    "q_select_tc", "gru_unroll_bwd_tc", "dW_fc1_fc2_tc")
    for wl, ragged in (("ragged", True), ("full", False)):
        fields = torch_episode_fields(shape, B, T, seed=4242, ragged=ragged, device="cuda", with_onehot=False)
        batch = _DictBatch(fields, B, T)
        ms = {"off": [], "on": []}
        for r in range(a.rounds):
            for arm, skip in (("off", False), ("on", True)):
                run(batch, skip, a.warmup)
                ms[arm].append(run(batch, skip, a.steps))
        ph = {"off": profiled(batch, False), "on": profiled(batch, True)}
        v = learner.workspace_views(learner._last_dims)
        n_tiles = -(-B * shape.n_agents // 128)
        live = float(v["tile_steps"].double().sum()) / (T * n_tiles)
        (p_off, s_off), (p_on, s_on) = outputs(batch, False), outputs(batch, True)
        restore()
        w = {"ms_off": [round(x, 3) for x in ms["off"]], "ms_on": [round(x, 3) for x in ms["on"]],
             "median_ms_off": round(statistics.median(ms["off"]), 3), "median_ms_on": round(statistics.median(ms["on"]), 3),
             "live_item_fraction": round(live, 4), "phases_ms_off": ph["off"], "phases_ms_on": ph["on"],
             "agent_phase_ratio_on_off": {k: round(ph["on"][k] / ph["off"][k], 3) for k in agent_phases
                                          if k in ph["on"] and k in ph["off"] and ph["off"][k] > 0},
             "skip_schedule_ms": ph["on"].get("skip_schedule")}
        w["ratio_on_off"] = round(w["median_ms_on"] / w["median_ms_off"], 4)
        if ragged:
            w["params_rel_diff"] = float((p_on - p_off).abs().max() / p_off.abs().max())
            w["loss_sums_rel_diff"] = float(((s_on[:5] - s_off[:5]).abs() / s_off[:5].abs()).max())
        else:
            w["outputs_bit_identical"] = bool(th.equal(p_on, p_off) and th.equal(s_on, s_off))
        rec["workloads"][wl] = w
        del fields, batch
        th.cuda.empty_cache()
    rec["gpu_after"] = _gpu_info()
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
