"""The data-parallel exchange and the replicated update on ONE GPU, against float64 references.

A. pmb_dp_pack / pmb_dp_unpack: the five loss sums as (hi, lo) float pairs behind the gradient.  Round trips, the zeroed
   tail floats, and the fp32 rank-order sum of W packed tails: mask_sum exact (an odd global count above 2^24 included),
   the other sums within (W - 1) 2^-24 of the sum of their magnitudes, and bit for bit what a float64 model of the packing
   predicts.
B. pmb_dp_fused_allreduce_update with simulated peers: W exchange buffers on the one device, the peers' ready / done flags
   pre-set in the launching rank's flag block, so one launch runs to completion with no concurrent peer.  Three
   consecutive step ids on one zeroed scratch (the grid barrier's counter grows across steps); clip inactive / active,
   target sync on / off, target NULL.  Against the float64 reference and, bit for bit, against the all-reduce path
   (pack, fp32 rank-order sum, unpack, pmb_clip_rmsprop_update) on the same inputs.  Host only: the refusals.
C. QLearner.train sharded over W real ranks (processes, gloo) that share cuda:0, on the all-reduce path (dp_exchange =
   "nccl"; the transport is a rank-order fp32 sum of host copies, as NCCL refuses two ranks on one device).  Every batch
   kind, both tiers, ranks without episodes.  Replicas bit-identical; against one learner on the whole batch and, on the
   fp32 tier, against the float64 oracle over three chained steps.
D. The learner's fused-path plumbing (grad_view binding, step ids, the PeerExchange branch) as rank 0 of 2 whose peer
   contributes zeros: equal to the whole-batch single-GPU step.
The fused kernel never runs from two processes here, and no test leaves a flag missing (the ~2 s spin timeout).
"""
import copy
import ctypes as C
import datetime
import os
import sys

import numpy as np
import pytest
import torch as th

from pymarl_b200 import _lib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PX_MAX_WORLD = 8
LR, ALPHA, EPS = 5e-4, 0.99, 1e-5
# the values the kernels compute with (fp32 arguments; 1.f - alpha is 1e-6 off 0.01)
A32, LR32, EPS32 = float(np.float32(ALPHA)), float(np.float32(LR)), float(np.float32(EPS))
ONE_MINUS_A32 = float(np.float32(1.0) - np.float32(ALPHA))


def _align4(x):
    return -(-x // 4) * 4


def _rel(a, b):
    """max|a - b| / max|b|"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


# ---- A. pack / unpack --------------------------------------------------------------------------------------------------

def _pack_model(v):
    """float64 model of dp_pack_sum (common.cuh) for stats[0:5] -> the 16 tail floats."""
    out = np.zeros(16, np.float32)
    for i, x in enumerate(np.asarray(v, np.float64)):
        hi = np.floor(x / 4096.0) * 4096.0 if i == 0 else float(np.float32(x))
        out[2 * i], out[2 * i + 1] = np.float32(hi), np.float32(x - hi)
    return out


def _unpack_model(tail):
    return np.array([float(tail[2 * i]) + float(tail[2 * i + 1]) for i in range(5)])


def _dev_pack(sums, n=3, garbage=float("nan")):
    """pmb_dp_pack of stats[0:5] = sums into a gradient buffer of n floats whose tail held `garbage`; -> the tail."""
    g = th.full((n + _lib.DP_TAIL_FLOATS,), garbage, dtype=th.float32, device="cuda")
    st = th.zeros(_lib.STATS_LEN, dtype=th.float64, device="cuda")
    st[:5] = th.tensor(np.asarray(sums, np.float64))
    _lib.check(_lib.lib().pmb_dp_pack(n, _lib.ptr(g), _lib.ptr(st), _lib.stream_ptr()), "pmb_dp_pack")
    return g[n:].cpu().numpy()


def _dev_unpack(tail, n=5):
    g = th.zeros(n + _lib.DP_TAIL_FLOATS, dtype=th.float32, device="cuda")
    g[n:] = th.from_numpy(np.asarray(tail, np.float32))
    st = th.full((_lib.STATS_LEN,), -7.0, dtype=th.float64, device="cuda")
    _lib.check(_lib.lib().pmb_dp_unpack(n, _lib.ptr(g), _lib.ptr(st), _lib.stream_ptr()), "pmb_dp_unpack")
    out = st.cpu().numpy()
    assert (out[5:] == -7.0).all()                          # only the five sums are written
    return out[:5]


def _rank_sums(rng, mask):
    """One rank's five loss sums: the mask count and four doubles of the sizes and signs a step produces."""
    return np.array([float(mask), mask * rng.uniform(0.1, 3.0), mask * rng.uniform(0.1, 1.5),
                     mask * rng.normal(0.0, 2.0), mask * rng.normal(0.0, 2.0)])


@pytest.mark.gpu
def test_pack_unpack_round_trip():
    rng = np.random.default_rng(1)
    ints = [[2 ** 24 - 1, 16777215, 1, 0, 12345], [1, 2, 3, 4, 5], [8388609, 2 ** 23, 77, 4095, 4097]]
    ints += [[c, 1, 2, 3, 4] for c in (2 ** 24 + 1, 19795969, 2 ** 31 + 12345, 2 ** 36 - 1)]   # counts above 2^24
    for v in ints:
        tail = _dev_pack(v)
        assert (tail[10:] == 0).all(), tail
        np.testing.assert_array_equal(tail, _pack_model(v))
        np.testing.assert_array_equal(_dev_unpack(tail), np.asarray(v, np.float64))
    for garbage in (float("nan"), 1e30, -3.0):
        for _ in range(4):
            v = np.concatenate([[float(rng.integers(0, 2 ** 24))],
                                rng.choice([-1, 1], 4) * 10.0 ** rng.uniform(-20, 20, 4) * rng.random(4)])
            tail = _dev_pack(v, n=int(rng.integers(1, 9)), garbage=garbage)
            assert (tail[10:] == 0).all(), tail                  # tail floats 10..15 zeroed whatever they held
            np.testing.assert_array_equal(tail, _pack_model(v))
            got = _dev_unpack(tail)
            assert got[0] == v[0]
            assert (np.abs(got[1:] - v[1:]) <= 2.0 ** -48 * np.abs(v[1:])).all(), (got, v)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_rank_sum_of_packed_tails(world):
    """The tails of W ranks summed in fp32 in rank order (what the all-reduce does to them), then unpacked."""
    rng = np.random.default_rng(world)
    totals = [int(rng.integers(world, 2 ** 22)), 2 ** 24 + 1, 4096 * 179 * 27 + 1]     # two odd totals above 2^24
    for total in totals:
        cut = np.sort(rng.integers(0, total + 1, world - 1))
        masks = np.diff(np.concatenate([[0], cut, [total]]))                            # uneven per-rank counts
        sums = [_rank_sums(rng, m) for m in masks]
        tails = [_dev_pack(s) for s in sums]
        for t, s in zip(tails, sums):
            np.testing.assert_array_equal(t, _pack_model(s))
        acc = tails[0].copy()
        for t in tails[1:]:
            acc += t                                                                     # fp32, rank order
        got = _dev_unpack(acc)
        exact = np.sum(sums, axis=0)
        assert got[0] == total, (total, got[0])
        mag = np.sum(np.abs(sums), axis=0)
        err = np.abs(got[1:] - exact[1:])
        assert (err <= (world - 1) * 2.0 ** -24 * mag[1:] + 2.0 ** -46 * mag[1:]).all(), (world, err / mag[1:])
        np.testing.assert_array_equal(got, _unpack_model(acc))


# ---- B. the fused kernel with simulated peers --------------------------------------------------------------------------

def _n_27m_qmix():
    from pymarl_b200.synthetic import SMAC_SHAPES
    s = SMAC_SHAPES["27m_vs_30m"]
    d = _lib.make_dims(1, 2, s.n_agents, s.obs_dim, s.state_dim, s.n_actions, 64, 32, mixer="qmix")
    return int(_lib.flat_layout(d).n_total)


def _error_word(scratch, n):
    off = ((4 * n + 255) // 256) * 256 + 1024 + 16                 # PeerExchange.error_word
    return int(scratch[off:off + 4].view(th.int32).item())


# per step: (clip: None = inactive, else this fraction of the step's norm; do_target_sync; pass the target buffer)
FUSED_STEPS = ((None, 0, True), (0.5, 1, True), (0.8, 1, False))


@pytest.mark.gpu
@pytest.mark.parametrize("n", ["1", "3", "5", "150", "200003", "27m_qmix"])
@pytest.mark.parametrize("world,rank", [(2, 0), (2, 1), (3, 0), (3, 2), (8, 0), (8, 7)])
def test_fused_update_with_simulated_peers(world, rank, n):
    """n: no float4 body (1, 3), a float4 body with tails (5, 150 = 4 k + 2), a grid-stride loop that turns (200003 >
    64 blocks x 256 threads x 4), and the flat parameter count of 27m_vs_30m QMIX."""
    n = _n_27m_qmix() if n == "27m_qmix" else int(n)
    L = _lib.lib()
    dev = "cuda"
    rng = np.random.default_rng(1000 * world + 10 * rank + n % 7)
    nx = L.pmb_dp_exchange_floats(n)
    flag_off = _align4(n + _lib.DP_TAIL_FLOATS)
    assert nx == flag_off + 2 * PX_MAX_WORLD * 2
    bufs = [th.zeros(nx, dtype=th.float32, device=dev) for _ in range(world)]
    ptrs = (C.c_void_p * world)(*[b.data_ptr() for b in bufs])
    flags = bufs[rank][flag_off:].view(th.int64)                     # ready[8] | done[8] of the launching rank
    scratch = th.zeros(4 * n + 4096, dtype=th.uint8, device=dev)    # zeroed once, kept for the three steps
    opt_scratch = th.empty(4096, dtype=th.float32, device=dev)
    p0 = (rng.standard_normal(n) * 1e-3).astype(np.float32)        # of the size of an update: the p check sees it
    sq0 = rng.uniform(1e-3, 1e-2, n).astype(np.float32)
    tg0 = rng.standard_normal(n).astype(np.float32)
    p, sq, tg = (th.from_numpy(x).to(dev) for x in (p0, sq0, tg0))       # fused path
    pc, sqc, tgc = p.clone(), sq.clone(), tg.clone()                      # all-reduce path
    p64, sq64, tg64 = p0.astype(np.float64), sq0.astype(np.float64), tg0.astype(np.float64)
    stats = th.zeros(_lib.STATS_LEN, dtype=th.float64, device=dev)
    s = _lib.stream_ptr()
    for step, (clip_frac, do_sync, with_target) in enumerate(FUSED_STEPS, 1):
        masks = rng.integers(1, 50, world)
        sums = [_rank_sums(rng, m) for m in masks]
        g = [(rng.standard_normal(n) * 30.0).astype(np.float32) for _ in range(world)]
        # float64 reference (orc.clip_grad_norm / orc.rmsprop_step on the flat vector)
        M = float(np.sum(masks))
        gs = np.sum([x.astype(np.float64) for x in g], axis=0) / M
        norm = float(np.sqrt((gs ** 2).sum()))
        clip = np.float32(1e30 if clip_frac is None else clip_frac * norm)
        coef = min(1.0, float(clip) / (norm + 1e-6))
        gv = gs * coef
        sq64 = A32 * sq64 + ONE_MINUS_A32 * gv * gv
        p64 = p64 - LR32 * gv / (np.sqrt(sq64) + EPS32)
        if do_sync and with_target:
            tg64 = p64.copy()

        # the peers' gradients and packed tails (what their own P0 would have written), the launching rank's gradient
        for r in range(world):
            bufs[r][:n] = th.from_numpy(g[r])
            if r != rank:
                st_r = th.zeros(_lib.STATS_LEN, dtype=th.float64, device=dev)
                st_r[:5] = th.from_numpy(sums[r])
                _lib.check(L.pmb_dp_pack(n, _lib.ptr(bufs[r]), _lib.ptr(st_r), s), "pmb_dp_pack")
        for r in range(world):
            if r != rank:
                flags[r] = step
                flags[PX_MAX_WORLD + r] = step
        stats.zero_()
        stats[:5] = th.from_numpy(sums[rank])
        tg_before = tg.clone()
        _lib.check(L.pmb_dp_fused_allreduce_update(world, rank, ptrs, n, step, _lib.ptr(p), _lib.ptr(sq),
                                                   _lib.ptr(tg) if with_target else None, do_sync, _lib.ptr(stats),
                                                   LR, ALPHA, EPS, float(clip), _lib.ptr(scratch), scratch.numel(), s),
                   "pmb_dp_fused_allreduce_update")

        # the all-reduce path on the same inputs
        packed = []
        for r in range(world):
            b = th.empty(n + _lib.DP_TAIL_FLOATS, dtype=th.float32, device=dev)
            b[:n] = th.from_numpy(g[r])
            st_r = th.zeros(_lib.STATS_LEN, dtype=th.float64, device=dev)
            st_r[:5] = th.from_numpy(sums[r])
            _lib.check(L.pmb_dp_pack(n, _lib.ptr(b), _lib.ptr(st_r), s), "pmb_dp_pack")
            packed.append(b)
        acc = packed[0].clone()
        for b in packed[1:]:
            acc += b                                                       # fp32, rank order
        stc = th.zeros(_lib.STATS_LEN, dtype=th.float64, device=dev)
        _lib.check(L.pmb_dp_unpack(n, _lib.ptr(acc), _lib.ptr(stc), s), "pmb_dp_unpack")
        _lib.check(L.pmb_clip_rmsprop_update(n, _lib.ptr(pc), _lib.ptr(acc), _lib.ptr(sqc),
                                             _lib.ptr(tgc) if with_target else None, do_sync, _lib.ptr(stc), LR, ALPHA,
                                             EPS, float(clip), _lib.ptr(opt_scratch), s), "pmb_clip_rmsprop_update")
        th.cuda.synchronize()
        where = (world, rank, n, step)
        assert _error_word(scratch, n) == 0, where
        st, st_c = stats.cpu().numpy(), stc.cpu().numpy()
        g_loc = bufs[rank][:n].cpu().numpy()                               # what .grad shows after the step

        # float64 reference, fp32 tolerance
        exact = np.sum(sums, axis=0)
        assert st[0] == M, where
        mag = np.sum(np.abs(sums), axis=0)
        assert (np.abs(st[1:5] - exact[1:]) <= 1e-6 * mag[1:]).all(), where
        assert abs(st[5] - norm) <= 1e-6 * norm, (where, st[5], norm)
        assert abs(st[6] - exact[1] / M) <= 1e-6 * exact[1] / M, where
        if clip_frac is None:
            assert st[7] == 1.0, (where, st[7])                            # clamped to exactly 1
        else:
            assert st[7] < 1.0 and abs(st[7] - coef) <= 1e-6 * coef, (where, st[7], coef)
        assert _rel(g_loc, gv) < 1e-6, (where, _rel(g_loc, gv))
        assert _rel(sq.cpu().numpy(), sq64) < 1e-6, where
        assert _rel(p.cpu().numpy(), p64) < 1e-6, where
        if with_target:
            assert _rel(tg.cpu().numpy(), tg64) < 1e-6, where
        else:
            assert th.equal(tg, tg_before), where

        # the all-reduce path: norm and coefficient within one fp32 ulp, equal coefficients on these seeds, and then
        # the same bits everywhere
        for k in (5, 7):
            assert abs(st[k] - st_c[k]) <= np.spacing(np.float32(st_c[k])), (where, k, st[k], st_c[k])
        assert st[7] == st_c[7], where
        np.testing.assert_array_equal(st[[0, 1, 2, 3, 4, 6]], st_c[[0, 1, 2, 3, 4, 6]])
        assert th.equal(bufs[rank][:n], acc[:n]), where
        assert th.equal(p, pc) and th.equal(sq, sqc) and th.equal(tg, tgc), where


def test_fused_update_refusals():
    """Host only: every malformed call returns an error code and a message before anything is launched.  The pointers
    are never dereferenced: peer 1 is NULL in every call, so even a check that let a call through would stop at it."""
    L = _lib.lib()
    n = 1000
    fake = 1 << 24
    need = ((4 * n + 255) // 256) * 256 + 1024 + 64
    bufs = (C.c_void_p * 9)(*([fake, None] + [fake] * 7))

    def call(world=2, rank=0, step=1, scratch_bytes=need):
        return L.pmb_dp_fused_allreduce_update(world, rank, bufs, n, step, fake, fake, fake, 1, fake, 5e-4, 0.99, 1e-5,
                                               10.0, fake, scratch_bytes, None)

    launches = L.pmb_launch_count()
    cases = dict(world_1=(dict(world=1), "world must be"), world_9=(dict(world=9), "world must be"),
                 rank_negative=(dict(rank=-1), "world must be"), rank_world=(dict(rank=2), "world must be"),
                 step_0=(dict(step=0), "step ids start at 1"), null_peer=(dict(world=3, rank=2), "peer buffer 1 is NULL"),
                 scratch_short=(dict(scratch_bytes=need - 1), "scratch too small"))
    for what, (kw, why) in cases.items():
        rc = call(**kw)
        msg = L.pmb_last_error().decode()
        assert rc != 0, what
        assert msg.startswith("dp_fused") and why in msg, (what, msg)
    assert L.pmb_launch_count() == launches


# ---- C. QLearner.train sharded over real ranks that share cuda:0 (all-reduce path) -------------------------------------

SHAPE, T_EP = "3m", 10
# per step: (t_env, episode_num, grad_norm_clip); target_update_interval = 1, so the second step syncs the targets, and
# its clip is active
STEPS = ((0, 0, 1e30), (1, 1, 1e-3), (2, 1, 10.0))
# id: (mixer, precision, batch kind, B (None: world - 1, so the last rank has no episodes), extra args)
DP_CASES = {
    "qmix_fp32": ("qmix", "fp32", "device", 7, {}),
    "vdn_fp32": ("vdn", "fp32", "device", 7, {}),
    "iql_fp32": (None, "fp32", "device", 7, {}),
    "qmix_bf16": ("qmix", "bf16", "device", 7, {}),
    "vdn_bf16": ("vdn", "bf16", "device", 7, {}),
    "hbm_sample": ("qmix", "bf16", "hbm", 7, {}),            # ep_index: tensor-core tier only
    "pinned_sample": ("qmix", "fp32", "pinned", 7, {}),
    "pageable_host": ("qmix", "fp32", "pageable", 7, {}),
    "host_stream_dp": ("qmix", "fp32", "pinned_host", 13, dict(host_stream_dp=True, host_stream_chunk=2)),
    "skip_padded": ("qmix", "bf16", "device", 7, dict(skip_padded_steps=True)),
    "uneven": ("vdn", "fp32", "device", 5, {}),
    "no_shard": ("qmix", "fp32", "device", 7, dict(dp_shard_batch=False)),
    # last, so that a failure here leaves the results of the cases above in place
    "empty_rank_device": ("qmix", "fp32", "device", None, {}),
    "empty_rank_hbm": ("vdn", "bf16", "hbm", None, {}),
    "empty_rank_pinned": ("qmix", "fp32", "pinned", None, {}),
    "empty_rank_pageable": ("qmix", "bf16", "pageable", None, {}),
}


def _case_fields(case, world):
    """(numpy fields of the whole batch in episode order, episode ids into the buffer or None, buffer fields or None)."""
    from pymarl_b200.synthetic import SMAC_SHAPES, numpy_episode_fields
    _, _, kind, B, _ = DP_CASES[case]
    B = world - 1 if B is None else B
    shape = SMAC_SHAPES[SHAPE]
    if kind in ("hbm", "pinned"):
        buf = numpy_episode_fields(shape, B + 4, T_EP, seed=21, ragged=True)
        ids = np.random.default_rng(22).permutation(B + 4)[:B]
        return {k: v[ids] for k, v in buf.items()}, ids, buf
    return numpy_episode_fields(shape, B, T_EP, seed=23, ragged=True), None, None


def _case_batch(case, fields, ids, buf_fields):
    from cuda_utils import to_batch
    from pymarl_b200.components.episode_buffer import IndexedEpisodeBatch, ReplayBuffer
    from pymarl_b200.components.transforms import OneHot
    from pymarl_b200.synthetic import SMAC_SHAPES, make_scheme
    shape = SMAC_SHAPES[SHAPE]
    kind = DP_CASES[case][2]
    if kind == "device":
        return to_batch(shape, fields)
    if kind in ("pageable", "pinned_host"):
        b = to_batch(shape, fields, device="cpu")
        if kind == "pinned_host":
            for k, v in b.data.transition_data.items():
                b.data.transition_data[k] = v.pin_memory()
        return b
    scheme, groups = make_scheme(shape)
    pre = {"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])}
    n_buf = buf_fields["obs"].shape[0]
    where = "cuda" if kind == "hbm" else "cpu"
    rb = ReplayBuffer(scheme, groups, n_buf, T_EP, pre, where, pin_memory=(kind == "pinned"))
    rb.insert_episode_batch(to_batch(shape, buf_fields, device=where))
    host_ids = th.as_tensor(ids, dtype=th.int64)
    return IndexedEpisodeBatch(rb, host_ids.cuda(), host_ids=host_ids if kind == "pinned" else None)


def _init_params(args):
    from oracle import qlearner_oracle as orc
    from pymarl_b200.synthetic import SMAC_SHAPES
    shape = SMAC_SHAPES[SHAPE]
    rng = np.random.default_rng(5)
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + shape.n_actions + shape.n_agents, 64, shape.n_actions), rng)
    mixer = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, 32), rng) if args.mixer == "qmix" else None
    return agent, mixer


def _case_args(case, **over):
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args
    mixer, precision, _, _, extra = DP_CASES[case]
    kw = dict(learner_log_interval=0, precision=precision, target_update_interval=1, dp_exchange="nccl")
    kw.update(extra)
    kw.update(over)
    return default_args(SMAC_SHAPES[SHAPE], mixer=mixer, **kw)


def _run_case(case, world, rank=None):
    """Three steps of QLearner.train; rank None: one learner on the whole batch without data parallelism."""
    from cuda_utils import build_learner
    from pymarl_b200 import data_parallel
    from pymarl_b200.synthetic import SMAC_SHAPES
    fields, ids, buf_fields = _case_fields(case, world)
    args = _case_args(case)
    if rank is not None and not getattr(args, "dp_shard_batch", True):
        lo, hi = data_parallel.shard_slice(fields["obs"].shape[0], rank, world)      # the caller passes its own episodes
        fields = {k: v[lo:hi] for k, v in fields.items()}
    agent, mixer = _init_params(args)
    learner, _ = build_learner(SMAC_SHAPES[SHAPE], args, agent, agent, mixer, mixer)
    assert learner._px is None
    learner._flat["sq"].fill_(1e-2)
    batch = _case_batch(case, fields, ids, buf_fields)
    out = {"p_init": learner._flat["p"].cpu().numpy()}
    for i, (t_env, ep, clip) in enumerate(STEPS):
        learner.args.grad_norm_clip = clip
        learner.train(batch, t_env, ep)
        for k in ("p", "sq", "target"):
            out["%s%d" % (k, i)] = learner._flat[k].cpu().numpy()
        out["stats%d" % i] = learner._stats.cpu().numpy()
    if DP_CASES[case][2] == "pinned_host":
        assert learner._hs is not None                       # the streamed path ran
    return out


def _dp_child(rank, world, port, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    th.cuda.set_device(0)
    from pymarl_b200 import data_parallel

    def allreduce_step(buf):
        """Rank-order fp32 sum of host copies (NCCL refuses two ranks on one device)."""
        parts = [th.empty(buf.shape, dtype=buf.dtype) for _ in range(world)]
        dist.all_gather(parts, buf.cpu())
        acc = parts[0]
        for x in parts[1:]:
            acc += x
        buf.copy_(acc)

    data_parallel.allreduce_step = allreduce_step
    assert data_parallel.is_active() and data_parallel.rank() == rank
    for case in DP_CASES:
        out = _run_case(case, world, rank)
        np.savez(os.path.join(out_dir, "%s_r%d.npz" % (case, rank)), **out)
    dist.barrier()
    dist.destroy_process_group()


_SPAWNED = {}


@pytest.fixture(scope="module")
def dp_results(tmp_path_factory):
    """world -> (directory of the ranks' results, error of the spawn or None); the ranks are spawned once per world."""
    import torch.multiprocessing as mp

    def get(world):
        if world not in _SPAWNED:
            out = tmp_path_factory.mktemp("dp_world%d" % world)
            err = None
            try:
                mp.spawn(_dp_child, args=(world, 31000 + os.getpid() % 2000 + world, str(out)), nprocs=world, join=True)
            except Exception as e:          # a failing rank: the others are terminated, the results so far kept
                err = "the ranks stopped at an earlier or this case:\n" + str(e)[-3000:]
            _SPAWNED[world] = (str(out), err)
        return _SPAWNED[world]
    yield get
    _SPAWNED.clear()


def _layout_slices(mixer):
    from pymarl_b200.synthetic import SMAC_SHAPES
    s = SMAC_SHAPES[SHAPE]
    lay = _lib.flat_layout(_lib.make_dims(1, 2, s.n_agents, s.obs_dim, s.state_dim, s.n_actions, 64, 32, mixer=mixer))
    return {name: (lay.offset[i], lay.numel[i]) for i, name in enumerate(_lib.PARAM_ORDER) if lay.numel[i]}


def _stat_values(st, n_agents):
    m = st[0]
    return dict(loss=st[1] / m, grad_norm=st[5], td_error_abs=st[2] / m, q_taken_mean=st[3] / (m * n_agents),
                target_mean=st[4] / (m * n_agents))


def _oracle_steps(case, world):
    """The same three steps in the float64 oracle on the whole batch: per step (stats, flat p, flat target)."""
    from oracle import qlearner_oracle as orc
    fields, _, _ = _case_fields(case, world)
    args = _case_args(case)
    agent, mixer = _init_params(args)
    o = orc.OracleQLearner({k: v.astype(np.float64) for k, v in agent.items()},
                           {k: v.astype(np.float64) for k, v in (mixer or {}).items()}, copy.copy(args))
    for sq in list(o.sq_agent.values()) + list(o.sq_mixer.values()):
        sq[...] = 1e-2
    f64 = {k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in fields.items()}
    out = []
    for t_env, ep, clip in STEPS:
        o.args.grad_norm_clip = clip
        stats, _, _ = o.train(f64, t_env, ep)
        p = {"agent." + k: v.copy() for k, v in o.agent.items()}
        p.update({"mixer." + k: v.copy() for k, v in o.mixer_p.items()})
        tg = {"agent." + k: v.copy() for k, v in o.target_agent.items()}
        tg.update({"mixer." + k: v.copy() for k, v in o.target_mixer_p.items()})
        out.append((stats, p, tg))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", list(DP_CASES))
def test_sharded_learner_on_one_gpu(dp_results, world, case):
    """Three steps (the second syncs the targets with the clip active) of QLearner.train over W ranks on cuda:0.
    Replicas bit-identical.  Against one learner on the whole batch: mask_sum exact; fp32 tier loss, grad_norm and every
    parameter / target tensor (max|a - b| / max|b|) within 1e-6, as bench.dp_self_check; bf16 tier 1e-3 and the update
    1e-2 in relative L2.  fp32 tier also against the float64 oracle at test_config_matrix's bounds (stats 2e-5,
    parameters 5e-5)."""
    from pymarl_b200.synthetic import SMAC_SHAPES
    out_dir, err = dp_results(world)
    paths = [os.path.join(out_dir, "%s_r%d.npz" % (case, r)) for r in range(world)]
    assert all(os.path.exists(p) for p in paths), err
    ranks = [dict(np.load(p)) for p in paths]
    for k in ranks[0]:
        for r in range(1, world):
            a, b = (ranks[r][k], ranks[0][k]) if not k.startswith("stats") else (ranks[r][k][:8], ranks[0][k][:8])
            np.testing.assert_array_equal(a, b, err_msg="%s differs on rank %d" % (k, r))     # stats: the 8 named slots
    got = ranks[0]
    ref = _run_case(case, world)
    mixer, precision = DP_CASES[case][:2]
    n_agents = SMAC_SHAPES[SHAPE].n_agents
    slices = _layout_slices(mixer)
    tol = 1e-6 if precision == "fp32" else 1e-3
    oracle = _oracle_steps(case, world) if precision == "fp32" else None
    for i in range(len(STEPS)):
        st, st_ref = got["stats%d" % i], ref["stats%d" % i]
        assert st[0] == st_ref[0], (i, st[0], st_ref[0])
        if i == 1:
            assert st[7] < 1.0 and st_ref[7] < 1.0, (st[7], st_ref[7])             # the clip is active
        if i == 0:
            assert st[7] == 1.0 and st_ref[7] == 1.0
        for k in ("loss", "grad_norm"):
            a, b = _stat_values(st, n_agents)[k], _stat_values(st_ref, n_agents)[k]
            assert abs(a - b) <= tol * abs(b), (i, k, a, b)
        for k in ("p", "target"):
            for name, (o, n) in slices.items():
                e = _rel(got["%s%d" % (k, i)][o:o + n], ref["%s%d" % (k, i)][o:o + n])
                assert e <= tol, (i, k, name, e)
        if precision == "bf16":
            prev = "p%d" % (i - 1) if i else "p_init"
            u = got["p%d" % i].astype(np.float64) - got[prev]
            u_ref = ref["p%d" % i].astype(np.float64) - ref[prev]
            e = float(np.linalg.norm(u - u_ref) / np.linalg.norm(u_ref))
            assert e <= 1e-2, (i, e)
        if oracle is not None:
            ost, op, otg = oracle[i]
            mine = _stat_values(st, n_agents)
            for k in ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean"):
                assert abs(mine[k] - ost[k]) <= 2e-5 * max(1.0, abs(ost[k])), (i, k, mine[k], ost[k])
            for name, (o, n) in slices.items():
                e = _rel(got["p%d" % i][o:o + n], op[name].ravel())
                assert e < 5e-5, (i, "param", name, e)
                e = _rel(got["target%d" % i][o:o + n], otg[name].ravel())
                assert e < 5e-5, (i, "target", name, e)


# ---- D. the fused-path plumbing of the learner with a silent peer ------------------------------------------------------

@pytest.mark.gpu
def test_learner_fused_path_with_a_silent_peer(monkeypatch):
    """The learner as rank 0 of 2 with dp_shard_batch = False, its PeerExchange's second buffer all zeros (a peer without
    episodes) and that peer's flags raised before each step: three steps equal the whole-batch single-GPU step within
    1e-6, mask_sum exact, and fc1.weight.grad holds the same normalised, clipped gradient."""
    from cuda_utils import build_learner, to_batch
    from pymarl_b200 import data_parallel
    from pymarl_b200.synthetic import SMAC_SHAPES, default_args, numpy_episode_fields
    shape = SMAC_SHAPES["2s3z"]
    args = default_args(shape, mixer="qmix", learner_log_interval=0, target_update_interval=1)
    fields = numpy_episode_fields(shape, 9, 12, seed=31, ragged=True)
    batch = to_batch(shape, fields)
    rng = np.random.default_rng(8)
    from oracle import qlearner_oracle as orc
    agent = orc.init_params(orc.agent_param_shapes(shape.obs_dim + shape.n_actions + shape.n_agents, 64, shape.n_actions), rng)
    mixer = orc.init_params(orc.qmix_param_shapes(shape.state_dim, shape.n_agents, 32), rng)

    def run(learner):
        learner._flat["sq"].fill_(1e-2)
        res = []
        for t_env, ep, clip in STEPS:
            learner.args.grad_norm_clip = clip
            learner.train(batch, t_env, ep)
            res.append((learner._stats.cpu().numpy(), learner._flat["p"].cpu().numpy(),
                        learner._flat["target"].cpu().numpy(), learner.mac.agent.fc1.weight.grad.cpu().numpy()))
        return res

    ref_learner, _ = build_learner(shape, copy.copy(args), agent, agent, mixer, mixer)
    ref = run(ref_learner)

    class SilentPeer(data_parallel.PeerExchange):
        def __init__(self, n, device):
            L = _lib.lib()
            self.n, self.step, self.ok, self.world, self.rank = n, 0, True, 2, 0
            self.buf = th.zeros(L.pmb_dp_exchange_floats(n), dtype=th.float32, device=device)
            self.peer = th.zeros_like(self.buf)
            self.scratch = th.zeros(4 * n + 4096, dtype=th.uint8, device=device)
            self._mapped = []
            self.ptrs = (C.c_void_p * 2)(self.buf.data_ptr(), self.peer.data_ptr())

        def fused_update(self, *a, **kw):
            flags = self.buf[_align4(self.n + _lib.DP_TAIL_FLOATS):].view(th.int64)
            flags[1] = flags[PX_MAX_WORLD + 1] = self.step + 1      # the peer is ready and done for the coming step
            super().fused_update(*a, **kw)

    monkeypatch.setattr(data_parallel, "is_active", lambda: True)
    monkeypatch.setattr(data_parallel, "rank", lambda: 0)
    monkeypatch.setattr(data_parallel, "world_size", lambda: 2)
    monkeypatch.setattr(data_parallel, "PeerExchange", SilentPeer)
    args.dp_shard_batch = False
    learner, _ = build_learner(shape, args, agent, agent, mixer, mixer)
    px = learner._px
    assert isinstance(px, SilentPeer)
    assert learner._flat["g"].data_ptr() == px.buf.data_ptr()
    got = run(learner)
    assert px.step == len(STEPS) and px.error_word() == 0
    assert not px.peer[:px.n + _lib.DP_TAIL_FLOATS].any()
    for i, ((st, p, tg, g), (st_r, p_r, tg_r, g_r)) in enumerate(zip(got, ref)):
        assert st[0] == st_r[0], i
        assert st[7] == 1.0 if i == 0 else (i != 1 or st[7] < 1.0), (i, st[7])
        for k in (1, 2, 3, 4, 5, 6, 7):
            assert abs(st[k] - st_r[k]) <= 1e-6 * abs(st_r[k]), (i, k, st[k], st_r[k])
        assert _rel(p, p_r) <= 1e-6 and _rel(tg, tg_r) <= 1e-6, i
        assert _rel(g, g_r) <= 1e-6, (i, _rel(g, g_r))
