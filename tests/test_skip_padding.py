"""Padded-step skipping in the tensor-core learner step (args.skip_padded_steps, pmb_dims.reserved bit 1).

The step sorts the episodes by the forward steps they need, F_b = min(T, l_b + 2) (l_b = last filled step, F_b = 0 for an
empty episode), longest first and stable, and the agent kernels run only the (t, tile) items some row still needs.
- the schedule (ep_order, tile_steps) matches the host computation, for a plain batch and a zero-copy replay sample;
- on a full-length batch nothing can be skipped and the step is bit-identical to the step without the flag;
- fed in the same (sorted) order, the skipping step computes the same values as the full step;
- against today's unsorted step the results differ only by fp32 summation order;
- all-padding episodes change nothing, and their tiles run no steps;
- a CUDA graph captured with one set of lengths replays correctly with others;
- the host-streamed path and the places where the flag is ignored (fp32 tier, no-fold shapes).
"""
import ctypes as C

import numpy as np
import pytest
import torch as th

from pymarl_b200 import _lib
from pymarl_b200.components.episode_buffer import IndexedEpisodeBatch
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, numpy_episode_fields

NOFOLD = SmacShape("nofold", 30, 290, 64, 33, 6)          # agent id does not fit the K padding of obs (tests/test_fc1_tmem.py)


def _args(shape, mixer="qmix", skip=False, precision="bf16", **over):
    return default_args(shape, mixer=mixer, learner_log_interval=0, precision=precision, skip_padded_steps=skip, **over)


def _learner(shape, mixer="qmix", skip=False, precision="bf16", seed=0, **over):
    from cuda_utils import build_learner
    th.manual_seed(seed)
    return build_learner(shape, _args(shape, mixer, skip, precision, **over))[0]


def _fields(shape, B, T, seed=3, ragged=True, n_empty=0):
    f = numpy_episode_fields(shape, B, T, seed=seed, ragged=ragged)
    if n_empty:
        f = {k: np.concatenate([v, np.zeros((n_empty,) + v.shape[1:], dtype=v.dtype)]) for k, v in f.items()}
    return f


def _steps_host(filled):
    """F_b from filled [B, T, 1]."""
    f = np.asarray(filled)[..., 0] != 0
    T = f.shape[1]
    last = np.where(f.any(1), T - 1 - np.argmax(f[:, ::-1], axis=1), -1)
    return np.where(last < 0, 0, np.minimum(T, last + 2))


def _tile_steps_host(F_sorted, N, n_tiles):
    return np.array([F_sorted[(tile * 128) // N] for tile in range(n_tiles)])


def _state(learner):
    th.cuda.synchronize()
    f = learner._flat
    return dict(p=f["p"].clone(), sq=f["sq"].clone(), target=f["target"].clone(), g=f["g"][:f["p"].numel()].clone(),
                stats=learner.last_stats.clone())


def _views(learner):
    return learner.workspace_views(learner._last_dims)


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / max(float(b.double().abs().max()), 1e-30))


# ---- 9. plumbing (no GPU) ----------------------------------------------------------------------------------------------

def test_make_dims_skip_padding_bit():
    d = _lib.make_dims(4, 10, 3, 30, 48, 9, 64, 32, precision="bf16")
    assert d.reserved & 2 == 0
    d = _lib.make_dims(4, 10, 3, 30, 48, 9, 64, 32, precision="bf16", skip_padding=True)
    assert d.reserved == 2
    names = [k for k, _ in _lib.WsViews._fields_]
    assert names[-2:] == ["ep_order", "tile_steps"]


def test_learner_args_reach_reserved_bit():
    from types import SimpleNamespace
    from pymarl_b200.learners.q_learner import QLearner
    shape = SMAC_SHAPES["3m"]
    for skip, want in ((False, 0), (True, 2)):
        args = _args(shape, skip=skip)
        fake = SimpleNamespace(args=args, mac=SimpleNamespace(agent=SimpleNamespace(d_in=shape.obs_dim + shape.n_actions +
                                                                                   shape.n_agents)),
                               mixer=SimpleNamespace(state_dim=shape.state_dim), precision="bf16")
        d = QLearner._layout_dims(fake, B=8, T=20)
        assert d.reserved & 2 == want
    del args.skip_padded_steps
    assert QLearner._layout_dims(fake, B=8, T=20).reserved & 2 == 0


# ---- 1. the schedule ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("zero_copy", [False, True])
def test_schedule_matches_host(zero_copy):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T, N = 300, 60, shape.n_agents
    fields = _fields(shape, B, T, n_empty=10)
    rng = np.random.default_rng(5)
    # make some holes: a hole must not shorten an episode
    fl = fields["filled"]
    fl[3, 2] = 0
    fl[7, 10] = 0
    batch = to_batch(shape, fields)
    learner = _learner(shape, skip=True)
    F = _steps_host(fields["filled"])
    if zero_copy:
        ids = rng.permutation(B + 10)[:250]
        learner.train(IndexedEpisodeBatch(batch, th.as_tensor(ids, device="cuda")), 0, 0)
        F_rows = F[ids]
    else:
        ids = np.arange(B + 10)
        learner.train(batch, 0, 0)
        F_rows = F
    v = _views(learner)
    perm = np.argsort(-F_rows, kind="stable")
    assert np.array_equal(v["ep_order"].cpu().numpy(), ids[perm])
    n_tiles = -(-len(F_rows) * N // 128)
    assert np.array_equal(v["tile_steps"].cpu().numpy(), _tile_steps_host(F_rows[perm], N, n_tiles))
    assert np.isfinite(learner.last_stats.cpu().numpy()).all()


# ---- 2. full-length batch: bit-identical ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape,B,T", [("27m_vs_30m", 64, 40), ("3m", 32, 60)])
def test_full_length_batch_bit_identical(shape, B, T):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape]
    batch = to_batch(shape, _fields(shape, B, T, ragged=False))
    out = []
    for skip in (False, True):
        learner = _learner(shape, skip=skip)
        learner.train(batch, 0, 0)
        learner.train(batch, 1, 1)
        out.append(_state(learner))
        if skip:
            v = _views(learner)
            assert np.array_equal(v["ep_order"].cpu().numpy(), np.arange(B))
            assert (v["tile_steps"] == T).all()
    for k in out[0]:
        assert th.equal(out[0][k], out[1][k]), k


# ---- 3. same order with and without skipping -----------------------------------------------------------------------

def _named_grads(learner, g):
    L = learner._flat["layout"]
    names = ["fc1_w", "fc1_b", "w_ih", "w_hh", "b_ih", "b_hh", "fc2_w", "fc2_b"]
    out = {n: g[L.offset[i]:L.offset[i] + L.numel[i]] for i, n in enumerate(names)}
    out["mixer"] = g[L.n_agent:L.n_total]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape,mixer,B,T", [("27m_vs_30m", "qmix", 512, 120),   # many tiles, two tiles per forward CTA
                                             ("2s3z", "qmix", 40, 60),           # one tile per CTA, forked target pass
                                             ("MMM2", "vdn", 128, 80),
                                             ("MMM2", None, 128, 80)])
def test_same_order_with_and_without_skipping(shape, mixer, B, T):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape]
    fields = _fields(shape, B, T, seed=11)
    batch = to_batch(shape, fields)
    on = _learner(shape, mixer, skip=True, keep_q=0)
    on.train(batch, 0, 0)
    s_on = _state(on)
    v_on = {k: t.clone() for k, t in _views(on).items()}
    order = v_on["ep_order"]
    off = _learner(shape, mixer, skip=False)
    off.train(IndexedEpisodeBatch(batch, order.clone()), 0, 0)
    s_off = _state(off)
    v_off = _views(off)
    assert "ep_order" not in v_off

    F = _steps_host(fields["filled"])[order.cpu().numpy()]
    live = th.as_tensor(np.arange(T - 1)[None, :] < (F - 1)[:, None], device="cuda")      # t <= l_b, [B, T-1]
    for k in ("chosen", "tmax", "q_tot", "t_tot"):
        a, b = v_on[k], v_off[k]
        m = live[..., None].expand_as(a)
        assert th.equal(a[m], b[m]), k
    assert th.equal(s_on["stats"][:5], s_off["stats"][:5])
    g_on, g_off = _named_grads(on, s_on["g"]), _named_grads(off, s_off["g"])
    for k in ("w_ih", "w_hh", "b_ih", "b_hh", "mixer"):
        assert th.equal(g_on[k], g_off[k]), k
    # the fc1 / fc2 weight gradients are summed over a per-CTA split of the items that moves with the live item count:
    # fp32 summation order only (2.0e-6 measured on 27m_vs_30m / 512 x 120, B200)
    for k in ("fc1_w", "fc1_b", "fc2_w", "fc2_b"):
        assert _rel(g_on[k], g_off[k]) < 5e-6, (k, _rel(g_on[k], g_off[k]))


# ---- 4. against today's unsorted step ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape,mixer,B,T", [("27m_vs_30m", "qmix", 256, 100), ("MMM2", "vdn", 128, 80)])
def test_against_unsorted_step(shape, mixer, B, T):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape]
    batch = to_batch(shape, _fields(shape, B, T, seed=21))
    st = []
    for skip in (False, True):
        learner = _learner(shape, mixer, skip=skip)
        learner.train(batch, 0, 0)
        st.append((learner, _state(learner)))
    (l0, a), (l1, b) = st
    for i in range(5):
        assert abs(float(a["stats"][i]) - float(b["stats"][i])) <= 1e-9 * abs(float(a["stats"][i])) + 1e-12, i
    ga, gb = _named_grads(l0, a["g"]), _named_grads(l1, b["g"])
    for k in ga:
        if ga[k].numel():
            assert _rel(gb[k], ga[k]) < 1e-5, (k, _rel(gb[k], ga[k]))
    assert _rel(b["p"], a["p"]) < 1e-5


# ---- 5. all-padding episodes -------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_padding_episodes_change_nothing():
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T, N = 128, 60, shape.n_agents
    res = []
    for n_empty in (0, 12):
        learner = _learner(shape, skip=True)
        learner.train(to_batch(shape, _fields(shape, B, T, seed=9, n_empty=n_empty)), 0, 0)
        res.append((learner, _state(learner), _views(learner)["tile_steps"].cpu().numpy()))
    (l0, a, _), (l1, b, ts) = res
    for i in range(5):
        assert abs(float(a["stats"][i]) - float(b["stats"][i])) <= 1e-6 * abs(float(a["stats"][i])), i
    assert _rel(b["g"], a["g"]) < 1e-6
    # rows B*N .. (B+12)*N are the empty episodes (sorted last): every tile made only of them runs no step
    first_empty_tile = -(-B * N // 128)
    assert (ts[first_empty_tile:] == 0).all() and len(ts) > first_empty_tile
    assert (ts[:first_empty_tile] > 0).all()


# ---- 6. CUDA graph with changing lengths ----------------------------------------------------------------------------

@pytest.mark.gpu
def test_cuda_graph_with_changing_lengths():
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["2s3z"]
    B, T = 48, 50
    contents = [_fields(shape, B, T, seed=s) for s in (1, 2, 3, 4)]
    graphed = _learner(shape, skip=True, cuda_graph=True)
    eager = _learner(shape, skip=True)
    batch = to_batch(shape, contents[0])
    for i, c in enumerate(contents):
        for k, v in c.items():                        # new content, same tensors: the graph key does not change
            batch.data.transition_data[k].copy_(th.from_numpy(np.ascontiguousarray(v)).cuda())
        # the eager learner starts from the graphed learner's parameters
        for k in ("p", "sq", "target"):
            eager._flat[k].copy_(graphed._flat[k])
        eager.optimiser.step_count = graphed.optimiser.step_count
        graphed.train(batch, i, i)
        eager.train(batch, i, i)
        a, b = _state(graphed), _state(eager)
        for k in a:
            assert th.equal(a[k], b[k]), (i, k)
    assert any(isinstance(e, tuple) for e in graphed._graphs.values())       # captured and replayed


# ---- 7. host-streamed batch --------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_host_streamed_batch():
    from cuda_utils import to_batch
    shape = SMAC_SHAPES["2s3z"]
    B, T = 200, 60
    fields = _fields(shape, B, T, seed=13)
    dev = _learner(shape, skip=True)
    dev.train(to_batch(shape, fields), 0, 0)
    host = _learner(shape, skip=True, host_stream_chunk=64)
    hb = to_batch(shape, fields, device="cpu")
    host.train(hb, 0, 0)
    a, b = _state(host), _state(dev)
    for i in range(5):
        assert abs(float(a["stats"][i]) - float(b["stats"][i])) <= 1e-5 * abs(float(b["stats"][i])), i
    assert _rel(a["g"], b["g"]) < 1e-5
    assert _rel(a["p"], b["p"]) < 1e-5


# ---- 8. flag ignored where unsupported -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape,precision", [("3m", "fp32"), (NOFOLD, "bf16")])
def test_flag_ignored_where_unsupported(shape, precision):
    from cuda_utils import to_batch
    shape = SMAC_SHAPES[shape] if isinstance(shape, str) else shape
    batch = to_batch(shape, _fields(shape, 20, 30, seed=4))
    out = []
    for skip in (False, True):
        learner = _learner(shape, skip=skip, precision=precision)
        learner.train(batch, 0, 0)
        out.append(_state(learner))
        d = learner._last_dims
        v = _lib.WsViews()
        _lib.check(_lib.lib().pmb_learner_workspace_views(C.byref(d), _lib.ptr(learner._workspace),
                                                          learner._workspace.numel(), C.byref(v)), "views")
        assert not v.ep_order and not v.tile_steps
        if skip:
            d0 = _lib.make_dims(d.B, d.T, d.N, d.O, d.S, d.A, d.H, d.E, mixer="qmix", precision=precision)
            assert _lib.lib().pmb_learner_workspace_bytes(C.byref(d)) == _lib.lib().pmb_learner_workspace_bytes(C.byref(d0))
    for k in out[0]:
        assert th.equal(out[0][k], out[1][k]), k
