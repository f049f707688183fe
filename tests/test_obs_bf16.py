"""bf16-stored observations (a scheme with ``"obs": {..., "dtype": th.bfloat16}``, pmb_batch.obs_dtype = PMB_DTYPE_BF16).

The bf16 tier rounds obs to bf16 before its first use, so where the kernels read bf16 obs natively a bf16-stored batch must
give exactly the bits of an fp32-stored batch holding the same bf16-representable values:
- the learner step (parameters, gradients, square_avg, loss sums, grad_norm; the forward images of keep_q = 3) for the four
  SMAC shapes, both streaming fc1 kernels (PMB_FC1_TS), full and ragged last tiles;
- through a zero-copy replay sample with padded-step skipping, CUDA-graph replay and a host batch streamed in chunks;
- the rollout step (actions, hidden state, q) for device and host runner batches;
- no hidden fp32 copy of obs is made;
- the fp32 tier, COMA and a no-fold shape convert, and match their result on obs.float();
- entry points that do not read bf16 obs reject it.
"""
import copy
import ctypes as C
import os

import numpy as np
import pytest
import torch as th

from pymarl_b200 import _lib
from pymarl_b200.components.episode_buffer import IndexedEpisodeBatch
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, numpy_episode_fields

NOFOLD = SmacShape("nofold", 30, 290, 64, 33, 6)          # agent id does not fit the K padding of obs (tests/test_fc1_tmem.py)
WIDE = SmacShape("wide", 4, 400, 64, 9, 6)               # O > 320: generic fc1 GEMM


def _dims(shape, precision="bf16", mixer="qmix", E=32, H=64):
    return _lib.make_dims(64, 20, shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, H, E, mixer=mixer,
                          precision=precision)


# ---- host-only checks ----------------------------------------------------------------------------------------------------

def test_batch_struct_matches_header():
    assert C.sizeof(_lib.Batch) == 128
    assert _lib.Batch.obs_dtype.offset == 120
    assert [k for k, _ in _lib.Batch._fields_][-1] == "obs_dtype"


def test_predicate():
    T, S = _lib.ENTRY_TRAIN_STEP, _lib.ENTRY_SELECT_ACTIONS
    for name in ("3m", "2s3z", "MMM2", "27m_vs_30m"):
        shape = SMAC_SHAPES[name]
        for mixer in ("qmix", "vdn", None):
            assert _lib.obs_bf16_supported(_dims(shape, mixer=mixer), T), (name, mixer)
        assert _lib.obs_bf16_supported(_dims(shape), S), name
        assert not _lib.obs_bf16_supported(_dims(shape, precision="fp32"), T)
        assert not _lib.obs_bf16_supported(_dims(shape, precision="fp32"), S)
        assert not _lib.obs_bf16_supported(_dims(shape, E=16), T)           # QMIX mixer off the tensor-core path
        assert not _lib.obs_bf16_supported(_dims(shape, H=32), T)
        assert not _lib.obs_bf16_supported(_dims(shape), 7)
    assert not _lib.obs_bf16_supported(_dims(NOFOLD), T)
    assert _lib.obs_bf16_supported(_dims(NOFOLD), S)                      # the rollout reads the agent id from a table
    assert not _lib.obs_bf16_supported(_dims(WIDE), T)
    assert not _lib.obs_bf16_supported(_dims(WIDE), S)
    bad = _dims(SMAC_SHAPES["3m"])
    bad.H = 48
    assert not _lib.obs_bf16_supported(bad, T)


def _fake_fields(shape, B=4, T=6, obs_dtype=th.bfloat16):
    N, O, A = shape.n_agents, shape.obs_dim, shape.n_actions
    return {"obs": th.zeros(B, T, N, O, dtype=obs_dtype), "state": th.zeros(B, T, shape.state_dim),
            "actions": th.zeros(B, T, N, 1, dtype=th.int64), "avail_actions": th.zeros(B, T, N, A, dtype=th.int32),
            "reward": th.zeros(B, T, 1), "terminated": th.zeros(B, T, 1, dtype=th.uint8),
            "filled": th.zeros(B, T, 1, dtype=th.int64)}


def test_make_batch_pass_through_and_convert(monkeypatch):
    monkeypatch.setattr(_lib, "require_cuda", lambda t, name: None)       # host tensors stand in for device ones here
    shape = SMAC_SHAPES["27m_vs_30m"]
    f = _fake_fields(shape)
    keep = []
    b = _lib.make_batch(f, keep=keep, dims=_dims(shape), entry=_lib.ENTRY_TRAIN_STEP)
    assert b.obs_dtype == 1 and b.obs == f["obs"].data_ptr() and b.obs_sb == f["obs"][0].numel()
    for dims, entry in ((None, None), (_dims(shape, precision="fp32"), _lib.ENTRY_TRAIN_STEP),
                        (_dims(NOFOLD), _lib.ENTRY_TRAIN_STEP)):
        keep = []
        b = _lib.make_batch(f, keep=keep, dims=dims, entry=entry)
        assert b.obs_dtype == 0 and b.obs != f["obs"].data_ptr()
        assert any(t.dtype == th.float32 and t.data_ptr() == b.obs for t in keep)
    f32 = _fake_fields(shape, obs_dtype=th.float32)
    b = _lib.make_batch(f32, dims=_dims(shape), entry=_lib.ENTRY_TRAIN_STEP)
    assert b.obs_dtype == 0 and b.obs == f32["obs"].data_ptr()
    # other fields keep their conversions
    f["reward"] = f["reward"].double()
    keep = []
    b = _lib.make_batch(f, keep=keep, dims=_dims(shape), entry=_lib.ENTRY_TRAIN_STEP)
    assert b.reward != f["reward"].data_ptr() and b.obs_dtype == 1


def _batch_ptrs(dtype):
    b = _lib.Batch()
    for k in ("obs", "state", "actions", "avail", "reward", "terminated", "filled"):
        setattr(b, k, 256)                      # never dereferenced: the calls must fail before any device work
        setattr(b, k + "_sb", 1)
    b.obs_dtype = dtype
    return b


def test_unsupported_entry_points_reject_bf16():
    L = _lib.lib()
    P = C.c_void_p(256)
    d_bf16, d_fp32 = _dims(SMAC_SHAPES["3m"]), _dims(SMAC_SHAPES["3m"], precision="fp32")
    b = _batch_ptrs(1)
    assert L.pmb_agent_fc1_fwd(C.byref(d_bf16), C.byref(b), 0, 1, P, P, None) == 1
    assert b"bf16 obs" in L.pmb_last_error()
    assert L.pmb_agent_unroll_bwd(C.byref(d_bf16), C.byref(b), P, P, P, P, P, P, P, P, 1 << 20, None) == 1
    hp = _lib.HParams(0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 0, 0)
    assert L.pmb_qlearner_train_step(C.byref(d_fp32), C.byref(b), C.byref(hp), P, P, P, P, P, 1 << 40, P, None) == 1
    assert L.pmb_qlearner_train_step(C.byref(_dims(NOFOLD)), C.byref(b), C.byref(hp), P, P, P, P, P, 1 << 40, P, None) == 1
    assert L.pmb_select_actions_step(C.byref(d_fp32), C.byref(b), 0, P, P, C.c_float(0), None, None, 0, 0, P, P, P,
                                     1 << 40, None) == 1
    dc = _dims(SMAC_SHAPES["3m"], precision="fp32", mixer=None, E=128)
    chp = _lib.ComaHParams(0.99, 0.8, 5e-4, 5e-4, 0.99, 1e-5, 10.0, 0.1)
    assert L.pmb_coma_train_step(C.byref(dc), C.byref(b), C.byref(chp), P, P, P, P, P, P, P, P, 1 << 40, P, None) == 1
    assert L.pmb_coma_critic_fwd(C.byref(dc), C.byref(b), P, 0, 1, P, P, 1 << 40, None) == 1
    b7 = _batch_ptrs(7)
    assert L.pmb_qlearner_train_step(C.byref(d_bf16), C.byref(b7), C.byref(hp), P, P, P, P, P, 1 << 40, P, None) == 1
    assert b"obs_dtype" in L.pmb_last_error()


# ---- GPU: learner step ---------------------------------------------------------------------------------------------------

def _args(shape, mixer="qmix", precision="bf16", **over):
    return default_args(shape, mixer=mixer, learner_log_interval=0, precision=precision, **over)


def _learner(shape, mixer="qmix", precision="bf16", seed=0, **over):
    from cuda_utils import build_learner
    th.manual_seed(seed)
    return build_learner(shape, _args(shape, mixer, precision, **over))[0]


def _pair(shape, B, T, seed=3, ragged=True, device="cuda"):
    """(fp32-stored batch, bf16-stored batch) with the same bf16-representable obs."""
    from cuda_utils import to_batch
    f = numpy_episode_fields(shape, B, T, seed=seed, ragged=ragged)
    f["obs"] = th.from_numpy(f["obs"]).to(th.bfloat16).float().numpy()
    b32 = to_batch(shape, f, device=device)
    b16 = to_batch(shape, f, device=device)
    b16.scheme["obs"]["dtype"] = th.bfloat16
    b16.data.transition_data["obs"] = b32.data.transition_data["obs"].to(th.bfloat16)
    return b32, b16


def _state(learner):
    th.cuda.synchronize()
    f = learner._flat
    return dict(p=f["p"].clone(), sq=f["sq"].clone(), target=f["target"].clone(), g=f["g"][:f["p"].numel()].clone(),
                stats=learner.last_stats.clone())


def _assert_equal(a, b):
    for k in a:
        assert th.equal(a[k], b[k]), k


def _with_ts(ts, fn):
    old = os.environ.get("PMB_FC1_TS")
    os.environ["PMB_FC1_TS"] = str(ts)
    try:
        return fn()
    finally:
        if old is None:
            del os.environ["PMB_FC1_TS"]
        else:
            os.environ["PMB_FC1_TS"] = old


def _train_twice(shape, mixer, batch, **over):
    lr = _learner(shape, mixer, **over)
    lr.train(batch, 0, 0)
    lr.train(batch, 1, 1)
    return _state(lr)


def _forward_workspace(shape, mixer, batch):
    """keep_q = 3: forward + loss sums only, every intermediate (obs / x images, ReLU mask, q) left in the workspace."""
    lr = _learner(shape, mixer, keep_q=3)
    lr.train(batch, 0, 0)
    lr._workspace.zero_()
    lr.train(batch, 0, 0)
    th.cuda.synchronize()
    return lr._workspace.clone()


CASES = [("27m_vs_30m", "qmix", 256, 12), ("27m_vs_30m", "qmix", 100, 12),
         ("3m", "vdn", 40, 30), ("3m", None, 40, 30), ("2s3z", "vdn", 60, 20), ("2s3z", None, 60, 20),
         ("MMM2", "vdn", 50, 16), ("MMM2", None, 50, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("ts", [1, 0])
@pytest.mark.parametrize("name,mixer,B,T", CASES)
def test_train_step_bit_identical(name, mixer, B, T, ts):
    shape = SMAC_SHAPES[name]
    b32, b16 = _pair(shape, B, T)
    a = _with_ts(ts, lambda: _train_twice(shape, mixer, b32))
    b = _with_ts(ts, lambda: _train_twice(shape, mixer, b16))
    _assert_equal(a, b)
    w32 = _with_ts(ts, lambda: _forward_workspace(shape, mixer, b32))
    w16 = _with_ts(ts, lambda: _forward_workspace(shape, mixer, b16))
    assert th.equal(w32, w16)


@pytest.mark.gpu
def test_zero_copy_sample_with_skipping():
    shape = SMAC_SHAPES["27m_vs_30m"]
    b32, b16 = _pair(shape, 120, 24)
    ids = th.as_tensor(np.random.default_rng(4).permutation(120)[:90], device="cuda")
    out = []
    for batch in (b32, b16):
        lr = _learner(shape, skip_padded_steps=True)
        lr.train(IndexedEpisodeBatch(batch, ids), 0, 0)
        lr.train(IndexedEpisodeBatch(batch, ids), 1, 1)
        out.append(_state(lr))
    _assert_equal(*out)


@pytest.mark.gpu
def test_cuda_graph_replay():
    shape = SMAC_SHAPES["2s3z"]
    pairs = [_pair(shape, 48, 30, seed=s) for s in (1, 2)]
    out = []
    for k in (0, 1):
        lr = _learner(shape, cuda_graph=True)
        for i in range(3):
            for j, p in enumerate(pairs):
                lr.train(p[k], 2 * i + j, 2 * i + j)
        assert any(isinstance(e, tuple) for e in lr._graphs.values())
        out.append(_state(lr))
    _assert_equal(*out)


@pytest.mark.gpu
def test_host_streamed_batch():
    shape = SMAC_SHAPES["MMM2"]
    b32, b16 = _pair(shape, 150, 20, seed=13, device="cpu")
    out = []
    for batch in (b32, b16):
        lr = _learner(shape, "vdn", host_stream_chunk=64)         # 3 chunks
        lr.train(batch, 0, 0)
        out.append(_state(lr))
    _assert_equal(*out)


@pytest.mark.gpu
def test_no_hidden_obs_copy():
    shape = SMAC_SHAPES["27m_vs_30m"]
    b32, b16 = _pair(shape, 64, 60)
    obs32_bytes = b32["obs"].numel() * 4
    lr = _learner(shape)
    ids = th.arange(64, device="cuda").flip(0).contiguous()
    for batch in (b16, IndexedEpisodeBatch(b16, ids)):
        lr.train(batch, 0, 0)                  # warm-up: workspace
        th.cuda.synchronize()
        base = th.cuda.memory_allocated()
        th.cuda.reset_peak_memory_stats()
        lr.train(batch, 1, 1)
        th.cuda.synchronize()
        assert th.cuda.max_memory_allocated() - base < obs32_bytes // 4


@pytest.mark.gpu
@pytest.mark.parametrize("shape,precision,mixer", [(SMAC_SHAPES["3m"], "fp32", "qmix"), (NOFOLD, "bf16", "qmix"),
                                                   (SMAC_SHAPES["3m"], "bf16", "qmix_e16")])
def test_converting_paths_match_float_obs(shape, precision, mixer):
    b32, b16 = _pair(shape, 20, 16, seed=4)
    over = dict(mixing_embed_dim=16) if mixer == "qmix_e16" else {}
    a = _train_twice(shape, "qmix", b32, precision=precision, **over)
    b = _train_twice(shape, "qmix", b16, precision=precision, **over)
    _assert_equal(a, b)


@pytest.mark.gpu
def test_coma_converts():
    from test_coma_gpu import COMA_KW, build_coma
    shape = SMAC_SHAPES["3m"]
    b32, b16 = _pair(shape, 8, 16, seed=6)
    out = []
    for batch in (b32, b16):
        th.manual_seed(0)
        lr, _ = build_coma(shape, default_args(shape, mixer=None, **COMA_KW))
        lr.train(batch, 0, 0)
        lr.train(batch, 1, 0)
        th.cuda.synchronize()
        out.append((lr._flat["ap"].clone(), lr._flat["cp"].clone(), lr.last_stats.clone()))
    for x, y in zip(*out):
        assert th.equal(x, y)


# ---- GPU: rollout --------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("device", ["cuda", "cpu"])
@pytest.mark.parametrize("shape", [SMAC_SHAPES["27m_vs_30m"], SMAC_SHAPES["3m"], NOFOLD], ids=lambda s: s.name)
def test_select_actions_bit_identical(shape, device):
    # NOFOLD: the agent id comes from a table, not from the K padding of obs (fold_id = 0)
    B, N, A = 300, shape.n_agents, shape.n_actions
    pair = _pair(shape, B, 6, seed=8, ragged=False, device=device)
    g = th.Generator(device="cuda").manual_seed(5)
    draws = [(th.rand(B, N, generator=g, device="cuda"), th.empty(B, N, A, device="cuda").exponential_(generator=g))
             for _ in range(3)]
    out = []
    for batch in pair:
        mac = _learner(shape).mac
        mac.init_hidden(B)
        res = []
        for t, (u, expo) in enumerate(draws):
            q, act = mac._run_step(batch, t, epsilon=0.3, u=u, expo=expo, want_actions=True, want_q=True)
            res += [q.clone(), act.clone(), mac.hidden_states.clone()]
        th.cuda.synchronize()
        out.append(res)
    for x, y in zip(*out):
        assert th.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim", [30, 285])
def test_vector_runner_stores_rounded_obs(obs_dim):
    from cuda_utils import build_learner
    from pymarl_b200.runners import SyntheticVectorEnv, VectorRunner
    shape = SMAC_SHAPES["3m"]._replace(obs_dim=obs_dim)
    args = default_args(shape, mixer="qmix", learner_log_interval=0, precision="bf16", device="cuda", batch_size_run=32,
                        action_rng="philox")
    learner, _ = build_learner(shape, args)
    env = SyntheticVectorEnv(32, shape.n_agents, obs_dim, shape.state_dim, shape.n_actions, episode_limit=6, seed=3, p_end=0.0)
    seen = []
    get_obs = env.get_obs
    env.get_obs = lambda: seen.append(get_obs().clone()) or seen[-1]
    runner = VectorRunner(args, env)
    info = env.get_env_info()
    from pymarl_b200.components.transforms import OneHot
    scheme = {"state": {"vshape": info["state_shape"]},
              "obs": {"vshape": obs_dim, "group": "agents", "dtype": th.bfloat16},
              "actions": {"vshape": (1,), "group": "agents", "dtype": th.long},
              "avail_actions": {"vshape": (info["n_actions"],), "group": "agents", "dtype": th.int},
              "reward": {"vshape": (1,)}, "terminated": {"vshape": (1,), "dtype": th.uint8}}
    runner.setup(learner.mac, scheme=scheme, groups={"agents": shape.n_agents},
                 preprocess={"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])})
    batch = runner.run(test_mode=False)
    obs = batch["obs"]
    assert obs.dtype == th.bfloat16 and len(seen) == 7
    for t, o in enumerate(seen):
        assert th.equal(obs[:, t], o.to(th.bfloat16)), t
    learner.train(batch, runner.t_env, 32)
    assert np.isfinite(learner.stats()["loss"])
