"""Compact state / avail_actions storage: a scheme with ``"state": {..., "dtype": th.bfloat16}`` and
``"avail_actions": {..., "dtype": th.uint8}`` (or ``th.bool``), pmb_batch.state_dtype / avail_dtype.

The tensor-core mixer rounds state to bf16 before its first use and avail holds 0 / 1, so where the kernels read the
compact cells natively a compact batch must give exactly the bits of fp32 / int32 storage of the same values:
- the learner step (parameters, gradients, square_avg, loss sums, grad_norm, target after a sync) for QMIX, VDN and IQL on
  the bf16 tier, with bf16 obs too, through the device batch, HBM and pinned-host zero-copy samples (chunked and in one
  piece), the host-streamed path, CUDA graphs, ragged batches with padded-step skipping and a strided batch[:, :t] view;
- the rollout step (actions, q, hidden state) with injected draws and with Philox, for device and host runner batches;
- no hidden conversion of the replay buffer's state / avail;
- the fp32 tier, COMA and the shapes off the tensor-core kernels convert, and match explicitly converted inputs;
- entry points that do not read a compact dtype reject it, as they reject unknown dtype values.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch as th

from pymarl_b200 import _lib
from pymarl_b200.components.episode_buffer import EpisodeBatch, IndexedEpisodeBatch, ReplayBuffer
from pymarl_b200.components.transforms import OneHot
from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, make_scheme, numpy_episode_fields

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDE_A = SmacShape("wide_a", 4, 40, 52, 70, 6)            # A > 64: the agent runs off the tensor-core kernels
T_, S_ = _lib.ENTRY_TRAIN_STEP, _lib.ENTRY_SELECT_ACTIONS
F32, BF16, U8 = _lib.DTYPE_F32, _lib.DTYPE_BF16, _lib.DTYPE_U8


def _dims(shape, precision="bf16", mixer="qmix", E=32, H=64):
    return _lib.make_dims(64, 20, shape.n_agents, shape.obs_dim, shape.state_dim, shape.n_actions, H, E, mixer=mixer,
                          precision=precision)


# ---- host-only checks ----------------------------------------------------------------------------------------------------

def test_batch_tail_matches_header():
    hdr = open(os.path.join(REPO, "include", "pymarl_b200.h")).read()
    body = re.search(r"typedef struct pmb_batch \{(.*?)\} pmb_batch;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    assert re.findall(r"(\w+);", body)[-3:] == ["obs_dtype", "state_dtype", "avail_dtype"]
    assert "int16_t state_dtype" in body and "int16_t avail_dtype" in body
    assert C.sizeof(_lib.Batch) == 128
    assert [(k, getattr(_lib._BatchTail, k).offset) for k, _ in _lib._BatchTail._fields_] == \
        [("obs_dtype", 0), ("state_dtype", 4), ("avail_dtype", 6)]
    b = _lib.Batch()
    assert (b.obs_dtype, b.state_dtype, b.avail_dtype) == (0, 0, 0)
    b.obs_dtype, b.state_dtype, b.avail_dtype = 1, 1, 2
    assert bytes(b)[120:128] == bytes([1, 0, 0, 0, 1, 0, 2, 0])


def test_predicate():
    sup = _lib.field_dtype_supported
    for name in ("3m", "2s3z", "MMM2", "27m_vs_30m"):
        shape = SMAC_SHAPES[name]
        d = _dims(shape)
        for entry in (T_, S_):
            for field in ("obs", "state", "avail_actions"):
                assert sup(d, entry, field, F32)                              # the reference types: everywhere
                assert sup(_dims(shape, precision="fp32"), entry, field, F32)
            assert sup(d, entry, "obs", BF16) == _lib.obs_bf16_supported(d, entry)
            assert not sup(d, entry, "obs", U8) and not sup(d, entry, "state", U8) and not sup(d, entry, "avail_actions", BF16)
        assert sup(d, T_, "state", BF16) and not sup(d, S_, "state", BF16)
        assert sup(d, T_, "avail_actions", U8) and sup(d, S_, "avail_actions", U8)
        for mixer in ("vdn", None):                                           # no mixer reads state
            assert not sup(_dims(shape, mixer=mixer), T_, "state", BF16)
            assert sup(_dims(shape, mixer=mixer), T_, "avail_actions", U8)
        assert not sup(_dims(shape, E=16), T_, "state", BF16)                 # QMIX mixer off the tensor-core path
        assert sup(_dims(shape, E=16), T_, "avail_actions", U8)               # ... the agent still on it
        for entry in (T_, S_):
            for field, dt in (("state", BF16), ("avail_actions", U8)):
                assert not sup(_dims(shape, precision="fp32"), entry, field, dt)
            assert not sup(_dims(shape, H=32), entry, "avail_actions", U8)    # the agent off the tensor-core kernels
            assert sup(_dims(shape, H=32), entry, "state", BF16) == (entry == T_)   # ... the mixer still on them
            assert not sup(d, entry, "avail_actions", 3)                      # unknown dtype value
        assert not sup(d, 7, "avail_actions", U8) and not sup(d, 7, "state", F32)
        assert _lib.lib().pmb_field_dtype_supported(C.byref(d), T_, 3, 0) == 0     # unknown field
    for entry in (T_, S_):
        assert not sup(_dims(WIDE_A), entry, "avail_actions", U8)
    bad = _dims(SMAC_SHAPES["3m"])
    bad.H = 48
    assert not sup(bad, T_, "avail_actions", U8)


def _fake_fields(shape, B=4, T=6, state=th.bfloat16, avail=th.uint8, obs=th.float32):
    N, O, A = shape.n_agents, shape.obs_dim, shape.n_actions
    return {"obs": th.zeros(B, T, N, O, dtype=obs), "state": th.zeros(B, T, shape.state_dim, dtype=state),
            "actions": th.zeros(B, T, N, 1, dtype=th.int64), "avail_actions": th.zeros(B, T, N, A, dtype=avail),
            "reward": th.zeros(B, T, 1), "terminated": th.zeros(B, T, 1, dtype=th.uint8),
            "filled": th.zeros(B, T, 1, dtype=th.int64)}


@pytest.mark.parametrize("avail", [th.uint8, th.bool])
def test_make_batch_pass_through_and_convert(monkeypatch, avail):
    monkeypatch.setattr(_lib, "require_cuda", lambda t, name: None)       # host tensors stand in for device ones here
    shape = SMAC_SHAPES["27m_vs_30m"]
    f = _fake_fields(shape, avail=avail)
    b = _lib.make_batch(f, dims=_dims(shape), entry=T_)
    assert (b.state_dtype, b.avail_dtype) == (BF16, U8)
    assert b.state == f["state"].data_ptr() and b.avail == f["avail_actions"].data_ptr()
    assert b.state_sb == f["state"][0].numel() and b.avail_sb == f["avail_actions"][0].numel()
    b = _lib.make_batch(f, need_state=False, dims=_dims(shape), entry=S_)    # the rollout
    assert (b.state_dtype, b.avail_dtype) == (F32, U8) and b.avail == f["avail_actions"].data_ptr()
    # QMIX with E = 16: state converted, avail passed through
    keep = []
    b = _lib.make_batch(f, keep=keep, dims=_dims(shape, E=16), entry=T_)
    assert (b.state_dtype, b.avail_dtype) == (F32, U8) and b.avail == f["avail_actions"].data_ptr()
    assert any(t.dtype == th.float32 and t.data_ptr() == b.state for t in keep)
    # converted everywhere else
    for dims, entry in ((None, None), (_dims(shape, precision="fp32"), T_), (_dims(shape, precision="fp32"), S_),
                        (_dims(shape), 7)):
        keep = []
        b = _lib.make_batch(f, keep=keep, dims=dims, entry=entry)
        assert (b.obs_dtype, b.state_dtype, b.avail_dtype) == (0, 0, 0)
        assert any(t.dtype == th.float32 and t.data_ptr() == b.state for t in keep)
        assert any(t.dtype == th.int32 and t.data_ptr() == b.avail for t in keep)
    # A > 64: avail converted, state (the mixer is on the tensor-core path) passed through
    keep = []
    b = _lib.make_batch(_fake_fields(WIDE_A, avail=avail), keep=keep, dims=_dims(WIDE_A), entry=T_)
    assert (b.state_dtype, b.avail_dtype) == (BF16, F32)
    assert any(t.dtype == th.int32 and t.data_ptr() == b.avail for t in keep)
    # other dtypes keep converting to the reference type, on the compact path too
    for st, av in ((th.float16, th.int64), (th.float64, th.int8)):
        keep = []
        b = _lib.make_batch(_fake_fields(shape, state=st, avail=av), keep=keep, dims=_dims(shape), entry=T_)
        assert (b.state_dtype, b.avail_dtype) == (0, 0)
        assert {t.dtype for t in keep if t.data_ptr() in (b.state, b.avail)} == {th.float32, th.int32}
    # reference storage is untouched
    f32 = _fake_fields(shape, state=th.float32, avail=th.int32)
    b = _lib.make_batch(f32, dims=_dims(shape), entry=T_)
    assert (b.state_dtype, b.avail_dtype) == (0, 0) and b.state == f32["state"].data_ptr()


def _batch_ptrs(obs=0, state=0, avail=0):
    b = _lib.Batch()
    for k in ("obs", "state", "actions", "avail", "reward", "terminated", "filled"):
        setattr(b, k, 256)                      # never dereferenced: the calls must fail before any device work
        setattr(b, k + "_sb", 1)
    b.obs_dtype, b.state_dtype, b.avail_dtype = obs, state, avail
    return b


def test_entry_points_reject_what_they_do_not_read():
    L = _lib.lib()
    P = C.c_void_p(256)
    hp = _lib.HParams(0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 0, 0)
    d_bf16, d_fp32 = _dims(SMAC_SHAPES["3m"]), _dims(SMAC_SHAPES["3m"], precision="fp32")
    dc = _dims(SMAC_SHAPES["3m"], precision="fp32", mixer=None, E=128)
    chp = _lib.ComaHParams(0.99, 0.8, 5e-4, 5e-4, 0.99, 1e-5, 10.0, 0.1)
    for kw, what in ((dict(state=BF16), b"bf16 state"), (dict(avail=U8), b"uint8 avail"),
                     (dict(state=7), b"state_dtype"), (dict(avail=1), b"avail_dtype"), (dict(avail=-1), b"avail_dtype")):
        b = _batch_ptrs(**kw)
        calls = [
            lambda: L.pmb_qlearner_train_step(C.byref(d_fp32), C.byref(b), C.byref(hp), P, P, P, P, P, 1 << 40, P, None),
            lambda: L.pmb_select_actions_step(C.byref(d_fp32), C.byref(b), 0, P, P, C.c_float(0), None, None, 0, 0, P, P,
                                              P, 1 << 40, None),
            lambda: L.pmb_target_select(C.byref(d_bf16), C.byref(b), P, P, P, P, None, None),
            lambda: L.pmb_mixer_fwd(C.byref(d_bf16), C.byref(b), P, P, 0, P, P, None),
            lambda: L.pmb_mixer_bwd(C.byref(d_bf16), C.byref(b), P, P, P, P, P, P, P, 1 << 40, None),
            lambda: L.pmb_td_loss(C.byref(d_bf16), C.byref(b), P, P, C.c_float(0.99), P, P, None),
            lambda: L.pmb_agent_fc1_fwd(C.byref(d_bf16), C.byref(b), 0, 1, P, P, None),
            lambda: L.pmb_agent_unroll_bwd(C.byref(d_bf16), C.byref(b), P, P, P, P, P, P, P, P, 1 << 20, None),
            lambda: L.pmb_coma_train_step(C.byref(dc), C.byref(b), C.byref(chp), P, P, P, P, P, P, P, P, 1 << 40, P, None),
            lambda: L.pmb_coma_critic_fwd(C.byref(dc), C.byref(b), P, 0, 1, P, P, 1 << 40, None),
        ]
        if "state" in kw and kw["state"] == BF16:     # the rollout never reads state: no native bf16 state there either
            calls.append(lambda: L.pmb_select_actions_step(C.byref(d_bf16), C.byref(b), 0, P, P, C.c_float(0), None, None,
                                                           0, 0, P, P, P, 1 << 40, None))
        if kw.get("avail") == U8:                     # A > 64: the agent off the tensor-core kernels
            calls.append(lambda: L.pmb_qlearner_train_step(C.byref(_dims(WIDE_A)), C.byref(b), C.byref(hp), P, P, P, P, P,
                                                           1 << 40, P, None))
        if kw.get("state") == BF16:                   # QMIX with E = 16: the mixer off the tensor-core kernels
            calls.append(lambda: L.pmb_qlearner_train_step(C.byref(_dims(SMAC_SHAPES["3m"], E=16)), C.byref(b), C.byref(hp),
                                                           P, P, P, P, P, 1 << 40, P, None))
        for i, call in enumerate(calls):
            assert call() == 1, (kw, i)
            assert what in L.pmb_last_error(), (kw, i, L.pmb_last_error())


def test_host_episode_batch_stores_compact_cells():
    shape = SMAC_SHAPES["3m"]
    B, T = 6, 9
    f = numpy_episode_fields(shape, B, T, seed=2)
    for st, av in ((th.bfloat16, th.uint8), (th.bfloat16, th.bool), (th.float32, th.uint8)):
        scheme, groups = make_scheme(shape)
        scheme["state"]["dtype"], scheme["avail_actions"]["dtype"], scheme["obs"]["dtype"] = st, av, th.bfloat16
        pre = {"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])}
        eb = EpisodeBatch(scheme, groups, B, T, preprocess=pre, device="cpu")
        for t in range(T):
            eb.update({k: th.from_numpy(np.ascontiguousarray(f[k][:, t])) for k in ("obs", "state", "avail_actions",
                                                                                  "actions", "reward", "terminated")},
                      ts=t)
        assert eb["state"].dtype == st and eb["avail_actions"].dtype == av and eb["obs"].dtype == th.bfloat16
        assert th.equal(eb["state"], th.from_numpy(f["state"]).to(st))
        assert th.equal(eb["avail_actions"], th.from_numpy(f["avail_actions"]).to(av))
        assert th.equal(eb["obs"], th.from_numpy(f["obs"]).to(th.bfloat16))
        buf = ReplayBuffer(scheme, groups, 10, T, pre, "cpu")
        buf.insert_episode_batch(eb[1:5])
        for k in ("obs", "state", "avail_actions", "actions"):
            assert buf.data.transition_data[k].dtype == eb[k].dtype
            assert th.equal(buf.data.transition_data[k][:4], eb[k][1:5]), k


# ---- GPU: the learner step -----------------------------------------------------------------------------------------------

def _scheme_dtypes(state=None, avail=None, obs=None):
    return {k: v for k, v in (("state", state), ("avail_actions", avail), ("obs", obs)) if v is not None}


def _rounded_fields(shape, B, T, seed, ragged=True):
    f = numpy_episode_fields(shape, B, T, seed=seed, ragged=ragged)
    for k in ("obs", "state"):
        f[k] = th.from_numpy(f[k]).to(th.bfloat16).float().numpy()
    return f


def _pair(shape, B, T, seed=3, ragged=True, device="cuda", **dtypes):
    """(reference-stored batch, compact-stored batch) holding the same values; dtypes: state / avail / obs."""
    from cuda_utils import to_batch
    f = _rounded_fields(shape, B, T, seed, ragged)
    ref = to_batch(shape, f, device=device)
    cmp = to_batch(shape, f, device=device)
    for k, dt in _scheme_dtypes(**dtypes).items():
        cmp.scheme[k]["dtype"] = dt
        cmp.data.transition_data[k] = ref.data.transition_data[k].to(dt)
    return ref, cmp


def _buffer(shape, n, T, seed, device, pin=False, **dtypes):
    """(reference ReplayBuffer, compact ReplayBuffer) with the same episodes."""
    from cuda_utils import to_batch
    out = []
    for dt in ({}, _scheme_dtypes(**dtypes)):
        scheme, groups = make_scheme(shape)
        for k, v in dt.items():
            scheme[k]["dtype"] = v
        pre = {"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])}
        buf = ReplayBuffer(scheme, groups, n, T, pre, device if device != "pinned" else "cpu", pin_memory=pin)
        buf.insert_episode_batch(to_batch(shape, _rounded_fields(shape, n, T, seed), device=buf.device))
        if device == "pinned":
            buf.pin_memory_()
        buf.zero_copy = True
        out.append(buf)
    for k in ("state", "avail_actions"):
        assert th.equal(out[0].data.transition_data[k].cpu(), out[1].data.transition_data[k].cpu().to(out[0].data.transition_data[k].dtype))
    return out


def _learner(shape, mixer="qmix", precision="bf16", seed=0, **over):
    from cuda_utils import build_learner
    th.manual_seed(seed)
    args = default_args(shape, mixer=mixer, learner_log_interval=0, precision=precision, **over)
    return build_learner(shape, args)[0]


def _state(learner):
    th.cuda.synchronize()
    f = learner._flat
    return dict(p=f["p"].clone(), sq=f["sq"].clone(), target=f["target"].clone(), g=f["g"][:f["p"].numel()].clone(),
                stats=learner.last_stats.clone())


def _assert_equal(a, b):
    for k in a:
        assert th.equal(a[k], b[k]), k


def _train(shape, mixer, batches, precision="bf16", **over):
    """Two steps (the second syncs the target network), or one per batch given."""
    lr = _learner(shape, mixer, precision, **over)
    batches = batches if isinstance(batches, list) else [batches, batches]
    for i, b in enumerate(batches):
        lr.train(b() if callable(b) else b, i, i * lr.args.target_update_interval)
    return _state(lr)


AV8, AVB, SBF = dict(avail=th.uint8), dict(avail=th.bool), dict(state=th.bfloat16)
BOTH = dict(state=th.bfloat16, avail=th.uint8)
ALL3 = dict(state=th.bfloat16, avail=th.bool, obs=th.bfloat16)

# name, mixer, B, T, dtypes: odd A (3m: 9, 2s3z: 11), N * A not a multiple of 16 (27m: 972), S not a multiple of 8 (27m:
# 1170, MMM2: 322), A % 4 != 0 (3m, 2s3z, 27m has A % 16 != 0), full and ragged last row tiles
CASES = [("27m_vs_30m", "qmix", 256, 12, BOTH), ("27m_vs_30m", "qmix", 100, 12, ALL3),
         ("3m", "qmix", 40, 30, BOTH), ("3m", "vdn", 40, 30, AVB), ("2s3z", "qmix", 60, 20, AVB),
         ("2s3z", None, 60, 20, AV8), ("MMM2", "qmix", 50, 16, SBF), ("MMM2", "vdn", 50, 16, ALL3)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mixer,B,T,dtypes", CASES)
def test_train_step_bit_identical(name, mixer, B, T, dtypes):
    shape = SMAC_SHAPES[name]
    ref, cmp = _pair(shape, B, T, **dtypes)
    _assert_equal(_train(shape, mixer, ref), _train(shape, mixer, cmp))


@pytest.mark.gpu
def test_strided_view_and_skipping():
    shape = SMAC_SHAPES["27m_vs_30m"]
    ref, cmp = _pair(shape, 96, 30, seed=5, **BOTH)
    t = 17                                                 # batch[:, :t] keeps the full-T batch stride
    _assert_equal(_train(shape, "qmix", ref[:, :t]), _train(shape, "qmix", cmp[:, :t]))
    _assert_equal(_train(shape, "qmix", ref, skip_padded_steps=True), _train(shape, "qmix", cmp, skip_padded_steps=True))


@pytest.mark.gpu
@pytest.mark.parametrize("mixer,dtypes,over", [("qmix", BOTH, dict(skip_padded_steps=True)), ("vdn", ALL3, {}),
                                               ("qmix", AVB, dict(cuda_graph=True))])
def test_hbm_zero_copy_sample(mixer, dtypes, over):
    shape = SMAC_SHAPES["27m_vs_30m"]
    bufs = _buffer(shape, 120, 24, 4, "cuda", **dtypes)
    out = []
    for buf in bufs:
        np.random.seed(1)
        samples = [buf.sample(90) for _ in range(3)]
        assert all(isinstance(s, IndexedEpisodeBatch) for s in samples)
        out.append(_train(shape, mixer, samples, **over))
    _assert_equal(*out)


@pytest.mark.gpu
@pytest.mark.parametrize("B,over", [(150, {}), (150, dict(skip_padded_steps=True)), (100, {}),
                                    (100, dict(cuda_graph=True))])
def test_pinned_host_zero_copy_sample(B, over):
    # host_stream_chunk = 64: B = 150 streams in chunks gathered from the buffer, B = 100 (or cuda_graph) in one piece
    shape = SMAC_SHAPES["27m_vs_30m"]
    bufs = _buffer(shape, B + 30, 22, 8, "pinned", **ALL3)
    out = []
    for buf in bufs:
        assert buf.pinned
        np.random.seed(2)
        samples = [buf.sample(B) for _ in range(3)]
        samples = [s[:, :s.max_t_filled()] for s in samples]
        out.append(_train(shape, "qmix", samples, host_stream_chunk=64, **over))
    _assert_equal(*out)


@pytest.mark.gpu
def test_host_streamed_batch():
    shape = SMAC_SHAPES["2s3z"]
    ref, cmp = _pair(shape, 150, 20, seed=13, device="cpu", **BOTH)
    _assert_equal(_train(shape, "qmix", [ref], host_stream_chunk=64), _train(shape, "qmix", [cmp], host_stream_chunk=64))


@pytest.mark.gpu
def test_cuda_graph_replay():
    shape = SMAC_SHAPES["3m"]
    pairs = [_pair(shape, 48, 30, seed=s, **BOTH) for s in (1, 2)]
    out = []
    for k in (0, 1):
        lr = _learner(shape, cuda_graph=True)
        for i in range(3):
            for j, p in enumerate(pairs):
                lr.train(p[k], 2 * i + j, (2 * i + j) * 100)
        assert any(isinstance(e, tuple) for e in lr._graphs.values())
        out.append(_state(lr))
    _assert_equal(*out)


@pytest.mark.gpu
def test_no_hidden_conversion(monkeypatch):
    shape = SMAC_SHAPES["27m_vs_30m"]
    _, buf = _buffer(shape, 64, 40, 3, "cuda", **BOTH)
    seen = []
    make_batch = _lib.make_batch
    monkeypatch.setattr(_lib, "make_batch", lambda *a, **k: seen.append(make_batch(*a, **k)) or seen[-1])
    lr = _learner(shape)
    lr.train(buf.sample(48), 0, 0)
    th.cuda.synchronize()
    base = th.cuda.memory_allocated()
    th.cuda.reset_peak_memory_stats()
    lr.train(buf.sample(48), 1, 1)
    th.cuda.synchronize()
    td = buf.data.transition_data
    for pb in seen:
        assert (pb.state, pb.state_dtype) == (td["state"].data_ptr(), BF16)
        assert (pb.avail, pb.avail_dtype) == (td["avail_actions"].data_ptr(), U8)
    assert th.cuda.max_memory_allocated() - base < td["avail_actions"].numel() // 4


@pytest.mark.gpu
@pytest.mark.parametrize("shape,precision,mixer,dtypes", [
    (SMAC_SHAPES["3m"], "fp32", "qmix", ALL3), (SMAC_SHAPES["3m"], "bf16", "qmix_e16", BOTH),
    (WIDE_A, "bf16", "qmix", BOTH), (WIDE_A, "bf16", "vdn", AVB)], ids=["fp32", "qmix_e16", "wide_a_qmix", "wide_a_vdn"])
def test_converting_paths_match(shape, precision, mixer, dtypes):
    ref, cmp = _pair(shape, 20, 16, seed=4, **dtypes)
    over = dict(mixing_embed_dim=16) if mixer == "qmix_e16" else {}
    mixer = "qmix" if mixer == "qmix_e16" else mixer
    _assert_equal(_train(shape, mixer, ref, precision, **over), _train(shape, mixer, cmp, precision, **over))


@pytest.mark.gpu
def test_coma_converts():
    from test_coma_gpu import COMA_KW, build_coma
    shape = SMAC_SHAPES["3m"]
    out = []
    for batch in _pair(shape, 8, 16, seed=6, **ALL3):
        th.manual_seed(0)
        lr, _ = build_coma(shape, default_args(shape, mixer=None, **COMA_KW))
        lr.train(batch, 0, 0)
        lr.train(batch, 1, 0)
        th.cuda.synchronize()
        out.append((lr._flat["ap"].clone(), lr._flat["cp"].clone(), lr.last_stats.clone()))
    for x, y in zip(*out):
        assert th.equal(x, y)


@pytest.mark.gpu
def test_device_buffer_moves_compact_cells():
    # pmb_batch_update (EpisodeBatch.update on the device) and pmb_gather_episodes (a sample without zero_copy)
    shape = SMAC_SHAPES["27m_vs_30m"]
    f = _rounded_fields(shape, 12, 9, seed=7)
    host, dev = _buffer(shape, 12, 9, 7, "cpu", **ALL3)[1], _buffer(shape, 12, 9, 7, "cuda", **ALL3)[1]
    for k in ("obs", "state", "avail_actions"):
        assert th.equal(dev.data.transition_data[k].cpu(), host.data.transition_data[k]), k
    ids = np.array([5, 0, 11, 3, 3, 8, 1])
    s = dev[ids]
    for k in ("obs", "state", "avail_actions"):
        assert th.equal(s[k].cpu(), host.data.transition_data[k][ids]), k
    assert th.equal(host["avail_actions"], th.from_numpy(f["avail_actions"]).to(th.bool))


# ---- GPU: the rollout ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("device", ["cuda", "cpu"])
@pytest.mark.parametrize("name,B,dtypes", [("27m_vs_30m", 300, AV8), ("3m", 700, AVB), ("2s3z", 257, ALL3)])
def test_select_actions_bit_identical(name, B, dtypes, device):
    shape = SMAC_SHAPES[name]
    N, A = shape.n_agents, shape.n_actions
    pair = _pair(shape, B, 6, seed=8, ragged=False, device=device, **dtypes)
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
        for t in range(3, 6):                                           # Philox draws
            q, act = mac._run_step(batch, t, epsilon=0.5, seed=11, offset=t, want_actions=True, want_q=True)
            res += [q.clone(), act.clone(), mac.hidden_states.clone()]
        th.cuda.synchronize()
        out.append(res)
    for i, (x, y) in enumerate(zip(*out)):
        assert th.equal(x, y), i
