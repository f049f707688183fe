"""Zero-copy sampling from a replay buffer in pinned host memory (pmb_gather_episode_steps).

Host-only: the ReplayBuffer signature, the learner's plan (chunked / one piece / not at all), the COMA rejection, the host
computation of the trimmed length F_j and the C struct.  GPU: the gather kernel bit-exact against ``buf[k][ids][:, :steps]``
for every dtype the learner reads, trim mode, the rejections; the learner step on a pinned zero-copy sample bit-identical
to the same ids sampled as a gathered host batch; no host gather during train; writes after train do not race its reads.
"""
import ctypes as C
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch as th

from pymarl_b200 import _lib
from pymarl_b200.components.episode_buffer import EpisodeBatch, IndexedEpisodeBatch, ReplayBuffer
from pymarl_b200.components.transforms import OneHot
from pymarl_b200.learners.coma_learner import COMALearner
from pymarl_b200.learners.q_learner import QLearner
from pymarl_b200.synthetic import SMAC_SHAPES, default_args, make_scheme, numpy_episode_fields

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def copy_steps(filled, ids, steps):
    """F_j = min(steps, l_j + 2), l_j = the last t < steps with filled[id, t] != 0; 0 for an empty episode."""
    out = []
    for i in ids:
        nz = np.flatnonzero(np.asarray(filled[i]).reshape(-1)[:steps])
        out.append(0 if nz.size == 0 else min(steps, int(nz[-1]) + 2))
    return np.asarray(out, dtype=np.int64)


def _host_buffer(shape, n, T, pin=False, seed=0, obs_dtype=None, ragged=True):
    scheme, groups = make_scheme(shape)
    if obs_dtype is not None:
        scheme["obs"]["dtype"] = obs_dtype
    pre = {"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])}
    buf = ReplayBuffer(scheme, groups, n, T, pre, "cpu", pin_memory=pin)
    if n:
        from cuda_utils import to_batch
        buf.insert_episode_batch(to_batch(shape, numpy_episode_fields(shape, n, T, seed=seed, ragged=ragged), device="cpu"))
    return buf


def _indexed(n, T=10):
    fake = SimpleNamespace(scheme={}, groups={}, device="cpu", max_seq_length=T)
    ids = th.arange(n, dtype=th.int64)
    return IndexedEpisodeBatch(fake, ids, host_ids=ids)


# ---- host-only -------------------------------------------------------------------------------------------------------

def test_reference_signature_and_unpinned_fallback():
    shape = SMAC_SHAPES["3m"]
    buf = _host_buffer(shape, 12, 6)
    assert not buf.pinned and buf.device_reads is None
    buf.zero_copy = True                                   # an unpinned host buffer keeps returning the gathered copy
    np.random.seed(0)
    s = buf.sample(5)
    assert isinstance(s, EpisodeBatch) and s.batch_size == 5 and not s["obs"].is_cuda
    with pytest.raises(ValueError):
        ReplayBuffer(*make_scheme(shape), 4, 6, None, "cuda", pin_memory=True)


def test_stream_plan():
    lr = QLearner.__new__(QLearner)
    lr.args = default_args(SMAC_SHAPES["3m"], host_stream_chunk=64)
    assert lr._host_stream_plan(_indexed(150), False) == (0, 150, 64)      # chunked
    assert lr._host_stream_plan(_indexed(127), False) is None              # under two chunks: one piece
    assert lr._host_stream_plan(_indexed(150), True) is None               # data parallel: one piece
    lr.args.cuda_graph = True
    assert lr._host_stream_plan(_indexed(150), False) is None              # CUDA graph: one piece
    lr.args.cuda_graph = False
    dev_sample = _indexed(150)
    dev_sample.host_ids = None                                             # a sample of a buffer in HBM: read in place
    assert lr._host_stream_plan(dev_sample, False) is None
    gathered = _host_buffer(SMAC_SHAPES["3m"], 150, 6)[:, :6]             # today's gathered host batch: as before
    assert lr._host_stream_plan(gathered, False) == (0, 150, 64)


def test_coma_rejects_host_sample():
    with pytest.raises(TypeError, match="zero_copy"):
        COMALearner.__new__(COMALearner).train(_indexed(4), 0, 0)


def test_copy_steps_reference():
    filled = np.zeros((5, 8), dtype=np.int64)
    filled[0, :8] = 1               # full length: all steps
    filled[1, :3] = 1               # l = 2 -> 4
    filled[2, [0, 1, 4]] = 1        # a hole does not shorten the episode: l = 4 -> 6
    filled[4, :7] = 1               # l = 6 -> min(steps, 8)
    assert copy_steps(filled, [0, 1, 2, 3, 4], 8).tolist() == [8, 4, 6, 0, 8]
    assert copy_steps(filled, [0, 1, 2, 3, 4], 5).tolist() == [5, 4, 5, 0, 5]


def test_step_field_struct_matches_header():
    assert C.sizeof(_lib.StepField) == 32
    hdr = open(os.path.join(REPO, "include", "pymarl_b200.h")).read()
    body = re.search(r"typedef struct pmb_step_field \{(.*?)\} pmb_step_field;", hdr, re.S).group(1)
    assert re.findall(r"(\w+);", body) == [k for k, _ in _lib.StepField._fields_]


# ---- GPU: the kernel -------------------------------------------------------------------------------------------------

FIELDS = {"f32": (th.float32, (37,)), "bf16_odd": (th.bfloat16, (3, 285)), "i64": (th.int64, (3, 1)),
          "i32": (th.int32, (3, 11)), "u8": (th.uint8, (1,))}


def _random(shape, dtype, gen):
    if dtype.is_floating_point:
        return th.randn(shape, generator=gen).to(dtype)
    return th.randint(0, 120, shape, generator=gen).to(dtype)


def _source(t, where):
    if where == "pinned":
        return _lib.host_empty(t.shape, t.dtype).copy_(t)
    return t.cuda()


def _rows(n, shape, dtype, extra_bytes, fill):
    """Destination rows with `extra_bytes` beyond the 16-byte rounding, the whole storage preset to `fill`."""
    es = th.empty((), dtype=dtype).element_size()
    inner = int(np.prod(shape))
    row = (-(-inner * es // 16) * 16 + extra_bytes) // es
    base = th.full((n * row * es,), fill, dtype=th.uint8, device="cuda")
    out = base.view(dtype).as_strided((n,) + tuple(shape), (row,) + th.empty(tuple(shape), device="meta").stride())
    return out, base.view(n, row * es)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned"])
@pytest.mark.parametrize("name", list(FIELDS))
def test_gather_bit_exact(name, where):
    dtype, cell = FIELDS[name]
    n_src, T_src, steps, n = 50, 13, 9, 40
    gen = th.Generator().manual_seed(1)
    ref = _random((n_src, T_src) + cell, dtype, gen)
    src = _source(ref, where)
    ids = th.randint(0, n_src, (n,), generator=gen)
    out, raw = _rows(n, (steps,) + cell, dtype, 32, 0xAB)
    _lib.gather_episode_steps({"x": src}, ids.cuda(), steps, {"x": out})
    th.cuda.synchronize()
    assert th.equal(out.cpu(), ref[ids][:, :steps])
    run = steps * int(np.prod(cell)) * ref.element_size()
    padded = -(-run // 16) * 16
    assert bool((raw[:, run:padded] == 0).all())            # the last word's bytes past the run are written as zero
    assert bool((raw[:, padded:] == 0xAB).all())            # the rest of the row stride is untouched


@pytest.mark.gpu
def test_gather_many_ids_several_fields():
    n_src, T_src, steps, n = 1000, 6, 4, 70000              # more ids than a grid dimension holds
    gen = th.Generator().manual_seed(2)
    refs = {k: _random((n_src, T_src) + c, d, gen) for k, (d, c) in FIELDS.items()}
    src = {k: _source(v, "pinned" if i % 2 else "device") for i, (k, v) in enumerate(refs.items())}
    ids = th.randint(0, n_src, (n,), generator=gen)
    out = {k: _lib.episode_rows(n, (steps,) + tuple(v.shape[2:]), v.dtype, "cuda") for k, v in refs.items()}
    _lib.gather_episode_steps(src, ids.cuda(), steps, out)
    th.cuda.synchronize()
    for k, v in refs.items():
        assert th.equal(out[k].cpu(), v[ids][:, :steps]), k


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned"])
def test_gather_trimmed(where):
    shape = SMAC_SHAPES["2s3z"]
    n_src, T_src, steps = 60, 24, 20
    f = numpy_episode_fields(shape, n_src, T_src, seed=5, ragged=True)
    f["filled"][7] = 0                                      # empty episode
    f["filled"][9, 3:6] = 0                                 # a hole
    gen = th.Generator().manual_seed(3)
    refs = {k: _random(th.from_numpy(v).shape, th.from_numpy(v).dtype, gen) for k, v in f.items() if k != "filled"}
    refs["obs"] = refs["obs"].to(th.bfloat16)
    refs["filled"] = th.from_numpy(f["filled"])
    src = {k: _source(v, where) for k, v in refs.items()}
    ids = th.as_tensor(np.r_[7, 9, np.random.default_rng(6).integers(0, n_src, 70)])
    out = {k: _rows(ids.numel(), (steps,) + tuple(v.shape[2:]), v.dtype, 0, 0x77)[0] for k, v in refs.items()}
    _lib.gather_episode_steps({k: src[k] for k in refs}, ids.cuda(), steps, out, filled=src["filled"])
    th.cuda.synchronize()
    F = copy_steps(f["filled"], ids.tolist(), steps)
    assert F[0] == 0 and F[1] == min(steps, int(np.flatnonzero(f["filled"][9, :steps, 0])[-1]) + 2)
    for k, v in refs.items():
        got, want = out[k].cpu(), v[ids][:, :steps]
        for j, Fj in enumerate(F):
            assert th.equal(got[j, :Fj], want[j, :Fj]), (k, j)
            assert bool((got[j, Fj:] == 0).all()), (k, j)


@pytest.mark.gpu
def test_gather_rejects_pageable_and_null():
    src = th.zeros(4, 5, 3)                                 # pageable host memory
    out = _lib.episode_rows(2, (5, 3), th.float32, "cuda")
    ids = th.tensor([0, 3], device="cuda")
    with pytest.raises(_lib.PmbError, match="pageable"):
        _lib.gather_episode_steps({"x": src}, ids, 5, {"x": out})
    arr = (_lib.StepField * 1)(_lib.StepField(None, out.data_ptr(), 12, out.stride(0) * 4))
    assert _lib.lib().pmb_gather_episode_steps(arr, 1, _lib.ptr(ids), 2, 4, 5, 5, None, 0, None) == 1
    assert b"NULL" in _lib.lib().pmb_last_error()
    dev = th.randn(4, 5, 3, device="cuda")                  # the library still works afterwards
    _lib.gather_episode_steps({"x": dev}, ids, 5, {"x": out})
    assert th.equal(out, dev[ids])


# ---- GPU: the learner ------------------------------------------------------------------------------------------------

def _learner(shape, mixer, precision, **over):
    from cuda_utils import build_learner
    th.manual_seed(0)
    args = default_args(shape, mixer=mixer, learner_log_interval=0, precision=precision, **over)
    return build_learner(shape, args)[0]


def _state(learner):
    th.cuda.synchronize()
    f = learner._flat
    return dict(p=f["p"].clone(), sq=f["sq"].clone(), target=f["target"].clone(), g=f["g"][:f["p"].numel()].clone(),
                stats=learner.last_stats.clone())


def _sample(buf, B, seed):
    np.random.seed(seed)
    s = buf.sample(B)
    return s[:, :s.max_t_filled()]


def _run(shape, mixer, precision, buf, B, steps=2, **over):
    lr = _learner(shape, mixer, precision, **over)
    for i in range(steps):
        lr.train(_sample(buf, B, 10 + i), i, i)
    return _state(lr)


# name, mixer, precision, obs dtype, B, learner args (chunk 64: B >= 128 streams in chunks, smaller B in one piece)
LEARNER_CASES = [
    ("27m_vs_30m", "qmix", "bf16", th.bfloat16, 150, {}),
    ("27m_vs_30m", "qmix", "bf16", th.bfloat16, 150, dict(skip_padded_steps=True)),
    ("MMM2", "vdn", "fp32", None, 140, {}),
    ("2s3z", "qmix", "bf16", None, 100, {}),
    ("3m", "qmix", "fp32", None, 90, dict(skip_padded_steps=True)),
    ("2s3z", "vdn", "bf16", th.bfloat16, 150, dict(cuda_graph=True)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mixer,precision,obs_dtype,B,over", LEARNER_CASES)
def test_learner_matches_gathered_host_batch(name, mixer, precision, obs_dtype, B, over):
    shape = SMAC_SHAPES[name]
    T = 22
    over = dict(host_stream_chunk=64, **over)
    plain = _host_buffer(shape, B + 30, T, seed=8, obs_dtype=obs_dtype)
    pinned = _host_buffer(shape, B + 30, T, seed=8, obs_dtype=obs_dtype).pin_memory_()
    pinned.zero_copy = True
    assert isinstance(_sample(pinned, B, 0), IndexedEpisodeBatch)
    steps = 3 if over.get("cuda_graph") else 2
    a = _run(shape, mixer, precision, plain, B, steps, **over)
    b = _run(shape, mixer, precision, pinned, B, steps, **over)
    for k in a:
        assert th.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_materialise_one_field():
    shape = SMAC_SHAPES["3m"]
    plain = _host_buffer(shape, 40, 12, seed=2)
    pinned = _host_buffer(shape, 40, 12, seed=2, pin=True)
    pinned.zero_copy = True
    a, b = _sample(plain, 30, 1), _sample(pinned, 30, 1)
    assert b.to("cuda") is b
    for k in ("obs", "avail_actions", "filled"):
        assert th.equal(a[k], b[k].cpu()), k


@pytest.mark.gpu
def test_no_hidden_host_gather(monkeypatch):
    shape = SMAC_SHAPES["27m_vs_30m"]
    pinned = _host_buffer(shape, 160, 16, seed=3, pin=True)
    pinned.zero_copy = True
    samples = [_sample(pinned, 150, 1), _sample(pinned, 100, 2)]      # chunked, one piece
    orig = EpisodeBatch.__getitem__

    def guarded(self, item):
        if not isinstance(item, (str, tuple)) or (isinstance(item, tuple) and not isinstance(item[0], (str, slice))):
            raise AssertionError("host gather of the replay buffer during train")
        return orig(self, item)

    monkeypatch.setattr(EpisodeBatch, "__getitem__", guarded)
    lr = _learner(shape, "qmix", "bf16", host_stream_chunk=64)
    for i, s in enumerate(samples):
        lr.train(s, i, i)
    th.cuda.synchronize()


@pytest.mark.gpu
def test_insert_after_train_does_not_race():
    shape = SMAC_SHAPES["27m_vs_30m"]
    B, T = 256, 30
    out = []
    for overwrite in (False, True):
        buf = _host_buffer(shape, B, T, seed=4, pin=True)
        buf.zero_copy = True
        fresh = _host_buffer(shape, B, T, seed=5)
        lr = _learner(shape, "qmix", "bf16", host_stream_chunk=64)
        np.random.seed(3)
        s = buf.sample(B - 8)
        lr.train(s, 0, 0)
        if overwrite:
            buf.insert_episode_batch(fresh[:, :T])            # every sampled episode, right after train returns
        out.append(_state(lr))
    for k in out[0]:
        assert th.equal(out[0][k], out[1][k]), k
