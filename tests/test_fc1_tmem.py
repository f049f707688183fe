"""The learner's streaming fc1 with the weights in tensor memory (fc1_stream_ts_kernel, transposed MMA with the A operand
read from TMEM) against fc1_stream_kernel (weights in shared memory), selected per call with PMB_FC1_TS.

On the same seeded batch and parameters (forward-only step):
- the obs tile images are bit-identical (the same converters write them);
- the x tile images of both nets differ at most by one bf16 ulp (the MMA sums with M and N swapped);
- ReLU mask bits differ only where x differs;
- x of the new kernel matches relu(bf16(obs) . bf16(W)^T + last-action column) computed in fp32 by torch.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch as th

from pymarl_b200.synthetic import SMAC_SHAPES, SmacShape, default_args, numpy_episode_fields

pytestmark = pytest.mark.gpu


def _decode_images(u8, lead):
    """bf16 tile images ([*lead][16 KB]: row r at byte r*128, 16-byte chunk j at (j ^ (r & 7)) << 4) -> float32 [*lead, 128, 64]."""
    x = u8.view(th.bfloat16).view(*lead, 128, 8, 8)
    r = th.arange(128, device=u8.device)[:, None]
    j = th.arange(8, device=u8.device)[None, :]
    idx = (j ^ (r & 7))[..., None].expand(128, 8, 8)
    return th.gather(x, len(lead) + 1, idx.expand_as(x).contiguous()).reshape(*lead, 128, 64).float()


def _ws(learner, dims, name, nbytes):
    from pymarl_b200 import _lib
    v = _lib.WsViews()
    _lib.check(_lib.lib().pmb_learner_workspace_views(C.byref(dims), _lib.ptr(learner._workspace), learner._workspace.numel(),
                                                      C.byref(v)), "workspace_views")
    off = getattr(v, name) - learner._workspace.data_ptr()
    return learner._workspace[off:off + nbytes]


def _fc1_outputs(learner, batch, ts):
    old = os.environ.get("PMB_FC1_TS")
    os.environ["PMB_FC1_TS"] = "1" if ts else "0"
    try:
        d = learner._last_dims
        if d is not None:                      # sentinel bytes: whatever the kernel under test does not write shows up
            for name, nb in _sizes(d).items():
                _ws(learner, d, name, nb).fill_(0xFF if name != "relu_mask" else 0)
        learner.train(batch, 0, 0)
        th.cuda.synchronize()
    finally:
        if old is None:
            del os.environ["PMB_FC1_TS"]
        else:
            os.environ["PMB_FC1_TS"] = old
    d = learner._last_dims
    return {name: _ws(learner, d, name, nb).clone() for name, nb in _sizes(d).items()}


def _sizes(d):
    n_tiles = -(-d.B * d.N // 128)
    nc = -(-d.O // 64)
    return {"x_on": d.T * n_tiles * 16384, "x_tg": d.T * n_tiles * 16384, "obs_img": d.T * n_tiles * nc * 16384,
            "relu_mask": d.T * n_tiles * 2 * 128 * 4}


@pytest.mark.parametrize("shape,B,T", [("27m_vs_30m", 256, 12),                                # 54 full row tiles
                                       ("27m_vs_30m", 100, 9),                                 # R = 2700: ragged last tile
                                       (SmacShape("nofold", 30, 290, 64, 33, 6), 20, 6)])      # agent id not in the K padding
def test_fc1_tmem_kernel_matches_smem_kernel(shape, B, T):
    from cuda_utils import build_learner, to_batch
    shape = SMAC_SHAPES[shape] if isinstance(shape, str) else shape
    args = default_args(shape, mixer="qmix", learner_log_interval=0, precision="bf16", keep_q=3)
    learner, _ = build_learner(shape, args)
    fields = numpy_episode_fields(shape, B, T, seed=17, ragged=True)
    batch = to_batch(shape, fields)
    learner.train(batch, 0, 0)                 # allocates the workspace
    ref = _fc1_outputs(learner, batch, ts=False)
    new = _fc1_outputs(learner, batch, ts=True)
    d = learner._last_dims
    N, O, R = d.N, d.O, d.B * d.N
    n_tiles = -(-R // 128)

    assert th.equal(new["obs_img"], ref["obs_img"])
    xs = {}
    n_ulp1 = 0
    for k in ("x_on", "x_tg"):
        a = new[k].view(th.int16).view(T, n_tiles * 128 * 64)
        b = ref[k].view(th.int16).view(T, n_tiles * 128 * 64)
        diff = (a.int() - b.int()).abs()       # bf16 of equal sign: one ulp = 1 in the bit pattern (values are >= 0)
        assert int(diff.max()) <= 1, k
        n_ulp1 += int((diff == 1).sum())
        xs[k] = (_decode_images(new[k], (T, n_tiles)).reshape(T, n_tiles * 128, 64)[:, :R],
                 _decode_images(ref[k], (T, n_tiles)).reshape(T, n_tiles * 128, 64)[:, :R])
    print("x elements one bf16 ulp apart:", n_ulp1, "of", 2 * T * R * 64)

    bits = []
    for m in (new["relu_mask"], ref["relu_mask"]):
        w = m.view(th.int32).view(T, n_tiles, 2, 128)
        bb = (w[..., None] >> th.arange(32, device=w.device, dtype=th.int32)) & 1
        bits.append(bb.permute(0, 1, 3, 2, 4).reshape(T, n_tiles * 128, 64)[:, :R].bool())
    x_new, x_ref = xs["x_on"]
    flip = bits[0] != bits[1]
    assert not (flip & (x_new == x_ref)).any()
    assert th.equal(bits[0], x_new > 0)

    # the TMEM-A GEMM against torch: bf16 operands, fp32 sums
    w = learner.mac.agent.fc1.weight.detach()
    bias = learner.mac.agent.fc1.bias.detach()
    bf = lambda t: t.to(th.bfloat16).float()
    obs = th.as_tensor(fields["obs"], device="cuda").float().permute(1, 0, 2, 3).reshape(T, R, O)
    pre = bf(obs) @ bf(w[:, :O]).t()
    A = d.A
    if d.N + 1 <= -(-O // 64) * 64 - O:        # agent id and bias folded into the K padding (bf16)
        pre = pre + bf(w[:, O + A:O + A + N]).t().repeat(B, 1)[None] + bf(bias)[None, None]
    else:
        pre = pre + (w[:, O + A:O + A + N].t()[None] + bias[None, None]).repeat(1, B, 1)
    act = th.as_tensor(fields["actions"], device="cuda").long()[..., 0]                  # [B, T, N]
    filled = th.as_tensor(fields["filled"], device="cuda").long()[..., 0]                # [B, T]
    prev = th.full((B, T, N), -1, dtype=th.long, device="cuda")
    prev[:, 1:] = th.where(filled[:, :-1, None] != 0, act[:, :-1], th.full_like(act[:, :-1], -1))
    prev = prev.permute(1, 0, 2).reshape(T, R)
    tab = bf(w[:, O:O + A]).t()                                                          # [A, 64]
    pre = pre + th.where(prev[..., None] >= 0, tab[prev.clamp(min=0)], th.zeros_like(pre))
    x_torch = th.relu(pre)
    err = (x_new - x_torch).abs() / (x_torch.abs() + 1e-2)
    assert float(err.max()) < 2e-2, float(err.max())
