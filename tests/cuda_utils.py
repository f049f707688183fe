"""Helpers for the -m gpu parity tests: build the CUDA-backed learner / MAC from a golden
fixture or from oracle parameters, and wrap numpy episode fields in an EpisodeBatch."""
from types import SimpleNamespace

import numpy as np
import torch as th

from pymarl_b200 import le_REGISTRY, mac_REGISTRY, EpisodeBatch
from pymarl_b200.components.transforms import OneHot
from pymarl_b200.synthetic import make_scheme, get_shape


class Logger:
    def __init__(self):
        self.stats, self.infos = {}, []
        self.console_logger = SimpleNamespace(info=lambda msg, *a: self.infos.append(msg))

    def log_stat(self, key, value, t):
        self.stats.setdefault(key, []).append((t, float(value)))


def to_batch(shape, fields, device="cuda"):
    shape = get_shape(shape)
    B, T = fields["obs"].shape[:2]
    scheme, groups = make_scheme(shape)
    preprocess = {"actions": ("actions_onehot", [OneHot(out_dim=shape.n_actions)])}
    batch = EpisodeBatch(scheme, groups, B, T, preprocess=preprocess, device=device)
    for k, v in fields.items():
        t = th.from_numpy(np.ascontiguousarray(v)).to(device)
        assert batch.data.transition_data[k].shape == t.shape, (k, t.shape)
        assert batch.data.transition_data[k].dtype == t.dtype, (k, t.dtype)
        batch.data.transition_data[k] = t
    return batch


def build_learner(shape, args, agent=None, target_agent=None, mixer=None, target_mixer=None):
    """CUDA learner with the given numpy parameter dicts loaded (reference state_dict names)."""
    shape = get_shape(shape)
    scheme, groups = make_scheme(shape)
    scheme["actions_onehot"] = {"vshape": (shape.n_actions,), "dtype": th.float32, "group": "agents"}
    args.device = "cuda"
    args.use_cuda = True
    mac = mac_REGISTRY[args.mac](scheme, groups, args)
    logger = Logger()
    learner = le_REGISTRY[args.learner](mac, scheme, logger, args)
    learner.cuda()
    def load(module, params):
        if params:
            module.load_state_dict({k: th.from_numpy(np.asarray(v, dtype=np.float32)) for k, v in params.items()})
    load(learner.mac.agent, agent)
    load(learner.target_mac.agent, target_agent if target_agent is not None else agent)
    if args.mixer == "qmix":
        load(learner.mixer, mixer)
        load(learner.target_mixer, target_mixer if target_mixer is not None else mixer)
    return learner, logger


def learner_from_golden(g, **over):
    return build_learner(g.shape, g.args(**over), g.group("init/agent"), g.group("init/target_agent"),
                         g.group("init/mixer"), g.group("init/target_mixer"))


def state_np(module):
    return {k: v.detach().cpu().numpy() for k, v in module.state_dict().items()}


def _decode_images(u8, lead):
    """bf16 tile images ([*lead][16 KB]: row r at byte r*128, 16-byte chunk j at (j ^ (r & 7)) << 4) -> float32 [*lead, 128, 64]."""
    x = u8.view(th.bfloat16).view(*lead, 128, 8, 8)
    r = th.arange(128, device=u8.device)[:, None]
    j = th.arange(8, device=u8.device)[None, :]
    idx = (j ^ (r & 7))[..., None].expand(128, 8, 8)
    return th.gather(x, len(lead) + 1, idx.expand_as(x).contiguous()).reshape(*lead, 128, 64).float()


def _ws_bytes(learner, dims, name, nbytes):
    import ctypes as C
    from pymarl_b200 import _lib
    v = _lib.WsViews()
    _lib.check(_lib.lib().pmb_learner_workspace_views(C.byref(dims), _lib.ptr(learner._workspace), learner._workspace.numel(),
                                                      C.byref(v)), "workspace_views")
    off = getattr(v, name) - learner._workspace.data_ptr()
    return learner._workspace[off:off + nbytes]


ALL_DECISIONS = ("relu_mask", "cur_max", "hypernet")


def gpu_decisions(shape, args, olr, fields, which=ALL_DECISIONS):
    """Run the GPU step FORWARD ONLY (pmb_hparams.keep_q = 3) and read its discontinuous decisions out of the workspace,
    in the form OracleQLearner.train(decisions=...) takes.  `which` names the decisions the step takes on bf16 operands:
      relu_mask  the fc1 ReLU mask [T, B*N, 64] (tensor-core agent: H = 64, A <= 64)
      cur_max    the double-Q arg-max [B, T-1, N] over the step's own online Q
      hypernet   sign_w1, sign_wf, v0_mask from the hypernet output images (tensor-core mixer: QMIX, E = 32)"""
    import copy
    a = copy.copy(args)
    a.keep_q = 3
    learner, _ = build_learner(shape, a, olr.agent, olr.target_agent, olr.mixer_p, olr.target_mixer_p)
    batch = to_batch(shape, fields)
    learner.train(batch, 0, 0)
    th.cuda.synchronize()
    d = learner._last_dims
    B, T, N, A = d.B, d.T, d.N, d.A
    R, n_tiles = B * N, -(-B * N // 128)
    dec = {}
    if "relu_mask" in which:
        assert d.H == 64 and A <= 64, "the ReLU mask image exists where the tensor-core agent runs"
        # ReLU decisions of the online fc1: bit mask [T][n_tiles][2][128] words, bit j of (half, row) = column 32*half + j
        words = _ws_bytes(learner, d, "relu_mask", T * n_tiles * 2 * 128 * 4).view(th.int32).view(T, n_tiles, 2, 128)
        bits = (words[..., None] >> th.arange(32, device=words.device, dtype=th.int32)) & 1          # [T, tiles, 2, 128, 32]
        dec["relu_mask"] = bits.permute(0, 1, 3, 2, 4).reshape(T, n_tiles * 128, 64)[:, :R].bool().cpu().numpy()
    if "cur_max" in which:
        # double-Q arg-max decisions from the step's own Q tensor (keep_q bit 1)
        ws = learner.workspace_views(d)
        q = ws["q_on"].view(T, B, N, A).permute(1, 0, 2, 3)
        avail = batch["avail_actions"]
        dec["cur_max"] = q.masked_fill(avail == 0, -9999999.0)[:, 1:].argmax(3).cpu().numpy()
    if "hypernet" in which:
        E = d.E
        assert args.mixer == "qmix" and E == 32, "the hypernet output images exist where the tensor-core mixer runs"
        n_cblk, rt = (N + 3 + 1) // 2, -(-B * T // 128)
        raw = _decode_images(_ws_bytes(learner, d, "raw_on", rt * n_cblk * 16384), (rt, n_cblk))   # [rt, cblk, 128, 64]
        raw = raw.permute(0, 2, 1, 3).reshape(rt * 128, n_cblk * 64)[:B * T].view(B, T, -1)[:, :T - 1].reshape(B * (T - 1), -1)
        raw = raw.cpu().numpy().astype(np.float64)
        dec["sign_w1"] = np.sign(raw[:, :N * E])
        dec["sign_wf"] = np.sign(raw[:, (N + 1) * E:(N + 2) * E])
        dec["v0_mask"] = raw[:, (N + 2) * E:(N + 3) * E] > 0
    return dec
