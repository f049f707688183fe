"""ctypes binding of libpymarl_b200.so (C ABI in include/pymarl_b200.h).

There is NO CPU fallback: if the shared library is missing or a call fails, the caller gets
an exception.  The library is built in-tree by ``pymarl_b200.build.build()`` (nvcc, sm_100a).
"""
import ctypes as C
import os
import weakref

import torch as th

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpymarl_b200.so")

MIXER_IDS = {None: 0, "vdn": 1, "qmix": 2}
PREC_IDS = {"fp32": 0, "bf16": 1}
P_COUNT = 18
PARAM_ORDER = [  # enum pmb_param_id
    "agent.fc1.weight", "agent.fc1.bias", "agent.rnn.weight_ih", "agent.rnn.weight_hh",
    "agent.rnn.bias_ih", "agent.rnn.bias_hh", "agent.fc2.weight", "agent.fc2.bias",
    "mixer.hyper_w_1.weight", "mixer.hyper_w_final.weight", "mixer.hyper_b_1.weight", "mixer.V.0.weight",
    "mixer.hyper_w_1.bias", "mixer.hyper_w_final.bias", "mixer.hyper_b_1.bias", "mixer.V.0.bias",
    "mixer.V.2.weight", "mixer.V.2.bias",
]
STAT_IDS = dict(mask_sum=0, td2_sum=1, tdabs_sum=2, qtaken_sum=3, target_sum=4, grad_norm=5, loss=6, clip_coef=7)
STATS_LEN = 16
OBS_DTYPE_IDS = {th.float32: 0, th.bfloat16: 1}           # enum pmb_dtype
DTYPE_F32, DTYPE_BF16, DTYPE_U8 = 0, 1, 2                 # enum pmb_dtype (0 is the reference type: f32, i32 avail)
ENTRY_TRAIN_STEP, ENTRY_SELECT_ACTIONS = 0, 1             # enum pmb_entry
FIELD_IDS = {"obs": 0, "state": 1, "avail_actions": 2}    # enum pmb_field
DP_TAIL_FLOATS = 16          # PMB_DP_TAIL_FLOATS


class Dims(C.Structure):
    _fields_ = [(k, C.c_int32) for k in
                ("B", "T", "N", "O", "S", "A", "H", "E", "obs_last_action", "obs_agent_id", "mixer",
                 "double_q", "precision", "reserved")]


class Batch(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("obs_sb", C.c_int64),
                ("state", C.c_void_p), ("state_sb", C.c_int64),
                ("actions", C.c_void_p), ("actions_sb", C.c_int64),
                ("avail", C.c_void_p), ("avail_sb", C.c_int64),
                ("reward", C.c_void_p), ("reward_sb", C.c_int64),
                ("terminated", C.c_void_p), ("terminated_sb", C.c_int64),
                ("filled", C.c_void_p), ("filled_sb", C.c_int64),
                ("ep_index", C.c_void_p),
                ("obs_dtype", C.c_int32)]          # enum pmb_dtype


class _BatchTail(C.Structure):
    """pmb_batch from obs_dtype on: state_dtype and avail_dtype are int16 in the tail padding of Batch (sizeof stays 128)."""
    _fields_ = [("obs_dtype", C.c_int32), ("state_dtype", C.c_int16), ("avail_dtype", C.c_int16)]


def _tail_field(name):
    def get(self):
        return getattr(_BatchTail.from_buffer(self, Batch.obs_dtype.offset), name)

    def put(self, value):
        setattr(_BatchTail.from_buffer(self, Batch.obs_dtype.offset), name, value)
    return property(get, put)


Batch.state_dtype = _tail_field("state_dtype")           # enum pmb_dtype (0: f32)
Batch.avail_dtype = _tail_field("avail_dtype")           # enum pmb_dtype (0: i32)


class Layout(C.Structure):
    _fields_ = [("offset", C.c_int64 * P_COUNT), ("numel", C.c_int64 * P_COUNT),
                ("n_agent", C.c_int64), ("n_total", C.c_int64)]


class HParams(C.Structure):
    _fields_ = [("gamma", C.c_float), ("lr", C.c_float), ("alpha", C.c_float), ("eps", C.c_float),
                ("grad_norm_clip", C.c_float), ("do_target_sync", C.c_int32), ("skip_update", C.c_int32),
                ("keep_q", C.c_int32)]


class ComaHParams(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("gamma", "td_lambda", "lr", "critic_lr", "alpha", "eps", "grad_norm_clip", "epsilon")]


class GatherField(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("bytes_per_episode", C.c_int64)]


class StepField(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("cell_bytes", C.c_int64), ("dst_stride_bytes", C.c_int64)]


class UpdateField(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("cell_bytes", C.c_int64), ("dst_batch_stride_bytes", C.c_int64),
                ("dst_time_stride_bytes", C.c_int64), ("onehot_dim", C.c_int32), ("reserved", C.c_int32)]


class WsViews(C.Structure):
    _names = ("x_on", "x_tg", "h_stash", "gates", "q_on", "q_tg", "chosen", "tmax", "raw_on", "raw_tg",
              "q_tot", "t_tot", "g", "d_chosen", "scratch")
    _fields_ = [(k, C.c_void_p) for k in _names] + [("scratch_bytes", C.c_int64), ("obs_img", C.c_void_p),
                                                        ("state_img", C.c_void_p), ("h_tg", C.c_void_p),
                                                        ("relu_mask", C.c_void_p),
                                                        # padded-step skipping (NULL where pmb_dims.reserved bit 1 is not honoured)
                                                        ("ep_order", C.c_void_p), ("tile_steps", C.c_void_p)]


class PmbError(RuntimeError):
    pass


_lib = None

_P = C.c_void_p
_SIGS = {
    "pmb_last_error": (C.c_char_p, []),
    "pmb_version": (C.c_int, []),
    "pmb_launch_count": (C.c_int64, []),
    "pmb_profile_begin": (C.c_int, []),
    "pmb_profile_end": (C.c_int, [C.POINTER(C.c_float), C.c_char_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "pmb_gather_episodes": (C.c_int, [C.POINTER(GatherField), C.c_int32, _P, C.c_int64, C.c_int64, _P]),
    "pmb_gather_episode_steps": (C.c_int, [C.POINTER(StepField), C.c_int32, _P, C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                           _P, C.c_int32, _P]),
    "pmb_host_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p)]),
    "pmb_host_free": (C.c_int, [_P]),
    "pmb_batch_update": (C.c_int, [C.POINTER(UpdateField), C.c_int32, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                   C.c_int64, _P, C.c_int64, _P]),
    "pmb_max_t_filled": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int64, _P, _P]),
    "pmb_h2d_rows": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, _P]),
    "pmb_device_info": (C.c_int, [C.POINTER(C.c_int32)] * 3 + [C.POINTER(C.c_int64)]),
    "pmb_flat_layout": (C.c_int, [C.POINTER(Dims), C.POINTER(Layout)]),
    "pmb_obs_bf16_supported": (C.c_int, [C.POINTER(Dims), C.c_int32]),
    "pmb_field_dtype_supported": (C.c_int, [C.POINTER(Dims), C.c_int32, C.c_int32, C.c_int32]),
    "pmb_learner_workspace_bytes": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_learner_workspace_views": (C.c_int, [C.POINTER(Dims), _P, C.c_int64, C.POINTER(WsViews)]),
    "pmb_agent_fc1_fwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), C.c_int32, C.c_int32, _P, _P, _P]),
    "pmb_agent_fc1_dense_fwd": (C.c_int, [C.POINTER(Dims), C.c_int64, C.c_int32, _P, _P, _P, _P]),
    "pmb_agent_gru_unroll_fwd": (C.c_int, [C.POINTER(Dims), C.c_int64, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pmb_target_select": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, _P, _P, _P, _P, _P]),
    "pmb_mixer_fwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, _P, C.c_int32, _P, _P, _P]),
    "pmb_td_loss": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, _P, C.c_float, _P, _P, _P]),
    "pmb_stats_reset": (C.c_int, [_P, _P]),
    "pmb_mixer_bwd_workspace_bytes": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_mixer_bwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, _P, _P, _P, _P, _P, _P, C.c_int64, _P]),
    "pmb_agent_bwd_workspace_bytes": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_agent_unroll_bwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, _P]),
    "pmb_agent_step_bwd_workspace_bytes": (C.c_int64, [C.POINTER(Dims), C.c_int64]),
    "pmb_agent_step_bwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), C.c_int32, _P, C.c_int64, _P, _P, _P, _P, _P, _P,
                                     _P, _P, _P, C.c_int64, _P]),
    "pmb_clip_rmsprop_update": (C.c_int, [C.c_int64, _P, _P, _P, _P, C.c_int32, _P, C.c_float, C.c_float, C.c_float,
                                          C.c_float, _P, _P]),
    "pmb_dp_pack": (C.c_int, [C.c_int64, _P, _P, _P]),
    "pmb_dp_unpack": (C.c_int, [C.c_int64, _P, _P, _P]),
    "pmb_ipc_export": (C.c_int, [_P, _P, C.POINTER(C.c_int64)]),
    "pmb_ipc_open": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_void_p)]),
    "pmb_ipc_close": (C.c_int, [_P, C.c_int64]),
    "pmb_dp_exchange_floats": (C.c_int64, [C.c_int64]),
    "pmb_dp_fused_allreduce_update": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.c_int64, C.c_int64, _P, _P, _P,
                                                C.c_int32, _P, C.c_float, C.c_float, C.c_float, C.c_float, _P, C.c_int64, _P]),
    "pmb_epsilon_greedy": (C.c_int, [C.c_int64, C.c_int32, _P, _P, C.c_float, _P, _P, C.c_uint64, C.c_uint64, _P, _P]),
    "pmb_select_actions_workspace_bytes": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_select_actions_step": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), C.c_int32, _P, _P, C.c_float, _P, _P,
                                          C.c_uint64, C.c_uint64, _P, _P, _P, C.c_int64, _P]),
    "pmb_gemm_bf16_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "pmb_gemm_bf16_tn": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.c_int64, _P]),
    "pmb_gemm_bf16_atb_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "pmb_gemm_bf16_atb": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, C.c_int64, _P, C.c_int64, _P, _P, _P,
                                    C.c_int64, _P]),
    "pmb_coma_critic_numel": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_coma_workspace_bytes": (C.c_int64, [C.POINTER(Dims)]),
    "pmb_coma_workspace_views": (C.c_int, [C.POINTER(Dims), _P, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                           C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "pmb_coma_train_step": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), C.POINTER(ComaHParams), _P, _P, _P, _P, _P, _P, _P, _P,
                                      C.c_int64, _P, _P]),
    "pmb_coma_critic_fwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, C.c_int32, C.c_int32, _P, _P, C.c_int64, _P]),
    "pmb_coma_critic_step_fwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, C.c_int32, C.c_int32, _P, _P, _P, _P,
                                           C.c_int64, _P]),
    "pmb_coma_critic_step_bwd_workspace_bytes": (C.c_int64, [C.POINTER(Dims), C.c_int32]),
    "pmb_coma_critic_step_bwd": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P,
                                           C.c_int64, _P]),
    "pmb_policy_head": (C.c_int, [C.c_int64, C.c_int32, C.c_float, C.c_int32, _P, _P, _P, _P]),
    "pmb_multinomial": (C.c_int, [C.c_int64, C.c_int32, _P, _P, _P, C.c_int32, C.c_uint64, C.c_uint64, _P, _P]),
    "pmb_qlearner_train_step": (C.c_int, [C.POINTER(Dims), C.POINTER(Batch), C.POINTER(HParams), _P, _P, _P, _P, _P,
                                          C.c_int64, _P, _P]),
}
EXPORTED_SYMBOLS = sorted(_SIGS)


def lib():
    """Load (once) and return the CDLL.  Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PmbError("%s not found: build it with `python -m pymarl_b200.build` "
                           "(there is no CPU fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def profile_begin():
    check(lib().pmb_profile_begin(), "pmb_profile_begin")


def profile_end(max_phases=48, stride=40):
    """-> list of (phase name, milliseconds) for the calls issued since profile_begin()."""
    ms = (C.c_float * max_phases)()
    names = C.create_string_buffer(max_phases * stride)
    n = C.c_int32(0)
    check(lib().pmb_profile_end(ms, names, stride, max_phases, C.byref(n)), "pmb_profile_end")
    raw = names.raw
    return [(raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0].decode(), float(ms[i])) for i in range(n.value)]


def check(rc, what=""):
    if rc != 0:
        msg = lib().pmb_last_error().decode("utf-8", "replace")
        raise PmbError("%s failed (status %d): %s" % (what or "pymarl_b200 call", rc, msg))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(th.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name):
    if not t.is_cuda:
        raise PmbError("%s must live on a CUDA device (pymarl_b200 has no CPU path); got %s" % (name, t.device))


def autograd_mode(args):
    """True when a module called with these args builds an autograd graph: the ``autograd_modules`` key is set and grad
    mode is on (not under th.no_grad() / th.inference_mode()).  Otherwise the modules run their inference kernels."""
    return bool(getattr(args, "autograd_modules", False)) and th.is_grad_enabled()


def no_double_backward(what):
    """Called at the top of a module Function's backward: the hand-written backward kernels are not differentiable."""
    if th.is_grad_enabled():
        raise PmbError("%s: double backward (create_graph=True) is not supported by the pymarl_b200 kernels" % what)


def make_dims(B, T, N, O, S, A, H, E, obs_last_action=True, obs_agent_id=True, mixer="qmix", double_q=True,
              precision="fp32", skip_padding=False):
    """skip_padding sets pmb_dims.reserved bit 1: the learner step skips the padded timesteps of a ragged batch where
    the fused tensor-core path runs (see include/pymarl_b200.h); elsewhere the bit is ignored."""
    if mixer not in MIXER_IDS:
        raise ValueError("Mixer {} not recognised.".format(mixer))       # learners/q_learner.py:26
    return Dims(int(B), int(T), int(N), int(O), int(S), int(A), int(H), int(E), int(bool(obs_last_action)),
                int(bool(obs_agent_id)), MIXER_IDS[mixer], int(bool(double_q)), PREC_IDS[precision],
                2 if skip_padding else 0)


def flat_layout(dims):
    L = Layout()
    check(lib().pmb_flat_layout(C.byref(dims), C.byref(L)), "pmb_flat_layout")
    return L


def _batch_stride(t, inner):
    """batch stride in elements; the inner dims must be contiguous."""
    exp = 1
    for size, stride in zip(reversed(t.shape[1:]), reversed(t.stride()[1:])):
        if size != 1 and stride != exp:
            return None
        exp *= size
    return t.stride(0) if t.shape[0] > 1 else inner


_FIELD_DTYPES = {"obs": th.float32, "state": th.float32, "actions": th.int64, "avail_actions": th.int32,
                 "reward": th.float32, "terminated": th.uint8, "filled": th.int64}


def h2d_time_slice(t, lo, hi, dev, lead=0):
    """``t[:, lo:hi]`` of a host tensor [B, T, ...] as a dense device tensor, copied with ONE strided
    cudaMemcpy2DAsync (no contiguous host temporary).  Falls back to torch for exotic layouts.

    ``lead`` > 0 (single timestep only): the result is presented as a ``[B, lead + 1, ...]`` view whose LAST time
    index holds the copied step (batch stride = time stride = one step; the earlier time indices alias other rows
    and must not be read).  This lets a kernel that addresses every field with one common time index read a field
    of which only the current step was transferred next to fields that also carry the previous step."""
    import torch as th
    B, T = t.shape[0], t.shape[1]
    inner = 1
    for s in t.shape[2:]:
        inner *= s
    assert lead == 0 or hi - lo == 1
    if t.is_cuda or t.dim() < 2 or not t[0].is_contiguous() or t.stride(0) != T * inner or B == 0:
        if lead:
            buf = th.empty((B + lead, 1) + tuple(t.shape[2:]), dtype=t.dtype, device=dev)
            buf[lead:].copy_(t[:, lo:hi], non_blocking=True)
        else:
            return t[:, lo:hi].to(dev, non_blocking=True)
    else:
        buf = th.empty((B + lead, hi - lo) + tuple(t.shape[2:]), dtype=t.dtype, device=dev)
        es = t.element_size()
        check(lib().pmb_h2d_rows(C.c_void_p(buf.data_ptr() + lead * inner * es), C.c_void_p(t.data_ptr() + lo * inner * es), B,
                                 (hi - lo) * inner * es, T * inner * es, stream_ptr(dev)), "pmb_h2d_rows")
        if not lead:
            return buf
    return th.as_strided(buf, (B, lead + 1) + tuple(t.shape[2:]), (inner, inner) + tuple(buf.stride()[2:]))


def gather_episodes(src_tensors, ep_ids, n_src):
    """out[k][j] = src[k][ep_ids[j]] for a dict of contiguous CUDA tensors [n_src, ...] in one launch."""
    import torch as th
    keys = list(src_tensors)
    dev = src_tensors[keys[0]].device
    ids = th.as_tensor(ep_ids, dtype=th.int64).to(dev)
    n = ids.numel()
    out = {k: th.empty((n,) + tuple(v.shape[1:]), dtype=v.dtype, device=dev) for k, v in src_tensors.items()}
    for i in range(0, len(keys), 16):
        chunk = keys[i:i + 16]
        arr = (GatherField * len(chunk))()
        for j, k in enumerate(chunk):
            v = src_tensors[k]
            require_cuda(v, "buffer[%r]" % k)
            if not v.is_contiguous():
                raise PmbError("gather_episodes needs contiguous buffer fields (%r is not)" % k)
            arr[j] = GatherField(v.data_ptr(), out[k].data_ptr(), v[0].numel() * v.element_size())
        check(lib().pmb_gather_episodes(arr, len(chunk), ptr(ids), n, n_src, stream_ptr(dev)), "pmb_gather_episodes")
    return out


def host_empty(shape, dtype):
    """Uninitialised host tensor in page-locked memory that is mapped into the device's address space (pmb_host_alloc),
    so that gather_episode_steps reads it in place.  Freed when its last view dies.  torch's pinned allocator would
    round every field of a replay buffer up to a power of two (a 28 GB obs field takes 32 GB); this does not."""
    n = 1
    for s in shape:
        n *= int(s)
    nbytes = n * th.empty((), dtype=dtype).element_size()
    p = C.c_void_p()
    check(lib().pmb_host_alloc(max(nbytes, 1), C.byref(p)), "pmb_host_alloc")
    raw = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    weakref.finalize(raw, lib().pmb_host_free, C.c_void_p(p.value))      # runs when the storage lets go of `raw`
    return th.frombuffer(raw, dtype=th.uint8)[:nbytes].view(dtype).view(tuple(shape))


def episode_rows(n, shape, dtype, dev):
    """Device tensor [n, *shape] whose rows start 16-byte aligned (the row stride is rounded up to 16 bytes): the
    destination layout of gather_episode_steps.  The kernels take any batch stride."""
    es = th.empty((), dtype=dtype).element_size()
    inner = 1
    for s in shape:
        inner *= int(s)
    row = -(-inner * es // 16) * 16 // es
    buf = th.empty(max(n, 1) * row, dtype=dtype, device=dev)
    return buf.as_strided((n,) + tuple(shape), (row,) + th.empty(tuple(shape), device="meta").stride())


def gather_episode_steps(src, ep_ids, steps, out, filled=None):
    """out[k][j] = src[k][ep_ids[j], :steps] for every key, one launch per 8 fields on the current stream.  src[k]:
    contiguous [n_src, T_src, ...] buffer fields in HBM or in pinned mapped host memory; out[k]: device tensors from
    episode_rows(n_ids, (steps, ...)); ep_ids: int64 device tensor.  With `filled` (the buffer's filled field), episode j
    copies only its first min(steps, last filled step + 2) timesteps and the rest of its row is written as zeros."""
    keys = list(src)
    some = src[keys[0]]
    n_src, T_src = int(some.shape[0]), int(some.shape[1])
    n = int(ep_ids.numel())
    dev = out[keys[0]].device
    for k in keys:
        v, o = src[k], out[k]
        if not v.is_contiguous() or tuple(v.shape[:2]) != (n_src, T_src):
            raise PmbError("gather_episode_steps needs contiguous [n_src, T, ...] buffer fields (%r is not)" % k)
        if tuple(o.shape) != (n, steps) + tuple(v.shape[2:]) or o.dtype != v.dtype or (n > 0 and not o[0].is_contiguous()):
            raise PmbError("gather_episode_steps: out[%r] must be episode_rows(%d, %r)" % (k, n, (steps,) + tuple(v.shape[2:])))
    if filled is not None and (not filled.is_contiguous() or filled.dtype != th.int64 or tuple(filled.shape[:2]) != (n_src, T_src)):
        raise PmbError("gather_episode_steps: filled must be the buffer's contiguous int64 [n_src, T] field")
    for i in range(0, len(keys), 8):
        chunk = keys[i:i + 8]
        arr = (StepField * len(chunk))()
        for j, k in enumerate(chunk):
            v, o = src[k], out[k]
            es = v.element_size()
            arr[j] = StepField(v.data_ptr(), o.data_ptr(), v[0, 0].numel() * es, o.stride(0) * es)
        check(lib().pmb_gather_episode_steps(arr, len(chunk), ptr(ep_ids), n, n_src, T_src, int(steps), ptr(filled),
                                             int(filled is not None), stream_ptr(dev)), "pmb_gather_episode_steps")
    return out


def obs_bf16_supported(dims, entry):
    """Whether the kernels of ``entry`` (ENTRY_TRAIN_STEP / ENTRY_SELECT_ACTIONS) read bf16 obs natively for ``dims``."""
    return lib().pmb_obs_bf16_supported(C.byref(dims), int(entry)) == 1


def field_dtype_supported(dims, entry, field, dtype):
    """Whether the kernels of ``entry`` read ``field`` ("obs", "state" or "avail_actions") stored as ``dtype`` (DTYPE_*)
    natively for ``dims`` (pmb_field_dtype_supported)."""
    return lib().pmb_field_dtype_supported(C.byref(dims), int(entry), FIELD_IDS[field], int(dtype)) == 1


# the compact cell types a kernel may read natively: (field, torch dtype) -> enum pmb_dtype.  bool avail is passed as
# its uint8 view (one byte holding 0 or 1).
_COMPACT = {("obs", th.bfloat16): DTYPE_BF16, ("state", th.bfloat16): DTYPE_BF16,
            ("avail_actions", th.uint8): DTYPE_U8, ("avail_actions", th.bool): DTYPE_U8}


def make_batch(fields, need_state=True, keep=None, ep_index=None, dims=None, entry=None):
    """Build the pmb_batch view of an EpisodeBatch-like mapping (``fields[k]`` -> tensor).
    Tensors that are not on CUDA, have the wrong dtype or non-contiguous inner dims are
    converted (the converted tensors are appended to ``keep`` so they outlive the call).
    Compact storage chosen in the scheme - bf16 obs or state, uint8 or bool avail_actions - is passed through as it is
    when ``dims`` and ``entry`` name a call whose kernels read it natively (field_dtype_supported); otherwise it is
    converted to the reference type."""
    b = Batch()
    b.obs_dtype = b.state_dtype = b.avail_dtype = 0
    names = [("obs", "obs"), ("state", "state"), ("actions", "actions"), ("avail", "avail_actions"),
             ("reward", "reward"), ("terminated", "terminated"), ("filled", "filled")]
    for cname, key in names:
        if key == "state" and not need_state:
            setattr(b, cname, None)
            setattr(b, cname + "_sb", 0)
            continue
        t = fields[key]
        require_cuda(t, "batch[%r]" % key)
        code = _COMPACT.get((key, t.dtype))
        if code is not None and dims is not None and entry is not None and field_dtype_supported(dims, entry, key, code):
            setattr(b, cname + "_dtype", code)
            if t.dtype == th.bool:
                t = t.view(th.uint8)
        elif t.dtype != _FIELD_DTYPES[key]:
            t = t.to(_FIELD_DTYPES[key])
        inner = 1
        for s in t.shape[1:]:
            inner *= s
        sb = _batch_stride(t, inner)
        if sb is None:
            t = t.contiguous()
            sb = inner
        if keep is not None:
            keep.append(t)
        setattr(b, cname, t.data_ptr())
        setattr(b, cname + "_sb", sb)
    b.ep_index = None
    if ep_index is not None:
        require_cuda(ep_index, "ep_index")
        if ep_index.dtype != th.int64 or not ep_index.is_contiguous():
            raise PmbError("ep_index must be a contiguous int64 tensor")
        if keep is not None:
            keep.append(ep_index)
        b.ep_index = ep_index.data_ptr()
    return b
