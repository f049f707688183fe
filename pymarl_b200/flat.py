"""Flat fp32 parameter storage.  The CUDA kernels address the agent and the mixer through ONE
contiguous buffer (layout: include/pymarl_b200.h, pmb_flat_layout); the nn.Parameters keep the
reference's names and shapes and are re-pointed to views of that buffer, so state_dict(),
load_state_dict(), deepcopy, the rollout MAC and the optimizer all see the same storage."""
import torch as th

from . import _lib

AGENT_KEYS = ["fc1.weight", "fc1.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh",
              "fc2.weight", "fc2.bias"]
# flat order of the mixer block (hypernet weights first: they form one [(N+3)E, S] matrix)
MIXER_KEYS = ["hyper_w_1.weight", "hyper_w_final.weight", "hyper_b_1.weight", "V.0.weight",
              "hyper_w_1.bias", "hyper_w_final.bias", "hyper_b_1.bias", "V.0.bias", "V.2.weight", "V.2.bias"]
_FIRST_ID = {"agent": 0, "mixer": len(AGENT_KEYS)}
_KEYS = {"agent": AGENT_KEYS, "mixer": MIXER_KEYS}


def _named(module):
    return dict(module.named_parameters())


def bind(flat, layout, module, kind, grad=None, base=None):
    """Copy the module's current parameter values into `flat` (block starting at element
    `base`, default: the block's offset in the full layout) and re-point every parameter's
    .data (and .grad when `grad` is given) to the matching slice."""
    first, keys = _FIRST_ID[kind], _KEYS[kind]
    block0 = layout.offset[first]
    base = block0 if base is None else base
    params = _named(module)
    with th.no_grad():
        for i, k in enumerate(keys):
            p = params[k]
            off, n = base + layout.offset[first + i] - block0, layout.numel[first + i]
            assert n == p.numel(), (k, n, p.numel())
            view = flat[off:off + n].view(p.shape)
            view.copy_(p.data.to(device=flat.device, dtype=flat.dtype))
            p.data = view
            if grad is not None:
                p.grad = grad[off:off + n].view(p.shape)
    object.__setattr__(module, "_pmb_flat", flat)       # keep the storage alive with the module


def block_ptr(module, kind, layout):
    """Device address of the module's parameter block if its parameters are laid out
    back-to-back in flat-layout order (fp32, CUDA), else None."""
    first, keys = _FIRST_ID[kind], _KEYS[kind]
    params = _named(module)
    p0 = params[keys[0]]
    if not p0.is_cuda or p0.dtype != th.float32:
        return None
    base = p0.data_ptr()
    for i, k in enumerate(keys):
        p = params[k]
        if (p.device != p0.device or p.dtype != th.float32 or not p.is_contiguous()
                or p.data_ptr() != base + (layout.offset[first + i] - layout.offset[first]) * 4):
            return None
    return base


def ensure_block(module, kind, dims):
    """Return the device address of a valid flat block for `module`, binding the parameters
    to a fresh private buffer when they are not laid out that way (e.g. after .cuda())."""
    layout = _lib.flat_layout(dims)
    addr = block_ptr(module, kind, layout)
    if addr is not None:
        return addr
    p0 = _named(module)[_KEYS[kind][0]]
    _lib.require_cuda(p0, "%s parameters" % kind)
    flat = th.empty(block_numel(layout, kind), dtype=th.float32, device=p0.device)
    bind(flat, layout, module, kind, base=0)
    return flat.data_ptr()


def bind_in_order(module, keys, flat=None, grad=None):
    """Generic variant for modules outside the agent / mixer layout (the COMA critic): lay the named parameters out
    back to back in `keys` order in one flat fp32 buffer (created on the module's device when not given), re-point
    .data (and .grad) to views of it, and return the buffer."""
    params = _named(module)
    n = sum(params[k].numel() for k in keys)
    p0 = params[keys[0]]
    if flat is None:
        flat = th.empty(n, dtype=th.float32, device=p0.device)
    off = 0
    with th.no_grad():
        for k in keys:
            p = params[k]
            view = flat[off:off + p.numel()].view(p.shape)
            view.copy_(p.data.to(device=flat.device, dtype=flat.dtype))
            p.data = view
            if grad is not None:
                p.grad = grad[off:off + p.numel()].view(p.shape)
            off += p.numel()
    object.__setattr__(module, "_pmb_flat", flat)
    return flat


def is_bound_in_order(module, keys, flat):
    """True when the named parameters still are the back-to-back views of `flat` that bind_in_order made."""
    params = _named(module)
    off = 0
    for k in keys:
        p = params[k]
        if not p.is_cuda or p.dtype != th.float32 or p.data_ptr() != flat.data_ptr() + 4 * off:
            return False
        off += p.numel()
    return True


def grad_views(block, layout, module, kind):
    """Per-parameter views (in named_parameters() order) of a flat gradient block of `kind` that starts at the block's
    own offset: what a module Function's backward returns for the parameters."""
    first, keys = _FIRST_ID[kind], _KEYS[kind]
    block0 = layout.offset[first]
    view = {}
    for i, k in enumerate(keys):
        off, n = layout.offset[first + i] - block0, layout.numel[first + i]
        view[k] = block[off:off + n]
    return [view[k].view(p.shape) for k, p in module.named_parameters()]


def block_numel(layout, kind):
    first = _FIRST_ID[kind]
    return sum(layout.numel[first + i] for i in range(len(_KEYS[kind])))
