"""EpisodeBatch / ReplayBuffer with the reference's layout contract and call surface
(reference: components/episode_buffer.py:8-298), written for this package so rollout and
learner code keep working when the reference tree is not importable.

Layout contract (what the CUDA path relies on): every per-timestep field is one tensor
``[batch, max_seq_length, (group size,) *vshape]`` of the scheme dtype (default float32),
episode-constant fields drop the time axis, and an int64 ``filled [batch, T, 1]`` marks
written timesteps.  Slicing returns views that share storage (a ``[:, :t]`` slice keeps the
full-T batch stride); indexing with an id list/array copies (advanced indexing).
"""
from types import SimpleNamespace

import numpy as np
import torch as th


def _as_tuple(v):
    return (v,) if isinstance(v, int) else tuple(v)


class EpisodeBatch:
    pinned = False          # fields live in page-locked host memory mapped into the device (ReplayBuffer(pin_memory=True))

    def __init__(self, scheme, groups, batch_size, max_seq_length, data=None, preprocess=None, device="cpu"):
        self.scheme = scheme.copy()
        self.groups = groups
        self.batch_size = batch_size
        self.max_seq_length = max_seq_length
        self.preprocess = {} if preprocess is None else preprocess
        self.device = device
        if data is not None:
            self.data = data
            return
        self.data = SimpleNamespace(transition_data={}, episode_data={})
        self._setup_data(self.scheme, self.groups, batch_size, max_seq_length, self.preprocess)

    # ---- allocation ---------------------------------------------------------------------
    def _setup_data(self, scheme, groups, batch_size, max_seq_length, preprocess):
        for key, (new_key, transforms) in (preprocess or {}).items():
            assert key in scheme, "preprocess key {} is not in the scheme".format(key)
            vshape, dtype = self.scheme[key]["vshape"], self.scheme[key].get("dtype", th.float32)
            for tr in transforms:
                vshape, dtype = tr.infer_output_info(vshape, dtype)
            entry = {"vshape": vshape, "dtype": dtype}
            for carry in ("group", "episode_const"):
                if carry in self.scheme[key]:
                    entry[carry] = self.scheme[key][carry]
            self.scheme[new_key] = entry
        assert "filled" not in scheme, '"filled" is a reserved key for masking.'
        scheme.update({"filled": {"vshape": (1,), "dtype": th.long}})
        for key, info in scheme.items():
            assert "vshape" in info, "Scheme must define vshape for {}".format(key)
            shape = _as_tuple(info["vshape"])
            group = info.get("group")
            if group:
                assert group in groups, "Group {} must have its number of members defined in _groups_".format(group)
                shape = (groups[group],) + shape
            dtype = info.get("dtype", th.float32)
            if info.get("episode_const", False):
                self.data.episode_data[key] = self._zeros((batch_size,) + shape, dtype)
            else:
                self.data.transition_data[key] = self._zeros((batch_size, max_seq_length) + shape, dtype)

    def _zeros(self, shape, dtype):
        if self.pinned:
            from .. import _lib
            return _lib.host_empty(shape, dtype).zero_()
        return th.zeros(shape, dtype=dtype, device=self.device)

    def extend(self, scheme, groups=None):
        self._setup_data(scheme, self.groups if groups is None else groups, self.batch_size, self.max_seq_length, None)

    def to(self, device):
        for store in (self.data.transition_data, self.data.episode_data):
            for k in store:
                store[k] = store[k].to(device)
        self.device = device

    # ---- writes ---------------------------------------------------------------------------
    def update(self, data, bs=slice(None), ts=slice(None), mark_filled=True):
        slices = self._parse_slices((bs, ts))
        if self._update_on_device(data, slices, mark_filled):
            return
        for k, v in data.items():
            if k in self.data.transition_data:
                store, sl = self.data.transition_data, tuple(slices)
                if mark_filled:
                    store["filled"][sl] = 1
                    mark_filled = False
            elif k in self.data.episode_data:
                store, sl = self.data.episode_data, slices[0]
            else:
                raise KeyError("{} not found in transition or episode data".format(k))
            dtype = self.scheme[k].get("dtype", th.float32)
            v = th.as_tensor(v, dtype=dtype, device=self.device) if not isinstance(v, th.Tensor) \
                else v.to(device=self.device, dtype=dtype)
            dest = store[k][sl]
            self._check_safe_view(v, dest)
            store[k][sl] = v.view_as(dest)
            if k in self.preprocess:
                new_k, transforms = self.preprocess[k]
                out = store[k][sl]
                for tr in transforms:
                    out = tr.transform(out)
                store[new_k][sl] = out.view_as(store[new_k][sl])

    def update_masked(self, data, row_mask, ts, mark_filled=True):
        """update(data, bs=<rows where row_mask is set>, ts=ts) for a batch in HBM WITHOUT a host synchronisation: `data`
        holds a value for EVERY episode row ([batch_size, ...] per key, device tensors), `row_mask` is a device bool tensor
        [batch_size]; rows whose mask is clear are skipped inside the kernel (their index is -1).  What a vectorised
        runner needs each timestep (the reference's runners pass the list of live envs, parallel_runner.py:109,170-176,
        which costs a device -> host round trip when the mask lives on the GPU)."""
        idx = th.where(row_mask, th.arange(row_mask.numel(), device=row_mask.device), th.full_like(row_mask, -1, dtype=th.int64))
        slices = self._parse_slices((slice(None), ts))
        if not self._update_on_device(data, [idx, slices[1]], mark_filled, trusted_index=True):
            rows = row_mask.nonzero().flatten()
            self.update({k: v[rows] for k, v in data.items()}, bs=rows, ts=ts, mark_filled=mark_filled)

    def _update_on_device(self, data, slices, mark_filled, trusted_index=False):
        """A batch that lives in HBM: ALL fields of the call, `filled` and the fused OneHot preprocess in ONE launch
        (pmb_batch_update) instead of one indexed assignment + one scatter per field.  Returns False (caller takes the
        generic path) for what the kernel does not cover: episode-constant fields, boolean / strided-time indices,
        preprocess chains other than a single OneHot."""
        import ctypes as C
        from .transforms import OneHot
        store = self.data.transition_data
        if th.device(self.device).type != "cuda" or not data or len(data) > 8:
            return False
        bs, ts = slices
        some = next(iter(store.values()))
        n_rows, n_t = some.shape[0], some.shape[1]
        if not isinstance(ts, slice):
            return False
        t0, t1, tstep = ts.indices(n_t)
        if tstep != 1 or t1 <= t0:
            return False
        nt = t1 - t0
        b_index, b0, b_step = None, 0, 1
        if isinstance(bs, slice):
            b0, b1, b_step = bs.indices(n_rows)
            if b_step < 1:
                return False
            nb = max(0, -(-(b1 - b0) // b_step))
        else:
            if isinstance(bs, th.Tensor):
                if bs.dtype == th.bool:
                    return False
                b_index = bs.to(device=self.device, dtype=th.int64).reshape(-1).contiguous()
                if trusted_index:                          # update_masked: -1 marks skipped rows, the kernel bounds-checks
                    lo_hi = (0, 0)
                else:
                    lo_hi = (int(b_index.min()), int(b_index.max())) if b_index.numel() else (0, 0)
            else:
                arr = np.asarray(bs)
                if arr.dtype == np.bool_ or arr.ndim != 1:
                    return False
                lo_hi = (int(arr.min()), int(arr.max())) if arr.size else (0, 0)
                b_index = th.as_tensor(arr.astype(np.int64)).to(self.device)
            nb = int(b_index.numel())
            if nb and (lo_hi[0] < -n_rows or lo_hi[1] >= n_rows):
                raise IndexError("episode index out of range")
            if nb and lo_hi[0] < 0 and not trusted_index:
                b_index = th.where(b_index < 0, b_index + n_rows, b_index)
        if nb == 0:
            return True
        from .. import _lib
        descs, keep = [], []
        for k, v in data.items():
            if k not in store:
                return False
            dest = store[k]
            if not dest[0, 0].is_contiguous():
                return False
            dtype = self.scheme[k].get("dtype", th.float32)
            v = th.as_tensor(v, dtype=dtype, device=self.device) if not isinstance(v, th.Tensor) \
                else v.to(device=self.device, dtype=dtype)
            cell = dest[0, 0].numel()
            self._check_safe_view(v, SimpleNamespace(shape=(nb, nt) + tuple(dest.shape[2:])))
            if v.numel() != nb * nt * cell:
                raise ValueError("Unsafe reshape of {} to {}".format(tuple(v.shape), (nb, nt) + tuple(dest.shape[2:])))
            v = v.reshape(nb, nt, cell).contiguous()
            keep.append(v)
            es = dest.element_size()
            descs.append(_lib.UpdateField(v.data_ptr(), dest.data_ptr(), cell * es, dest.stride(0) * es, dest.stride(1) * es, 0, 0))
            if k in self.preprocess:
                new_k, transforms = self.preprocess[k]
                if len(transforms) != 1 or not isinstance(transforms[0], OneHot) or dtype != th.int64 \
                        or store[new_k].dtype != th.float32 or store[new_k][0, 0].numel() != cell * transforms[0].out_dim:
                    return False
                oh = store[new_k]
                descs.append(_lib.UpdateField(v.data_ptr(), oh.data_ptr(), cell * 8, oh.stride(0) * 4, oh.stride(1) * 4,
                                              transforms[0].out_dim, 0))
        arr = (_lib.UpdateField * len(descs))(*descs)
        filled = store["filled"] if mark_filled else None
        _lib.check(_lib.lib().pmb_batch_update(arr, len(descs), _lib.ptr(b_index), b0, b_step, nb, n_rows, t0, nt,
                                               _lib.ptr(filled), filled.stride(0) if filled is not None else 0,
                                               _lib.stream_ptr(some.device)), "pmb_batch_update")
        return True

    @staticmethod
    def _check_safe_view(v, dest):
        idx = len(v.shape) - 1
        for s in dest.shape[::-1]:
            if idx < 0 or v.shape[idx] != s:
                if s != 1:
                    raise ValueError("Unsafe reshape of {} to {}".format(v.shape, dest.shape))
            else:
                idx -= 1

    # ---- reads ----------------------------------------------------------------------------
    def __getitem__(self, item):
        if isinstance(item, str):
            if item in self.data.episode_data:
                return self.data.episode_data[item]
            if item in self.data.transition_data:
                return self.data.transition_data[item]
            raise ValueError(item)
        if isinstance(item, tuple) and all(isinstance(it, str) for it in item):
            new = SimpleNamespace(transition_data={}, episode_data={})
            for key in item:
                if key in self.data.transition_data:
                    new.transition_data[key] = self.data.transition_data[key]
                elif key in self.data.episode_data:
                    new.episode_data[key] = self.data.episode_data[key]
                else:
                    raise KeyError("Unrecognised key {}".format(key))
            scheme = {key: self.scheme[key] for key in item}
            groups = {self.scheme[key]["group"]: self.groups[self.scheme[key]["group"]]
                      for key in item if "group" in self.scheme[key]}
            return EpisodeBatch(scheme, groups, self.batch_size, self.max_seq_length, data=new, device=self.device)
        sl = self._parse_slices(item)
        new = SimpleNamespace(transition_data={}, episode_data={})
        if self._gpu_gather_ok(sl):
            # episode ids on a buffer that lives in HBM: ONE gather launch for all fields (pmb_gather_episodes),
            # then the (contiguous) time slice as a view
            from .. import _lib
            ids = np.asarray(sl[0].cpu() if isinstance(sl[0], th.Tensor) else sl[0]).reshape(-1)
            if ids.size and (ids.min() < 0 or ids.max() >= self.batch_size):
                raise IndexError("episode id out of range")
            tr = _lib.gather_episodes(self.data.transition_data, ids, self.batch_size)
            new.transition_data = {k: v[:, sl[1]] for k, v in tr.items()}
            if self.data.episode_data:
                new.episode_data = _lib.gather_episodes(self.data.episode_data, ids, self.batch_size)
            return EpisodeBatch(self.scheme, self.groups, int(ids.size), self._num_items(sl[1], self.max_seq_length),
                                data=new, device=self.device)
        for k, v in self.data.transition_data.items():
            new.transition_data[k] = v[tuple(sl)]
        for k, v in self.data.episode_data.items():
            new.episode_data[k] = v[sl[0]]
        return EpisodeBatch(self.scheme, self.groups, self._num_items(sl[0], self.batch_size),
                            self._num_items(sl[1], self.max_seq_length), data=new, device=self.device)

    def _gpu_gather_ok(self, sl):
        if not isinstance(sl[0], (list, np.ndarray, th.Tensor)) or not isinstance(sl[1], slice):
            return False
        if isinstance(sl[0], th.Tensor) and sl[0].dtype == th.bool:
            return False
        if isinstance(sl[0], np.ndarray) and sl[0].dtype == np.bool_:
            return False
        tensors = list(self.data.transition_data.values()) + list(self.data.episode_data.values())
        n = len(sl[0]) if not isinstance(sl[0], th.Tensor) else sl[0].numel()
        return bool(tensors) and 0 < n < 65536 and all(v.is_cuda and v.is_contiguous() for v in tensors) and \
            (sl[1].step in (None, 1))

    @staticmethod
    def _num_items(idx, max_size):
        if isinstance(idx, (list, np.ndarray)):
            return len(idx)
        if isinstance(idx, th.Tensor):
            return idx.numel()
        lo, hi, step = idx.indices(max_size)
        return 1 + (hi - lo - 1) // step

    @staticmethod
    def _parse_slices(items):
        if isinstance(items, (slice, int, list, np.ndarray, th.Tensor)):
            items = (items, slice(None))
        if isinstance(items[1], list):
            raise IndexError("Indexing across Time must be contiguous")
        return [slice(it, it + 1) if isinstance(it, int) else it for it in items]

    def max_t_filled(self):
        f = self.data.transition_data["filled"]
        if f.is_cuda and f.dtype == th.int64 and f.dim() == 3 and f.shape[2] == 1 and f.stride(1) == 1 and f.shape[0] > 0:
            from .. import _lib
            out = th.empty(1, dtype=th.int64, device=f.device)
            _lib.check(_lib.lib().pmb_max_t_filled(_lib.ptr(f), f.shape[0], f.shape[1], f.stride(0), _lib.ptr(out),
                                                   _lib.stream_ptr(f.device)), "pmb_max_t_filled")
            return out[0]
        return th.sum(f, 1).max(0)[0]

    def __repr__(self):
        return "EpisodeBatch. Batch Size:{} Max_seq_len:{} Keys:{} Groups:{}".format(
            self.batch_size, self.max_seq_length, self.scheme.keys(), self.groups.keys())


class IndexedEpisodeBatch:
    """What ``ReplayBuffer.sample`` returns when the buffer lives in HBM and ``zero_copy`` is on: the ids of the
    sampled episodes plus a reference to the buffer, instead of a gathered copy (29 GB at 27m_vs_30m / 4096).
    ``QLearner.train`` hands the ids to the kernels (``pmb_batch.ep_index``), which read the episodes in place.  It
    quacks like the EpisodeBatch the reference's train loop handles (``run.py:207-219``): ``max_t_filled()``,
    ``batch[:, :t]``, ``.to(device)``, ``batch[key]`` (materialises that field with the gather kernel).

    The buffer may also live in pinned host memory (``ReplayBuffer(..., pin_memory=True)``); then ``host_ids`` holds the
    ids on the host as well, and the learner's gather kernel pulls exactly the sampled episodes, fields and timesteps
    over PCIe (pmb_gather_episode_steps): nothing is gathered on the host."""

    def __init__(self, buffer, ep_ids, max_seq_length=None, host_ids=None):
        self.buffer = buffer
        self.ep_ids = ep_ids                       # int64 device tensor
        self.host_ids = host_ids                   # int64 host tensor when the buffer lives in pinned host memory
        self.batch_size = int(ep_ids.numel())
        self.max_seq_length = buffer.max_seq_length if max_seq_length is None else int(max_seq_length)
        self.scheme, self.groups, self.device = buffer.scheme, buffer.groups, buffer.device

    def max_t_filled(self):
        f = self.buffer.data.transition_data["filled"]
        ids = self.ep_ids if self.host_ids is None else self.host_ids
        return th.sum(f.index_select(0, ids)[:, :self.max_seq_length], 1).max(0)[0]

    def __getitem__(self, item):
        if isinstance(item, str):
            from .. import _lib
            src = self.buffer.data.transition_data
            if item not in src:
                raise ValueError(item)
            if self.host_ids is not None:
                T, v = self.max_seq_length, src[item]
                out = {item: _lib.episode_rows(self.batch_size, (T,) + tuple(v.shape[2:]), v.dtype, self.ep_ids.device)}
                return _lib.gather_episode_steps({item: v}, self.ep_ids, T, out)[item]
            return _lib.gather_episodes({item: src[item]}, self.ep_ids, self.buffer.batch_size)[item][:, :self.max_seq_length]
        if isinstance(item, tuple) and len(item) == 2 and item[0] == slice(None) and isinstance(item[1], slice):
            lo, hi, step = item[1].indices(self.max_seq_length)
            if lo != 0 or step != 1:
                raise IndexError("an IndexedEpisodeBatch can only be truncated in time: batch[:, :t]")
            return IndexedEpisodeBatch(self.buffer, self.ep_ids, hi, self.host_ids)
        raise IndexError("unsupported index for an IndexedEpisodeBatch: {!r}".format(item))

    def to(self, device):
        if th.device(device).type != "cuda":
            raise ValueError("an IndexedEpisodeBatch lives on the GPU")
        return self

    def __repr__(self):
        return "IndexedEpisodeBatch. Batch Size:{} Max_seq_len:{}".format(self.batch_size, self.max_seq_length)


class ReplayBuffer(EpisodeBatch):
    """Ring buffer of episodes with uniform sampling (episode_buffer.py:263-298).  Sampling
    draws ids on the legacy global numpy RandomState exactly like the reference, so a shared
    ``np.random.seed`` yields the same episode ids.

    ``pin_memory=True`` (host buffers) allocates every field in page-locked host memory mapped into the device, which
    lets ``zero_copy`` sampling read the buffer in place over PCIe; ``pin_memory_()`` moves an existing buffer there."""

    def __init__(self, scheme, groups, buffer_size, max_seq_length, preprocess=None, device="cpu", pin_memory=False):
        if pin_memory and th.device(device).type != "cpu":
            raise ValueError("pin_memory is for a buffer in host memory (device='cpu')")
        self.pinned = bool(pin_memory)
        super().__init__(scheme, groups, buffer_size, max_seq_length, preprocess=preprocess, device=device)
        self.buffer_size = buffer_size
        self.buffer_index = 0
        self.episodes_in_buffer = 0
        # opt-in: sample() returns an IndexedEpisodeBatch (ids only) instead of a gathered copy when the buffer is in HBM
        # or in pinned host memory
        self.zero_copy = False
        # CUDA event recorded after the learner's last reads of a zero-copy sample of this host buffer: train() returns
        # before its gathers have read the episodes, so writes wait on it
        self.device_reads = None

    def pin_memory_(self):
        """Move every field into page-locked host memory mapped into the device (one field at a time)."""
        if th.device(self.device).type != "cpu":
            raise ValueError("only a buffer in host memory can be pinned")
        if not self.pinned:
            from .. import _lib
            for store in (self.data.transition_data, self.data.episode_data):
                for k, v in store.items():
                    store[k] = _lib.host_empty(v.shape, v.dtype).copy_(v)
            self.pinned = True
        return self

    def update(self, data, bs=slice(None), ts=slice(None), mark_filled=True):
        if self.device_reads is not None:
            self.device_reads.synchronize()
            self.device_reads = None
        super().update(data, bs, ts, mark_filled)

    def insert_episode_batch(self, ep_batch):
        n = ep_batch.batch_size
        if self.buffer_index + n > self.buffer_size:          # wrap: split at the end of the ring
            left = self.buffer_size - self.buffer_index
            self.insert_episode_batch(ep_batch[0:left, :])
            self.insert_episode_batch(ep_batch[left:, :])
            return
        where = slice(self.buffer_index, self.buffer_index + n)
        self.update(ep_batch.data.transition_data, where, slice(0, ep_batch.max_seq_length), mark_filled=False)
        self.update(ep_batch.data.episode_data, where)
        self.buffer_index += n
        self.episodes_in_buffer = max(self.episodes_in_buffer, self.buffer_index)
        self.buffer_index %= self.buffer_size
        assert self.buffer_index < self.buffer_size

    def can_sample(self, batch_size):
        return self.episodes_in_buffer >= batch_size

    def sample(self, batch_size):
        assert self.can_sample(batch_size)
        if self.episodes_in_buffer == batch_size:
            return self[:batch_size]
        ep_ids = np.random.choice(self.episodes_in_buffer, batch_size, replace=False)
        if self.zero_copy and th.device(self.device).type == "cuda":
            return IndexedEpisodeBatch(self, th.as_tensor(ep_ids, dtype=th.int64).to(self.device))
        if self.zero_copy and self.pinned:
            ids = th.as_tensor(ep_ids, dtype=th.int64)
            return IndexedEpisodeBatch(self, ids.to("cuda"), host_ids=ids)
        return self[ep_ids]

    def __repr__(self):
        return "ReplayBuffer. {}/{} episodes. Keys:{} Groups:{}".format(
            self.episodes_in_buffer, self.buffer_size, self.scheme.keys(), self.groups.keys())
