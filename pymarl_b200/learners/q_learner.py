"""QLearner: QMIX / VDN / IQL learner (reference: learners/q_learner.py:9-143).

train(batch, t_env, episode_num) issues ONE C-ABI call (pmb_qlearner_train_step) that runs
the whole step on the GPU: both agent unrolls, double-Q target selection, both mixers, the
masked TD loss, the hand-written backward (mixer backward + GRU BPTT), grad-norm clipping,
RMSprop and the hard target sync.  Parameters, gradients, RMSprop state and target
parameters live in four flat fp32 buffers; the nn.Parameters (reference names) are views.

Data parallel: with torch.distributed initialised (one process per GPU, NCCL) every rank
trains on its shard of the episodes (train() slices the sampled batch itself); the un-normalised
gradients and the five loss sums travel in ONE all-reduce per step and every rank applies the
identical update.  args.cuda_graph = True replays the whole step as one CUDA graph.
args.skip_padded_steps = True lets the step skip the padded timesteps of a ragged batch (pmb_dims.reserved
bit 1; honoured on the fused tensor-core path, ignored elsewhere).
A zero-copy sample of a replay buffer in pinned host memory (IndexedEpisodeBatch with host_ids) is pulled over PCIe by
the gather kernel (pmb_gather_episode_steps): chunk by chunk into the streamed step's chunk buffers, or in one piece.
"""
import copy
import ctypes as C

import torch as th

from .. import _lib, flat as _flat, data_parallel
from ..modules.mixers.qmix import QMixer
from ..modules.mixers.vdn import VDNMixer


class FusedRMSprop:
    """State holder with torch.optim.RMSprop's state_dict format (square_avg, step) so that
    opt.th checkpoints interchange with the reference (q_learner.py:30,135,143).  The update
    itself is the fused clip + RMSprop kernel (pmb_clip_rmsprop_update)."""

    def __init__(self, params, lr, alpha, eps):
        self.params = list(params)
        self.defaults = dict(lr=lr, momentum=0, alpha=alpha, eps=eps, centered=False, weight_decay=0,
                             capturable=False, foreach=None, maximize=False, differentiable=False)
        self.square_avg = [th.zeros_like(p.data) for p in self.params]       # re-pointed into flat_sq by the learner
        self.step_count = 0

    def zero_grad(self):
        pass                                                                   # gradients are overwritten each step

    def state_dict(self):
        state = {i: {"step": th.tensor(float(self.step_count)), "square_avg": sq.detach().clone()}
                 for i, sq in enumerate(self.square_avg)} if self.step_count > 0 else {}
        group = dict(self.defaults)
        group["params"] = list(range(len(self.params)))
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        for i, st in sd.get("state", {}).items():
            self.square_avg[int(i)].copy_(st["square_avg"])
            self.step_count = int(st.get("step", self.step_count))
        for g in sd.get("param_groups", [])[:1]:
            for k in ("lr", "alpha", "eps"):
                if k in g:
                    self.defaults[k] = g[k]


def _host_sample(batch):
    """A zero-copy sample of a replay buffer that lives in pinned host memory."""
    return getattr(batch, "host_ids", None) is not None


def _mark_buffer_read(batch, stream):
    """Record on `stream`, after its last gather from the host buffer, the event the buffer's writes wait on."""
    ev = th.cuda.Event()
    ev.record(stream)
    batch.buffer.device_reads = ev


class QLearner:
    def __init__(self, mac, scheme, logger, args):
        self.args = args
        self.mac = mac
        self.logger = logger

        self.params = list(mac.parameters())
        self.last_target_update_episode = 0

        self.mixer = None
        if args.mixer is not None:
            if args.mixer == "vdn":
                self.mixer = VDNMixer()
            elif args.mixer == "qmix":
                self.mixer = QMixer(args)
            else:
                raise ValueError("Mixer {} not recognised.".format(args.mixer))
            self.params += list(self.mixer.parameters())
            self.target_mixer = copy.deepcopy(self.mixer)

        self.optimiser = FusedRMSprop(self.params, lr=args.lr, alpha=args.optim_alpha, eps=args.optim_eps)
        self.target_mac = copy.deepcopy(mac)
        self.log_stats_t = -self.args.learner_log_interval - 1

        self.precision = getattr(args, "precision", "fp32")
        self._flat = None               # dict(p, g, sq, target, layout, key)
        self._workspace = None
        self._stats = None
        self._dp_scratch = None         # 4096 floats for the replicated clip + RMSprop of the data-parallel path
        self._px = None                 # data_parallel.PeerExchange when the fused NVLink exchange is in use
        self._graphs = {}               # CUDA graphs of the step (args.cuda_graph)
        self._hs = None                 # host-batch streaming state (copy stream, two chunk buffers, accumulators)
        self.last_stats = None          # device tensor [16] float64 of the latest step

    # ---- flat storage -----------------------------------------------------------------------
    def _layout_dims(self, B=1, T=2, O=None, S=None):
        a = self.args
        d_in = self.mac.agent.d_in
        O = d_in - (a.n_actions if a.obs_last_action else 0) - (a.n_agents if a.obs_agent_id else 0) if O is None else O
        S = int(getattr(self.mixer, "state_dim", 1)) if S is None else S
        return _lib.make_dims(B=B, T=T, N=a.n_agents, O=O, S=S, A=a.n_actions, H=a.rnn_hidden_dim,
                              E=getattr(a, "mixing_embed_dim", 1) if a.mixer == "qmix" else 1,
                              obs_last_action=a.obs_last_action, obs_agent_id=a.obs_agent_id, mixer=a.mixer,
                              double_q=a.double_q, precision=self.precision,
                              skip_padding=getattr(a, "skip_padded_steps", False))

    def _ensure_flat(self):
        """(Re)build the four flat buffers when the parameters are not views of them (first
        call, or after cuda()/.to() moved the modules)."""
        dev = self.mac.agent.fc1.weight.device
        _lib.require_cuda(self.mac.agent.fc1.weight, "learner parameters (call learner.cuda())")
        dims = self._layout_dims()
        layout = _lib.flat_layout(dims)
        has_mixer_params = self.args.mixer == "qmix"
        f = self._flat
        if f is not None and f["p"].device == dev:
            ok = _flat.block_ptr(self.mac.agent, "agent", layout) == f["p"].data_ptr()
            ok = ok and _flat.block_ptr(self.target_mac.agent, "agent", layout) == f["target"].data_ptr()
            if has_mixer_params:
                ok = ok and _flat.block_ptr(self.mixer, "mixer", layout) == f["p"].data_ptr() + layout.n_agent * 4
                ok = ok and _flat.block_ptr(self.target_mixer, "mixer", layout) == f["target"].data_ptr() + layout.n_agent * 4
            if ok:
                return f
        n = layout.n_total
        # Data parallel: the gradient lives in an exchange buffer the other ranks of the node map through CUDA IPC, and ONE
        # fused kernel per step does all-reduce + clip + RMSprop over NVLink (data_parallel.PeerExchange, csrc/dp_peer.cu).
        # Built collectively; when any rank cannot (args.dp_exchange = "nccl", >8 ranks, several nodes, no IPC) every rank
        # falls back to one NCCL all-reduce + the stand-alone update kernel.
        self._px = None
        if data_parallel.is_active() and getattr(self.args, "data_parallel", True) \
                and getattr(self.args, "dp_exchange", "peer") == "peer":
            px = data_parallel.PeerExchange(n, dev)
            self._px = px if px.ok else None
        # the gradient buffer carries PMB_DP_TAIL_FLOATS extra floats: the loss sums of the data-parallel exchange
        new = dict(p=th.zeros(n, dtype=th.float32, device=dev),
                   g=self._px.grad_view() if self._px is not None else th.zeros(n + _lib.DP_TAIL_FLOATS, dtype=th.float32, device=dev),
                   sq=th.zeros(n, dtype=th.float32, device=dev), target=th.zeros(n, dtype=th.float32, device=dev),
                   layout=layout)
        _flat.bind(new["p"], layout, self.mac.agent, "agent", grad=new["g"])
        _flat.bind(new["target"], layout, self.target_mac.agent, "agent")
        if has_mixer_params:
            _flat.bind(new["p"], layout, self.mixer, "mixer", grad=new["g"])
            _flat.bind(new["target"], layout, self.target_mixer, "mixer")
        # RMSprop state: carry over existing values, then view into flat_sq (self.params order)
        base, sq_views = new["p"].data_ptr(), []
        for p, old in zip(self.params, self.optimiser.square_avg):
            off = (p.data_ptr() - base) // 4
            view = new["sq"][off:off + p.numel()].view(p.shape)
            view.copy_(old.to(dev))
            sq_views.append(view)
        self.optimiser.square_avg = sq_views
        self._flat = new
        self._graphs = {}
        return new

    def _ensure_workspace(self, dims, dev):
        need = _lib.lib().pmb_learner_workspace_bytes(C.byref(dims))
        if need < 0:
            _lib.check(1, "pmb_learner_workspace_bytes")
        if self._workspace is None or self._workspace.numel() < need or self._workspace.device != dev:
            self._workspace = None
            self._workspace = th.empty(need, dtype=th.uint8, device=dev)
        if self._stats is None or self._stats.device != dev:
            self._stats = th.zeros(_lib.STATS_LEN, dtype=th.float64, device=dev)
        return need

    def workspace_views(self, dims):
        """Named tensors over the step's workspace (tests / debugging)."""
        v = _lib.WsViews()
        _lib.check(_lib.lib().pmb_learner_workspace_views(C.byref(dims), _lib.ptr(self._workspace),
                                                          self._workspace.numel(), C.byref(v)), "workspace_views")
        base = self._workspace.data_ptr()
        f32 = self._workspace.view(th.float32)
        B, T, N, A, H, E = dims.B, dims.T, dims.N, dims.A, dims.H, dims.E
        R, M = B * N, B * (T - 1)
        W = N if dims.mixer == 0 else 1
        shapes = dict(x_on=(T, R, H), x_tg=(T, R, H), h_stash=(T + 1, R, H), gates=(T, R, 4 * H), q_on=(T, R, A),
                      q_tg=(T, R, A), chosen=(B, T - 1, N), tmax=(B, T - 1, N), q_tot=(B, T - 1, W),
                      t_tot=(B, T - 1, W), g=(B, T - 1, W), d_chosen=(B, T - 1, N))
        if dims.mixer == 2:
            shapes["raw_on"] = (M, (N + 3) * E)
        out = {}
        for k, shp in shapes.items():
            off = (getattr(v, k) - base) // 4
            n = 1
            for s in shp:
                n *= s
            out[k] = f32[off:off + n].view(shp)
        if v.ep_order:                  # padded-step skipping ran (args.skip_padded_steps where it is honoured)
            n_tiles = (R + 127) // 128
            out["ep_order"] = self._workspace[v.ep_order - base:v.ep_order - base + 8 * B].view(th.int64)
            out["tile_steps"] = self._workspace[v.tile_steps - base:v.tile_steps - base + 4 * n_tiles].view(th.int32)
        return out

    # ---- the step ---------------------------------------------------------------------------
    def _step_fields(self, batch, names, dev, dp):
        """The tensors one step reads: (fields, ep_index, B, T).  With data parallelism active (and unless
        args.dp_shard_batch is False: the caller already passes rank-local episodes) every rank keeps the contiguous
        episode slice data_parallel.shard_slice gives it - views, or a slice of the sampled ids for a zero-copy replay
        sample; a host-resident batch is sliced BEFORE the H2D copy (run.py:214), so each rank transfers 1/world of it."""
        lo = hi = None
        if dp and getattr(self.args, "dp_shard_batch", True):
            lo, hi = data_parallel.shard_slice(batch.batch_size, data_parallel.rank(), data_parallel.world_size())
        fields, ep_index = {}, None
        if hasattr(batch, "ep_ids") and hasattr(batch, "buffer"):
            # zero-copy replay sample (IndexedEpisodeBatch): the kernels read the buffer's episodes in place
            ep_index = batch.ep_ids if lo is None else batch.ep_ids[lo:hi]
            if _host_sample(batch):
                # buffer in pinned host memory, in one piece: the (rank's) episodes cross PCIe into device rows
                src, T = batch.buffer.data.transition_data, batch.max_seq_length
                n = int(ep_index.numel())
                for k in names:
                    fields[k] = _lib.episode_rows(n, (T,) + tuple(src[k].shape[2:]), src[k].dtype, dev)
                trim = src["filled"] if getattr(self.args, "skip_padded_steps", False) else None
                _lib.gather_episode_steps({k: src[k] for k in names}, ep_index.contiguous(), T, fields, filled=trim)
                _mark_buffer_read(batch, th.cuda.current_stream(dev))
                return fields, None, n, T
            for k in names:
                fields[k] = batch.buffer.data.transition_data[k]
            return fields, ep_index, int(ep_index.numel()), batch.max_seq_length
        for k in names:
            t = batch[k]
            if lo is not None:
                t = t[lo:hi]
            fields[k] = t if t.is_cuda else t.to(dev, non_blocking=True)       # host batch: H2D here (run.py:214)
        obs = fields["obs"]
        return fields, None, obs.shape[0], obs.shape[1]

    def _launch(self, dims, pb, hp, f, need, dev, dp):
        """The device work of one step on the current stream: ONE C call; with data parallelism the exchange
        (pack -> one all-reduce -> unpack) and the replicated update follow."""
        L = _lib.lib()
        s = _lib.stream_ptr(dev)
        n = f["layout"].n_total
        if dims.B > 0:
            _lib.check(L.pmb_qlearner_train_step(C.byref(dims), C.byref(pb), C.byref(hp), _lib.ptr(f["p"]),
                                                 _lib.ptr(f["g"]), _lib.ptr(f["sq"]), _lib.ptr(f["target"]),
                                                 _lib.ptr(self._workspace), need, _lib.ptr(self._stats), s),
                       "pmb_qlearner_train_step")
        else:                                   # a rank without episodes still takes part in the exchange
            f["g"].zero_()
            self._stats.zero_()
        self._exchange_and_update(hp, f, dev, dp)

    def _exchange_and_update(self, hp, f, dev, dp):
        """What follows a skip_update step: the data-parallel exchange and the replicated clip + RMSprop update."""
        L = _lib.lib()
        s = _lib.stream_ptr(dev)
        n = f["layout"].n_total
        if dp and self._px is not None:
            # exchange + update fused into one kernel over NVLink peer memory
            self._px.fused_update(f["p"], f["sq"], f["target"], hp.do_target_sync, self._stats, hp.lr, hp.alpha, hp.eps,
                                  hp.grad_norm_clip, s)
        elif dp:
            # one exchange per step: [gradients of sum((td*mask)^2) | the five loss sums as (hi, lo) floats]
            _lib.check(L.pmb_dp_pack(n, _lib.ptr(f["g"]), _lib.ptr(self._stats), s), "pmb_dp_pack")
            data_parallel.allreduce_step(f["g"])
            _lib.check(L.pmb_dp_unpack(n, _lib.ptr(f["g"]), _lib.ptr(self._stats), s), "pmb_dp_unpack")
            _lib.check(L.pmb_clip_rmsprop_update(n, _lib.ptr(f["p"]), _lib.ptr(f["g"]), _lib.ptr(f["sq"]),
                                                 _lib.ptr(f["target"]), hp.do_target_sync, _lib.ptr(self._stats), hp.lr,
                                                 hp.alpha, hp.eps, hp.grad_norm_clip, _lib.ptr(self._dp_scratch), s),
                       "pmb_clip_rmsprop_update")

    # ---- host-resident batches, streamed ----------------------------------------------------------
    # A batch that lives in host memory (buffer_cpu_only, run.py:214) is PCIe-bound: 29 GB at 27m_vs_30m / 4096.  Episodes
    # are independent and the step's gradient is a plain sum over them, so the batch is cut into chunks of
    # args.host_stream_chunk episodes (default 512): chunk i + 1 crosses PCIe on a copy stream into the other of two
    # chunk-sized device buffers while chunk i runs as a skip_update step (un-normalised gradient + the five loss sums);
    # the chunk gradients and sums are added up and ONE exchange / clip / RMSprop update follows - the same arithmetic as
    # the data-parallel path with the chunks in the role of the ranks.  The device then holds two chunks and a chunk-sized
    # workspace instead of the whole batch (7 GB + 6.5 GB instead of 29 GB + 52 GB) and the compute hides under the copy.
    # A zero-copy sample of a pinned host buffer streams the same way; its chunks are gathered from the buffer by the
    # gather kernel on the copy stream (with args.skip_padded_steps it leaves out each episode's padded tail).
    def _host_stream_plan(self, batch, dp):
        a = self.args
        chunk = int(getattr(a, "host_stream_chunk", 512))
        indexed = hasattr(batch, "ep_ids") and hasattr(batch, "buffer")
        if chunk <= 0 or getattr(a, "cuda_graph", False) or (indexed and not _host_sample(batch)):
            return None
        if dp and (indexed or not getattr(a, "host_stream_dp", False)):
            return None        # with data parallelism every rank holds 1/world of the batch already; opt-in (not measured on GPUs)
        if not indexed and batch["obs"].is_cuda:
            return None
        n_ep = batch.batch_size if indexed else int(batch["obs"].shape[0])
        lo, hi = 0, n_ep
        if dp and getattr(a, "dp_shard_batch", True):
            lo, hi = data_parallel.shard_slice(n_ep, data_parallel.rank(), data_parallel.world_size())
        if hi - lo < 2 * chunk:
            return None
        return lo, hi, chunk

    def _train_streamed(self, batch, names, plan, f, dev, dp, hp):
        lo, hi, chunk = plan
        L = _lib.lib()
        a = self.args
        n = f["layout"].n_total
        main = th.cuda.current_stream(dev)
        st = self._hs
        if st is None or st["dev"] != dev:
            st = self._hs = dict(dev=dev, copy=th.cuda.Stream(dev), bufs=[{}, {}],
                                 copied=[th.cuda.Event(), th.cuda.Event()], done=[th.cuda.Event(), th.cuda.Event()],
                                 g=None, sums=th.zeros(5, dtype=th.float64, device=dev))
        if st["g"] is None or st["g"].numel() != n:
            st["g"] = th.zeros(n, dtype=th.float32, device=dev)
        host = _host_sample(batch)
        if host:                                 # chunk rows of the gather kernel: 16-byte aligned
            src, T = batch.buffer.data.transition_data, batch.max_seq_length
            src = {k: src[k] for k in names}
            shapes = {k: (T,) + tuple(src[k].shape[2:]) for k in names}
            trim = src["filled"] if getattr(a, "skip_padded_steps", False) else None
        else:
            src = {k: batch[k] for k in names}
            shapes = {k: tuple(src[k].shape[1:]) for k in names}
            T = src["obs"].shape[1]
        if st.get("host") != host:
            st["bufs"], st["host"] = [{}, {}], host
        for slot in st["bufs"]:
            for k in names:
                t = src[k]
                if k not in slot or tuple(slot[k].shape) != (chunk,) + shapes[k] or slot[k].dtype != t.dtype:
                    slot[k] = _lib.episode_rows(chunk, shapes[k], t.dtype, dev) if host else \
                        th.empty((chunk,) + shapes[k], dtype=t.dtype, device=dev)
        st["g"].zero_()
        st["sums"].zero_()
        st["copy"].wait_stream(main)             # the chunk buffers may still be read by the previous call's kernels
        hp_chunk = _lib.HParams(hp.gamma, hp.lr, hp.alpha, hp.eps, hp.grad_norm_clip, 0, 1, hp.keep_q)
        N, O = src["obs"].shape[2], src["obs"].shape[3]
        S = 1
        if "state" in src:
            for dim in src["state"].shape[2:]:
                S *= int(dim)
        keep = []
        dims = None
        for i, s0 in enumerate(range(lo, hi, chunk)):
            s1 = min(s0 + chunk, hi)
            nb, slot = s1 - s0, i & 1
            with th.cuda.stream(st["copy"]):
                if i >= 2:
                    st["copy"].wait_event(st["done"][slot])
                if host:
                    _lib.gather_episode_steps(src, batch.ep_ids[s0:s1], T, {k: st["bufs"][slot][k][:nb] for k in names},
                                              filled=trim)
                else:
                    for k in names:
                        st["bufs"][slot][k][:nb].copy_(src[k][s0:s1], non_blocking=True)
                st["copied"][slot].record(st["copy"])
            main.wait_event(st["copied"][slot])
            fields = {k: st["bufs"][slot][k][:nb] for k in names}
            dims = self._layout_dims(B=nb, T=T, O=O, S=S)
            pb = _lib.make_batch(fields, need_state=(a.mixer == "qmix"), keep=keep, dims=dims, entry=_lib.ENTRY_TRAIN_STEP)
            need = self._ensure_workspace(self._layout_dims(B=chunk, T=T, O=O, S=S), dev)
            _lib.check(L.pmb_qlearner_train_step(C.byref(dims), C.byref(pb), C.byref(hp_chunk), _lib.ptr(f["p"]),
                                                 _lib.ptr(f["g"]), _lib.ptr(f["sq"]), _lib.ptr(f["target"]),
                                                 _lib.ptr(self._workspace), need, _lib.ptr(self._stats),
                                                 _lib.stream_ptr(dev)), "pmb_qlearner_train_step")
            st["g"].add_(f["g"][:n])
            st["sums"].add_(self._stats[:5])
            st["done"][slot].record(main)
        if host:
            batch.ep_ids.record_stream(st["copy"])
            _mark_buffer_read(batch, st["copy"])
        f["g"][:n].copy_(st["g"])
        self._stats[:5].copy_(st["sums"])
        if not dp:
            _lib.check(L.pmb_clip_rmsprop_update(n, _lib.ptr(f["p"]), _lib.ptr(f["g"]), _lib.ptr(f["sq"]),
                                                 _lib.ptr(f["target"]), hp.do_target_sync, _lib.ptr(self._stats), hp.lr,
                                                 hp.alpha, hp.eps, hp.grad_norm_clip, _lib.ptr(self._dp_scratch),
                                                 _lib.stream_ptr(dev)), "pmb_clip_rmsprop_update")
        else:
            self._exchange_and_update(hp, f, dev, True)
        return dims

    def train(self, batch, t_env: int, episode_num: int):
        a = self.args
        f = self._ensure_flat()
        dev = f["p"].device
        keep = []
        names = ["obs", "actions", "avail_actions", "reward", "terminated", "filled"]
        if a.mixer == "qmix":
            names.append("state")
        dp = data_parallel.is_active() and getattr(a, "data_parallel", True)
        stream_plan = self._host_stream_plan(batch, dp)
        if stream_plan is not None:
            return self._train_host_batch(batch, names, stream_plan, f, dev, dp, t_env, episode_num)
        fields, ep_index, B, T = self._step_fields(batch, names, dev, dp)
        obs = fields["obs"]
        N, O = obs.shape[2], obs.shape[3]
        S = 1
        if "state" in fields:
            for dim in fields["state"].shape[2:]:            # like QMixer: state_dim = prod(state_shape) (qmix.py:13)
                S *= int(dim)
        dims = self._layout_dims(B=max(B, 1), T=T, O=O, S=S)
        dims.B = B
        pb = _lib.make_batch(fields, need_state=(a.mixer == "qmix"), keep=keep, ep_index=ep_index, dims=dims,
                             entry=_lib.ENTRY_TRAIN_STEP)
        need = self._ensure_workspace(dims, dev) if B > 0 else 0
        if dp and (self._dp_scratch is None or self._dp_scratch.device != dev):
            self._dp_scratch = th.empty(4096, dtype=th.float32, device=dev)

        do_sync = (episode_num - self.last_target_update_episode) / a.target_update_interval >= 1.0
        # the optimiser's (possibly checkpoint-restored) hyper-parameters, like torch's param_groups (q_learner.py:30,143)
        od = self.optimiser.defaults
        hp = _lib.HParams(a.gamma, od["lr"], od["alpha"], od["eps"], a.grad_norm_clip, int(do_sync), int(dp),
                          int(getattr(a, "keep_q", 0)))
        if getattr(a, "cuda_graph", False) and not dp and B > 0:
            self._run_graphed(dims, pb, hp, f, need, dev, keep)
        else:
            self._launch(dims, pb, hp, f, need, dev, dp)
        self._after_step(dims, do_sync, t_env, episode_num)

    def _train_host_batch(self, batch, names, stream_plan, f, dev, dp, t_env, episode_num):
        a = self.args
        if self._dp_scratch is None or self._dp_scratch.device != dev:
            self._dp_scratch = th.empty(4096, dtype=th.float32, device=dev)
        do_sync = (episode_num - self.last_target_update_episode) / a.target_update_interval >= 1.0
        od = self.optimiser.defaults
        hp = _lib.HParams(a.gamma, od["lr"], od["alpha"], od["eps"], a.grad_norm_clip, int(do_sync), int(dp),
                          int(getattr(a, "keep_q", 0)))
        dims = self._train_streamed(batch, names, stream_plan, f, dev, dp, hp)
        self._after_step(dims, do_sync, t_env, episode_num)

    def _after_step(self, dims, do_sync, t_env, episode_num):
        a = self.args
        self.optimiser.step_count += 1
        if hasattr(self.mac, "params_changed"):
            self.mac.params_changed()          # the rollout path caches packed weight images between updates
        self.last_stats = self._stats
        self._last_dims = dims

        if do_sync:
            self.last_target_update_episode = episode_num
            self.logger.console_logger.info("Updated target network")

        if t_env - self.log_stats_t >= a.learner_log_interval:
            st = self._stats.tolist()                                            # one D2H sync
            mask_elems = st[_lib.STAT_IDS["mask_sum"]]
            self.logger.log_stat("loss", st[_lib.STAT_IDS["td2_sum"]] / mask_elems, t_env)
            self.logger.log_stat("grad_norm", st[_lib.STAT_IDS["grad_norm"]], t_env)
            self.logger.log_stat("td_error_abs", st[_lib.STAT_IDS["tdabs_sum"]] / mask_elems, t_env)
            self.logger.log_stat("q_taken_mean", st[_lib.STAT_IDS["qtaken_sum"]] / (mask_elems * a.n_agents), t_env)
            self.logger.log_stat("target_mean", st[_lib.STAT_IDS["target_sum"]] / (mask_elems * a.n_agents), t_env)
            self.log_stats_t = t_env

    # ---- CUDA graph of the whole step (args.cuda_graph) ---------------------------------------
    # The C ABI allocates nothing and takes the stream as an argument, so the ~25 launches of a step capture into one
    # graph.  At the small BASELINE configs (3m / 32, 2s3z / 1024) launch latency, not the kernels, bounds the step.
    # A graph is keyed on everything its launches bake in: dims, every field pointer / stride, the hyper-parameters
    # and the target-sync flag - so a batch that lives somewhere else (or needed a dtype / layout conversion, which
    # yields fresh tensors) simply misses the cache.  First sight of a key runs eagerly, the second captures and
    # replays, later ones replay.  Copies / conversions of the inputs stay outside the graph, ordered before it on the
    # same stream.
    def _run_graphed(self, dims, pb, hp, f, need, dev, keep):
        key = (tuple(getattr(dims, k) for k, _ in dims._fields_), tuple(getattr(pb, k) for k, _ in pb._fields_),
               pb.state_dtype, pb.avail_dtype, tuple(getattr(hp, k) for k, _ in hp._fields_), f["p"].data_ptr(), self._workspace.data_ptr(),
               self._stats.data_ptr())
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) >= 16:                     # bounded cache (ring of replay batches etc.)
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = "seen"
            return self._launch(dims, pb, hp, f, need, dev, False)
        if entry == "seen":
            g = th.cuda.CUDAGraph()
            th.cuda.synchronize(dev)
            with th.cuda.graph(g):
                self._launch(dims, pb, hp, f, need, dev, False)
            entry = self._graphs[key] = (g, list(keep))
        entry[0].replay()

    def stats(self):
        """The 5 logged scalars + grad_norm of the latest step as python floats (syncs)."""
        st = self.last_stats.tolist()
        m = st[0]
        n = self.args.n_agents
        return dict(loss=st[1] / m, grad_norm=st[5], td_error_abs=st[2] / m, q_taken_mean=st[3] / (m * n),
                    target_mean=st[4] / (m * n), mask_sum=m, clip_coef=st[7])

    def _update_targets(self):
        self.target_mac.load_state(self.mac)
        if self.mixer is not None:
            self.target_mixer.load_state_dict(self.mixer.state_dict())
        self.logger.console_logger.info("Updated target network")

    def cuda(self):
        self.mac.cuda()
        self.target_mac.cuda()
        if self.mixer is not None:
            self.mixer.cuda()
            self.target_mixer.cuda()
        self._ensure_flat()

    def save_models(self, path):
        self.mac.save_models(path)
        if self.mixer is not None:
            th.save(self.mixer.state_dict(), "{}/mixer.th".format(path))
        th.save(self.optimiser.state_dict(), "{}/opt.th".format(path))

    def load_models(self, path):
        self.mac.load_models(path)
        # Like the reference (q_learner.py:137-143): the target MAC loads the online weights
        # and the target mixer is left as it is.
        self.target_mac.load_models(path)
        if self.mixer is not None:
            self.mixer.load_state_dict(th.load("{}/mixer.th".format(path), map_location=lambda storage, loc: storage))
        self.optimiser.load_state_dict(th.load("{}/opt.th".format(path), map_location=lambda storage, loc: storage))
