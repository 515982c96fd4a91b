"""PPO / PPO-SimHash / RND / ICM learners with the reference's entry points, on the GPU.

Mirrors algorithms.py of the reference: BaseAlgorithm (:22-118), PPO (:121-308), PPO_RND (:310-543),
PPO_ICM (:546-756).  Constructor keyword names and defaults, `collect_samples()`, `train()` and
`learn()` keep their meaning; hyper-parameter dictionaries from the reference's hyperparameters.py
splat into these constructors unchanged.  What differs:
  * the env layer is out of scope (SURVEY §2 rows 19-20): pass `env=` (anything with num_envs,
    observation_space, action_space, reset(), step()) instead of `env_id` only;
  * train() runs the fused path  shuffle-gather -> advantage stats -> batched MLP forward ->
    fused PPO loss fwd+bwd -> MLP backward -> clip+Adam, all in libppx.so, and reads the loss
    scalars back ONCE per train() (the reference syncs 4-5 .item() per minibatch);
  * losses are returned per minibatch in `self.last_losses` ([steps, 5] numpy) and their means in
    `self.train_stats` under the reference's logger keys; pass `logger=` (a module/object with
    .record) to keep logging through the reference's logger.
The host numpy RNG is consumed in exactly the reference's order: one permutation per epoch
(buffer.py:239) and, for RND, one randn() per minibatch (algorithms.py:468).
"""
import ctypes as C
import time
from collections import deque

import numpy as np
import torch

from . import _lib as L
from . import dist as D
from .buffer import (RolloutStorage, IntrinsicStorage, HostRngStream, DevicePartners, device_shuffle_default,
                     rng_states_equal, _dev)
from .models import Policy, RndNetwork, IntrinsicCuriosityModule, ActionConverter, _Scratch
from .util import RunningMeanStd, normalize_obs


class BaseAlgorithm(object):
    """algorithms.py:22-118."""

    def __init__(self, env_id, lr, nstep, batch_size, n_epochs, gamma, gae_lam, clip_range, ent_coef, vf_coef,
                 max_grad_norm, env=None, device="cuda", logger=None):
        if env is None:
            raise ValueError("ppx accelerates the learner hot path only: construct the vectorised env yourself "
                             "and pass env=... (the reference builds it from env_id, algorithms.py:52)")
        self.env_id = env_id
        self.env = env
        self.device = torch.device(device)
        self.num_envs = env.num_envs
        self.state_dim = env.observation_space.shape[0]
        self.action_converter = ActionConverter(env.action_space)
        self.discrete = self.action_converter.action_type == "Discrete"
        self.lr, self.nstep, self.batch_size, self.n_epochs = lr, nstep, batch_size, n_epochs
        self.gamma, self.gae_lam, self.clip_range = gamma, gae_lam, clip_range
        self.ent_coef, self.vf_coef, self.max_grad_norm = ent_coef, vf_coef, max_grad_norm
        self._ep_pending, self._ep_free, self._ep_log = [], [], None   # device episode log (episode_stats() envs)
        self.ep_info_buffer = deque(maxlen=50)
        self._n_updates = 0
        self.num_timesteps = 0
        self._episodes_dev = None              # device path: episodes counted on the GPU, resolved when num_episodes is read
        self.num_episodes = 0
        self.obs_rms = RunningMeanStd(shape=(self.state_dim,), device=self.device, sharded=True)
        self.logger = logger
        self.train_stats = {}
        self.last_losses = None
        self._scratch = _Scratch(self.device)
        self._stats = torch.zeros(4, dtype=torch.float64, device=self.device)
        self._sums = torch.zeros(32, dtype=torch.float64, device=self.device)
        self._branch = torch.zeros(4, dtype=torch.float64, device=self.device)
        self.scale_batch_with_world = True     # sharded runs: batch_size is per rank (weak scaling)
        # sharded minibatch composition: "global" (default; exact) = every rank draws the SAME permutation over the
        # global [T, W*N] index space -- the reference's np.random.permutation(T*N_total), bit for bit -- the rollout
        # is replicated once per pass (all-gather of the env shards) and rank r takes rows [r*B, (r+1)*B) of every
        # global minibatch: a W-GPU run equals the 1-GPU run over all envs, shapes are static (CUDA graphs);
        # "local" = every rank shuffles its own rollout with its own numpy stream (the usual data-parallel sampler;
        # NOT the reference's global permutation -- a labelled secondary number in bench.py)
        self.shard_shuffle = "global"
        self._mrec = None
        self._spec = None                      # (HostRngStream, rng snapshot) pre-drawn for the next train() call
        self.speculative_shuffle = True
        self._px = False                       # PeerExchange (NVLink peer-memory kernels) | None; False = not probed yet
        self.use_cuda_graph = True             # replay the per-minibatch launch sequence as one CUDA graph
        self._graphs, self._graph_state = {}, None
        self._cursor = torch.zeros(1, dtype=torch.int64, device=self.device)    # optimiser step of the running train() call
        self._losses_buf = None                # [steps, 8] f64, persistent (graphs keep its address)
        self._readback = None                  # pinned host copy of the loss log (+ sharded status words)
        self._perm_all, self._perm_events, self._perm_keep, self._copy_stream = None, [], [], None
        self._perm_gen = 0
        self._perm_sets, self._next_set = None, 0               # two staging sets: the speculative stream of the NEXT pass fills the other one
        self._perm_j, self._perm_ws = None, None
        self._glob = None                      # sharded "global": the all-gathered rollout [W, T, N, ...] per field
        self.rng_wait_s = 0.0                  # cumulative host time train() spent waiting for permutations
        self.device_shuffle = device_shuffle_default()         # swaps of the epoch shuffle applied on the GPU (shuffle_dev.cu)

    def __del__(self):
        sp = getattr(self, "_spec", None)
        if sp is not None:
            sp[0].cancel()

    @property
    def num_episodes(self):
        """Episodes ended so far.  On the device path the count since the value was last set lives on the GPU
        (collect_samples never syncs for it); reading it synchronises once."""
        n = self._num_episodes
        if self._episodes_dev is not None:
            n += int(self._episodes_dev.item())
        return n

    @num_episodes.setter
    def num_episodes(self, value):
        self._num_episodes = value
        if self._episodes_dev is not None:
            self._episodes_dev.zero_()

    @property
    def ep_info_buffer(self):
        """The last finished episodes as {"r": return, "l": length} (the reference's Monitor entries).  On the device path
        with an env that has `episode_stats()`, each rollout's newest episodes are selected on the GPU and copied to pinned
        memory without blocking; reading the buffer appends them, waiting for the copy if it is still running."""
        self._ep_resolve(wait=True)
        return self._ep_info_buffer

    @ep_info_buffer.setter
    def ep_info_buffer(self, value):
        self._ep_free += self._ep_pending
        self._ep_pending = []
        self._ep_info_buffer = value

    def _ep_resolve(self, wait):
        """Append the pending episode-log tails in rollout order (wait=False: only those whose copy has landed)."""
        while self._ep_pending:
            slot = self._ep_pending[0]
            if wait:
                slot["event"].synchronize()
            elif not slot["event"].query():
                return
            K = slot["ret"].numel()
            n = int(slot["len"][K])
            rets, lens = slot["ret"][:n].tolist(), slot["len"][:n].tolist()   # newest first
            self._ep_info_buffer.extend({"r": round(r, 6), "l": int(l)} for r, l in zip(rets[::-1], lens[::-1]))
            self._ep_free.append(self._ep_pending.pop(0))

    def _episode_log_begin(self):
        """Device path: the env's `episode_stats` (None if it has none) and the [T, N] log of this rollout."""
        stats = getattr(self.env, "episode_stats", None)
        if not callable(stats):
            return None
        T, N = self.rollout.buffer_size, self.num_envs
        if self._ep_log is None or tuple(self._ep_log[0].shape) != (T, N):
            self._ep_log = (torch.zeros(T, N, dtype=torch.float64, device=self.device),
                            torch.zeros(T, N, dtype=torch.int64, device=self.device))
        self._ep_resolve(wait=False)
        return stats

    def _episode_log_step(self, stats, t):
        """One launch after record_step: the finished envs' (return, length) into row t of the log."""
        ret, lens = stats()
        if not (ret.is_cuda and ret.dtype == torch.float64 and lens.dtype == torch.int64 and ret.is_contiguous()
                and lens.is_contiguous() and ret.numel() == lens.numel() == self.num_envs):
            raise TypeError("env.episode_stats() must return contiguous CUDA (f64 [N] returns, int64 [N] lengths)")
        L.call("ppx_episode_log_record", self.rollout.masks[t].data_ptr(), ret.data_ptr(), lens.data_ptr(), self.num_envs,
               self._ep_log[0][t].data_ptr(), self._ep_log[1][t].data_ptr(), L.stream())

    def _episode_log_end(self):
        """One launch after the rollout: the newest maxlen finished episodes (the rollout's masks are the done flags), then
        an asynchronous copy to pinned memory; `ep_info_buffer` appends them when read."""
        masks = self.rollout.masks
        K = self._ep_info_buffer.maxlen or masks.numel()
        slot = next((s for s in self._ep_free if s["ret"].numel() == K), None)
        if slot is None:
            slot = dict(ret=torch.zeros(K, dtype=torch.float64).pin_memory(), len=torch.zeros(K + 1, dtype=torch.int64).pin_memory(),
                        d_ret=torch.zeros(K, dtype=torch.float64, device=self.device),
                        d_len=torch.zeros(K + 1, dtype=torch.int64, device=self.device), event=torch.cuda.Event())
        else:
            self._ep_free.remove(slot)
        L.call("ppx_episode_log_tail", masks.data_ptr(), self._ep_log[0].data_ptr(), self._ep_log[1].data_ptr(), masks.numel(), K,
               slot["d_ret"].data_ptr(), slot["d_len"].data_ptr(), slot["d_len"].data_ptr() + 8 * K, L.stream())
        slot["ret"].copy_(slot["d_ret"], non_blocking=True)
        slot["len"].copy_(slot["d_len"], non_blocking=True)
        slot["event"].record()
        self._ep_pending.append(slot)

    def _reset_env(self):
        """env.reset().  An env whose observations come back as CUDA tensors is stepped on the device path of
        collect_samples (INTEGRATION.md §4: CUDA actions in, CUDA observations / rewards / dones out); numpy envs keep the
        reference's loop."""
        self.last_obs = self.env.reset()
        self.device_env = isinstance(self.last_obs, torch.Tensor) and self.last_obs.is_cuda
        if self.device_env and self._episodes_dev is None:
            self._episodes_dev = torch.zeros(1, dtype=torch.int64, device=self.device)

    # ---- shared pieces of the fused update --------------------------------------------------
    def _record(self, key, value):
        self.train_stats[key] = value
        if self.logger is not None:
            self.logger.record(key, value)

    def update_info_buffer(self, infos, dones=None):
        for info in infos:
            ep = info.get('episode')
            if ep is not None:
                self.ep_info_buffer.extend([ep])

    def _loss_workspace(self):
        return self._scratch.get("ppo_loss_ws", L.call("ppx_ppo_loss_workspace", 0, 0) // 8 + 1, torch.float64)

    def _gather_with_stats(self, ro, sl, bufs, dual=False, opts=None, B=None, sources=None):
        """Minibatch gather; the advantage moments (algorithms.py:219, :431-434) come out of the same launch."""
        B = sl.numel() if B is None else int(B)
        n_stat = opts.stat_n if (opts is not None and opts.stat_n > 0) else B
        self._stats_merged = False
        if D.world_size() > 1 and sources is None and opts is not None and n_stat >= 2:
            px = self._peer_exchange()                          # per-rank shuffles: merge the moments inside the gather launch
            if px is not None:
                opts.W, opts.rank, opts.peer_moments_host = px.W, px.rank, C.cast(px.peer_xm, C.c_void_p)
                opts.seq_dev, opts.status_dev = px.seq_moments, px.status_ptr
                self._stats_merged = True
        stats = [('advantages', self._stats.data_ptr())] + ([('int_advantages', self._stats.data_ptr() + 16)] if dual else [])
        ro.gather_into(sl, bufs, stats=stats if n_stat >= 2 else None, opts=opts, sources=sources, B=B)
        return n_stat >= 2

    def _policy_step(self, bufs, B, losses_row, dual=False, policy_weight=1.0, int_vf_coef=0.0, B_total=0, stats_ready=False,
                     stats_global=False, row_dev=None, row_hold=False, fuse_adam=False):
        """One minibatch: forward, fused loss fwd+bwd, backward.  Gradients land in policy.bank.grad.
        Sharded runs (B_total = rows of the global minibatch) exchange only the 32 loss partial sums (and, with
        per-rank shuffles, the advantage moments); the caller all-reduces the flat gradient.  `losses_row` is the
        base of the loss log: with `row_dev` (device step counter) row *row_dev is written and the counter advanced
        (unless row_hold).  fuse_adam: clip + Adam run inside the backward's reduce kernel (single GPU, fused MLP)."""
        pol, sc = self.policy, self._scratch
        A = pol.action_dim
        obs = bufs['observations'][:B]
        outs = pol.forward_raw(obs)
        adv = bufs['advantages'][:B]
        sharded = D.world_size() > 1
        if not stats_ready:
            L.call("ppx_mean_std", adv.data_ptr(), B, self._stats.data_ptr(), L.stream())
            if dual:
                iadv = bufs['int_advantages'][:B]
                L.call("ppx_mean_std", iadv.data_ptr(), B, self._stats.data_ptr() + 16, L.stream())
        if sharded and not stats_global and not (stats_ready and getattr(self, "_stats_merged", False)):
            self._merge_stats(B, dual)
        d_actor = sc.get("d_actor", B * A)[:B * A].view(B, A)
        cfg = L.PpoCfg(B, int(B_total), A, int(self.discrete), int(dual), float(self.clip_range), float(self.ent_coef),
                       float(self.vf_coef), float(int_vf_coef), float(policy_weight), row_dev, int(bool(row_hold)))
        g = lambda k: bufs[k][:B].data_ptr() if k in bufs else None
        ws = self._loss_workspace().data_ptr()
        head_args = (C.byref(cfg), outs[0].data_ptr(), pol.bank.p("action_log_std"), g('actions'),
                     g('old_log_probs'), adv.data_ptr(), self._stats.data_ptr(), outs[1].data_ptr(), g('old_values'),
                     g('returns'), g('int_advantages'), self._stats.data_ptr() + 16,
                     outs[2].data_ptr() if dual else None, g('int_values'), g('int_returns'), d_actor.data_ptr())
        self._adam_fused = False
        if pol.mlp.fused():
            # head + partial sums (+ loss scalars / branch when single-GPU) in ONE launch; the value-head gradients are
            # evaluated inside the fused MLP backward from the branch weights.  Sharded: the 32 partial sums are
            # all-reduced (256 bytes) by the finalising block itself so the max-of-means branch is the global one.
            Bt = int(B_total) if B_total else B
            px = self._peer_exchange() if sharded else None
            if px is not None:                                  # the finalising block exchanges the sums over peer memory
                cfg.W, cfg.rank, cfg.peer_sums_host = px.W, px.rank, C.cast(px.peer_xs, C.c_void_p)
                cfg.seq_dev, cfg.status_dev = px.seq[1], px.status_ptr
            if not sharded or px is not None:
                L.call("ppx_ppo_loss_head_final", *head_args, pol.bank.g("action_log_std"), losses_row,
                       self._branch.data_ptr(), ws, L.stream())
            else:                                               # no peer memory: NCCL all-reduce between head and finalize
                L.call("ppx_ppo_loss_head", *head_args, self._sums.data_ptr(), ws, L.stream())
                D.all_reduce_sum_(self._sums)
                L.call("ppx_ppo_loss_finalize", C.byref(cfg), self._sums.data_ptr(), pol.bank.p("action_log_std"),
                       pol.bank.g("action_log_std"), losses_row, self._branch.data_ptr(), L.stream())
            vh = {1: (outs[1], bufs['old_values'][:B], bufs['returns'][:B], self._branch.data_ptr(),
                      float(policy_weight) * float(self.vf_coef))}
            if dual:
                vh[2] = (outs[2], bufs['int_values'][:B], bufs['int_returns'][:B], self._branch.data_ptr() + 16,
                         float(int_vf_coef))
            # single GPU: the reduce kernel also leaves the clip_grad_norm_ partials, and (fuse_adam) its last block
            # applies clip + Adam to the whole bank -- no sumsq launch, no Adam launch
            # sharded with peer memory (fuse_adam): the same tail also all-reduces the gradient (ppx_fused_adam.W >= 2)
            px = self._peer_exchange() if sharded else None
            fuse_here = fuse_adam and (not sharded or (px is not None and px.flag_blocks > 0))
            self._pre_sumsq = (self.max_grad_norm > 0 and not sharded) or fuse_here
            adam = None
            if fuse_here:
                adam = pol.bank.fused_adam(self.lr, self.max_grad_norm, extra_name="action_log_std", px=px)
                self._adam_fused = True
            pol.mlp.backward([d_actor, None] + ([None] if dual else []), value_heads=vh, clip_range=self.clip_range,
                             B_total=Bt, with_sumsq=self._pre_sumsq, adam=adam)
            return
        self._pre_sumsq = False
        d_val = sc.get("d_val", B)[:B].view(B, 1)
        d_ival = sc.get("d_ival", B)[:B].view(B, 1)
        L.call("ppx_ppo_loss_head", *head_args, self._sums.data_ptr(), ws, L.stream())
        if sharded:
            D.all_reduce_sum_(self._sums)
        L.call("ppx_ppo_loss_finish", C.byref(cfg), self._sums.data_ptr(), pol.bank.p("action_log_std"),
               outs[1].data_ptr(), g('old_values'), g('returns'), outs[2].data_ptr() if dual else None,
               g('int_values'), g('int_returns'), pol.bank.g("action_log_std"), d_val.data_ptr(),
               d_ival.data_ptr() if dual else None, losses_row, ws, L.stream())
        pol.mlp.backward([d_actor, d_val] + ([d_ival] if dual else []))

    def _peer_exchange(self):
        """Lazily move the policy bank's gradient vector, the loss partial sums and the moment records into symmetric
        peer memory so the per-minibatch exchanges run as ppx kernels over NVLink (p2p.cu) instead of NCCL."""
        if self._px is False:
            self._px = None
            if D.world_size() > 1 and self.policy.mlp.fused():
                bank = self.policy.bank
                mlp = self.policy.mlp
                outs = (C.c_int * mlp.G)(*[int(o) for o in mlp.outs])
                blocks = int(L.call("ppx_mlp3_fused_adam_blocks", int(mlp.D), int(mlp.h), int(mlp.G), outs))
                px = D.peer_exchange_or_none(bank.size, self.device, L.call("ppx_p2p_max_params"), flag_blocks=blocks)
                if px is not None:
                    px.grad.copy_(bank.grad)
                    bank.grad = px.grad                         # kernels now write the local gradient into peer-visible memory
                    self.policy.mlp._fa = None                  # cached gradient pointers are stale
                    self._sums = px.sums[:32]
                    self._sums_global = torch.zeros(32, dtype=torch.float64, device=self.device)
                    self._px = px
                    self._graphs.clear()
        return self._px

    def _merge_stats(self, B, dual):
        """Per-rank shuffles ("local"): local {mean, std} -> global, through one exchange of {n, mean, M2} records."""
        W = D.world_size()
        px = self._peer_exchange()
        if px is not None:
            L.call("ppx_moments_pack", self._stats.data_ptr(), B, px.rec.data_ptr(), L.stream())
            if dual:
                L.call("ppx_moments_pack", self._stats.data_ptr() + 16, B, px.rec.data_ptr() + 24, L.stream())
            L.call("ppx_p2p_moments_merge", px.peer_rec, px.peer_flags[0], W, px.rank, px.seq[0], px.status_ptr,
                   2 if dual else 1, self._stats.data_ptr(), L.stream())
            return
        if self._mrec is None or self._mrec_all.shape[0] != W:
            self._mrec = torch.zeros(6, dtype=torch.float64, device=self.device)
            self._mrec_all = torch.zeros(W, 6, dtype=torch.float64, device=self.device)
        L.call("ppx_moments_pack", self._stats.data_ptr(), B, self._mrec.data_ptr(), L.stream())
        if dual:
            L.call("ppx_moments_pack", self._stats.data_ptr() + 16, B, self._mrec.data_ptr() + 24, L.stream())
        D.all_gather_into(self._mrec_all, self._mrec)
        # records of one stream are strided by 6 doubles in the gathered buffer: merge from a compact copy
        a = self._mrec_all[:, 0:3].contiguous()
        L.call("ppx_moments_merge", a.data_ptr(), W, self._stats.data_ptr(), L.stream())
        if dual:
            b = self._mrec_all[:, 3:6].contiguous()
            L.call("ppx_moments_merge", b.data_ptr(), W, self._stats.data_ptr() + 16, L.stream())

    def _hp_state(self):
        """Everything a captured graph bakes into kernel arguments or addresses: the scalar hyper-parameters (a schedule
        that changes lr / clip_range between train() calls must not replay stale values) and the scratch generation (a
        buffer that was re-allocated since the capture leaves the graph with a dangling pointer)."""
        return (self.lr, self.clip_range, self.ent_coef, self.vf_coef, self.max_grad_norm, self.batch_size, self.n_epochs,
                getattr(self, "int_lr", None), getattr(self, "int_vf_coef", None), getattr(self, "policy_weight", None),
                getattr(self, "beta", None), self.shard_shuffle, D.world_size(), _Scratch.generation)

    def _graph_call(self, key, fn):
        """Run fn() -- a fixed sequence of libppx launches (and NCCL collectives when sharded without peer memory) on
        static buffers -- through a CUDA graph: eager the first time a key is seen (allocations settle), captured the
        second time, replayed afterwards.  Captured graphs are dropped whenever `_hp_state()` changes."""
        if not self.use_cuda_graph:
            return fn()
        st = self._hp_state()
        if st != self._graph_state:
            self._graphs.clear()
            self._graph_state = st
        ent = self._graphs.get(key)
        if ent is None:
            self._graphs[key] = "warm"
            fn()
            if self._hp_state() != st:                          # the warm pass itself grew a buffer: warm once more
                self._graph_state = self._hp_state()
            return
        if ent == "warm":
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):   # the RNG worker thread may pin memory meanwhile
                fn()
            ent = (g, L.launch_count() - n0)
            L.extra_launches -= ent[1]                      # the capture pass launched nothing
            self._graphs[key] = ent
        ent[0].replay()
        L.extra_launches += ent[1]

    def _rng_script(self, ro, randn_per_minibatch=False):
        total, Bg, n_mb = self._train_geometry(ro)
        script = []
        for _ in range(self.n_epochs):
            script.append(('perm', total))
            script += [('randn',)] * (n_mb if randn_per_minibatch else 0)
        return script

    def _rng_open(self, script):
        """The RNG stream of this train() call.  If the stream started speculatively at the end of the previous call was
        seeded with exactly the state np.random is in now (nobody drew in between) and has the same script, its
        permutations are already waiting (the first ones already staged on the device); otherwise it is dropped and a
        fresh stream starts from the current state.  Either way the draws are those the reference would make from this
        state."""
        cur = np.random.get_state()
        sp, self._spec = self._spec, None
        if sp is not None:
            stream, snapshot = sp
            if (stream.script == list(script) and rng_states_equal(cur, snapshot) and stream.err is None
                    and stream.device_apply == self._device_apply() and stream.generation == self._perm_gen):
                return stream
            stream.cancel()
            stream.t1.join()                                    # its uploader must not queue anything after the new stream's
        return self._new_stream(script, cur)

    def _new_stream(self, script, state):
        """A HostRngStream whose draw thread also stages every permutation on the device as soon as it is drawn (H2D of
        the partner list + the parallel swaps, on the copy stream) into the staging set this stream owns."""
        set_idx, self._next_set = self._next_set, self._next_set ^ 1
        total = next((int(op[1]) for op in script if op[0] == 'perm'), 0)
        up = None
        if self._device_apply() and self._perm_j is not None and 2 <= total <= (1 << 24):
            dst_all, js, ws, cs = self._perm_sets[set_idx], self._perm_j, self._perm_ws, self._copy_stream
            evs = self._stage_events[set_idx]

            def up(k, dp):                                      # runs on the draw thread: one GIL-free C call
                copied, ready = evs[k]
                L.call("ppx_np_shuffle_stage", dp.j.data_ptr(), total, js[k & 1].data_ptr(), ws.data_ptr(),
                       dst_all.data_ptr() + 8 * k * total, cs.cuda_stream, copied.cuda_event, ready.cuda_event)
                dp.ready = ready
                dp.release(copied)                              # the pinned partner buffer is free once the copy has run
                return copied
        stream = HostRngStream(script, state=state, device_apply=self._device_apply(), uploader=up)
        stream.set_idx, stream.generation = set_idx, self._perm_gen
        return stream

    def _device_apply(self):
        """The swaps of the shuffle run on the GPU (only the draws ARE the RNG stream); the permutation is only ever
        needed on the device."""
        return bool(self.device_shuffle)

    def _rng_close(self, rng, speculate=True):
        """Commit the consumed draws to the global numpy RNG and pre-draw the next call's stream from there."""
        final = rng.final_state()
        np.random.set_state(final)
        self._last_rng = rng
        if speculate and self.speculative_shuffle:
            self._spec = (self._new_stream(rng.script, final), final)

    def _train_geometry(self, ro):
        """(indices per permutation, rows of a global minibatch, minibatches per epoch)."""
        W = D.world_size() if self.shard_shuffle == "global" else 1
        total = ro.buffer_size * ro.n_envs * W
        Bg = min(self.batch_size * (W if self.scale_batch_with_world else 1), total)
        return total, Bg, -(-total // Bg)

    def _begin_train(self, ro, randn_per_minibatch=False):
        """Open the RNG stream, size the persistent per-call buffers (loss log, all-epoch permutation staging), zero the
        device step cursor and -- sharded "global" -- replicate the rollout.  Returns the RNG stream."""
        ro.await_load()                                         # load_rollout(overlap=True): the graphs below cannot wait for it
        total, Bg, n_mb = self._train_geometry(ro)
        steps = self.n_epochs * n_mb
        if self._losses_buf is None or self._losses_buf.shape[0] != steps:
            self._losses_buf = torch.zeros(steps, 8, dtype=torch.float64, device=self.device)
            _Scratch.generation += 1
        self._losses_buf.zero_()
        self._cursor.zero_()
        if self._perm_sets is None or self._perm_sets[0].numel() != self.n_epochs * total:
            self._perm_sets = [torch.empty(self.n_epochs * total, dtype=torch.int64, device=self.device) for _ in range(2)]
            self._copy_stream = self._copy_stream or torch.cuda.Stream(device=self.device)
            self._perm_j = None
            if self._device_apply() and 2 <= total <= (1 << 24):
                self._perm_j = [torch.empty(total, dtype=torch.int32, device=self.device) for _ in range(2)]
                self._perm_ws = torch.empty(L.call("ppx_np_shuffle_apply_device_workspace", total), dtype=torch.uint8, device=self.device)
            # events of the staging steps (copy done, permutation ready), recorded once so that their handles exist
            self._stage_events = [[(torch.cuda.Event(), torch.cuda.Event()) for _ in range(self.n_epochs)] for _ in range(2)]
            for evs in self._stage_events:
                for pair in evs:
                    for e in pair:
                        e.record(self._copy_stream)
            _Scratch.generation += 1
            self._perm_gen += 1                                 # retires a speculative stream that stages into the old sets
        self._perm_events, self._perm_keep = [None] * self.n_epochs, []
        rng = self._rng_open(self._rng_script(ro, randn_per_minibatch))
        self._perm_set = rng.set_idx
        self._perm_all = self._perm_sets[rng.set_idx]
        if rng.uploader is None:                                # uploads issued by this thread: after the previous readers of the set
            self._copy_stream.wait_stream(torch.cuda.current_stream())
        self._rng_check = None
        if D.world_size() > 1 and self.shard_shuffle == "global":
            # every rank must draw the SAME permutation: exchange a digest of the numpy state the stream starts from
            # (asynchronous; compared in _finish_train, where the host synchronises anyway)
            st = np.random.get_state()
            digest = D.rng_digest(st)
            self._rng_check = D.all_gather_cat(torch.tensor([digest], dtype=torch.int64, device=self.device))
            self._replicate_rollout(ro)
        return rng

    def _replicate_rollout(self, ro):
        """Sharded "global": all-gather the env shards of every RolloutSample source array -> [W, T, N, ...] (one
        collective per field and pass; the gather kernel decodes the global flat index into this layout)."""
        W = D.world_size()
        srcs = sorted({src for _, src in ro._fields})
        if self._glob is None or any(self._glob[k].shape[1:] != getattr(ro, k).shape for k in srcs):
            self._glob = {k: torch.empty((W,) + tuple(getattr(ro, k).shape), dtype=getattr(ro, k).dtype, device=self.device) for k in srcs}
            _Scratch.generation += 1
        for k in srcs:
            D.all_gather_into(self._glob[k], getattr(ro, k))

    def _perm_upload(self, rng, epoch, total):
        """Stage epoch `epoch`'s permutation in its slice of the all-epoch device buffer, on the copy stream (the H2D
        copy and the device-side swaps overlap the previous epoch's kernels)."""
        t0 = time.perf_counter()
        perm = rng.next()                                       # pinned int64 [total], or the partner list (DevicePartners)
        self.rng_wait_s += time.perf_counter() - t0             # host time blocked on the (sequential) numpy RNG stream
        on_device = isinstance(perm, DevicePartners)
        if on_device and perm.ready is not None:                # already staged by the stream's draw thread
            self._perm_events[epoch] = perm.ready
            return
        dst = self._perm_all[epoch * total:(epoch + 1) * total]
        with torch.cuda.stream(self._copy_stream):
            if on_device:                                       # 4 bytes per index up instead of 8, swaps resolved in parallel on the copy stream
                j = self._perm_j[epoch & 1]
                j.copy_(perm.j, non_blocking=True)
                L.call("ppx_np_shuffle_apply_device", j.data_ptr(), total, 1, self._perm_ws.data_ptr(), dst.data_ptr(), L.stream())
            else:
                dst.copy_(perm, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        if on_device:
            perm.release(ev)                                    # the pinned partner buffer is free once the copy has run
        self._perm_events[epoch] = ev
        self._perm_keep.append(perm)                            # keep the pinned source alive until train() has synchronised

    def _epoch_minibatches(self, ro, rng, epoch=0, n_epochs=1):
        """Yields (gather options, B_local, B_total, graph key, sources) for one epoch.  The indices are the reference's
        own permutation (buffer.py:239, :251-254) over the (global) rollout, staged on the device; the gather kernel
        finds the minibatch's slice through the device step cursor, so one CUDA graph serves every full minibatch.
        Sharded "global": rank r takes rows [lo, lo + b) of each global minibatch from the replicated rollout and the
        advantage moments over ALL its rows (identical on every rank, no exchange)."""
        W, r = D.world_size(), D.rank()
        T, N = ro.buffer_size, ro.n_envs
        glob = W > 1 and self.shard_shuffle == "global"
        total, Bg, n_mb = self._train_geometry(ro)
        if self._perm_events[epoch] is None:
            self._perm_upload(rng, epoch, total)
        torch.cuda.current_stream().wait_event(self._perm_events[epoch])
        for k in range(n_mb):
            bg = min(Bg, total - k * Bg)
            if glob:
                lo, b = D.global_slice(bg, W, r)
                if bg // W < 2:
                    raise RuntimeError(f"a global minibatch of {bg} rows cannot be split over {W} ranks")
                opts = L.GatherOpts(N, -lo, bg, self._cursor.data_ptr(), n_mb, total, Bg)
                yield opts, lo, b, bg, ("g", b, bg, lo, self._perm_set), self._glob
            else:
                opts = L.GatherOpts(0, 0, 0, self._cursor.data_ptr(), n_mb, total, Bg)
                yield opts, 0, bg, (bg * W if W > 1 else 0), ("l", bg, self._perm_set), None
        if epoch + 1 < n_epochs:                                # after this epoch's randn()s were consumed (RND)
            self._perm_upload(rng, epoch + 1, total)

    def _sync_grads(self, bank):
        if D.world_size() > 1:
            D.all_reduce_sum_(bank.grad)

    def _policy_optim_step(self):
        """Gradient exchange + clip + Adam for the policy bank.  Single GPU with the fused MLP: already done by the last
        block of the backward's reduce kernel (`_policy_step(fuse_adam=True)`).  Sharded with peer memory: ONE kernel reads
        every rank's gradient over NVLink, sums in rank order, clips and applies Adam (weights stay bit-identical replicas)."""
        bank = self.policy.bank
        if getattr(self, "_adam_fused", False):
            bank.refresh_tc()
            return
        px = self._peer_exchange() if D.world_size() > 1 else None
        if px is not None:
            n_clip = bank.size if self.max_grad_norm > 0 else 0
            L.call("ppx_p2p_clip_adam", bank.flat.data_ptr(), px.peer_grad, px.peer_flags[2], px.W, px.rank, px.seq[2],
                   px.status_ptr, bank.exp_avg.data_ptr(), bank.exp_avg_sq.data_ptr(), bank.size, float(self.max_grad_norm),
                   n_clip, float(self.lr), 0.9, 0.999, 1e-8, bank.step_dev.data_ptr(), bank.norm_dev.data_ptr(), None,
                   L.stream())
            bank.refresh_tc()
            return
        if getattr(self, "_pre_sumsq", False) and self.max_grad_norm > 0:
            ss, n_ss = self.policy.mlp.sumsq
            bank.adam_step_pre(self.lr, self.max_grad_norm, ss, n_ss, extra_name="action_log_std")
            return
        self._sync_grads(bank)
        bank.adam_step(self.lr, self.max_grad_norm)

    def _fuse_adam_ok(self):
        if not self.policy.mlp.fused() or self.policy.bank.tc_weights:
            return False
        if D.world_size() == 1:
            return True
        px = self._peer_exchange()
        return px is not None and px.flag_blocks > 0

    def _finish_train(self, steps, keys):
        # The only D2H read of train(): loss log (+ the RNG digests and the peer-barrier status when sharded) into PINNED
        # memory, then an event wait.  Not `.cpu()`: a pageable cudaMemcpy waits for the stream inside the driver and keeps
        # other host threads out of the CUDA API meanwhile -- the draw thread of the next pass's stream sat blocked in its
        # first staging call for the ~3 ms this wait lasts (tools/trace_sharded.py), i.e. no look-ahead at all.
        W = D.world_size()
        n_host = steps * 8 + W + 1
        if self._readback is None or self._readback.numel() != n_host:
            self._readback = torch.zeros(n_host, dtype=torch.float64, pin_memory=True)
        rb = self._readback
        rb[:steps * 8].view(steps, 8).copy_(self._losses_buf[:steps], non_blocking=True)
        if self._rng_check is not None:
            rb[steps * 8:steps * 8 + W].copy_(self._rng_check.view(-1).to(torch.float64), non_blocking=True)
        if self._px:
            rb[steps * 8 + W:].copy_(self._px.status.to(torch.float64), non_blocking=True)
        done = torch.cuda.Event()
        done.record()
        done.synchronize()
        losses = rb[:steps * 8].view(steps, 8).numpy().copy()
        if self._rng_check is not None:
            seen = rb[steps * 8:steps * 8 + W].numpy()
            if not (seen == seen[0]).all():
                raise RuntimeError("ppx: shard_shuffle='global' needs the numpy global RNG in the same state on every rank "
                                   "(seed all ranks alike and keep rank-dependent draws off np.random); digests: %s" % seen.tolist())
        self._perm_keep = []
        if self._px and int(rb[steps * 8 + W].item()) != 0:
            raise RuntimeError("ppx: a peer-memory barrier timed out (a rank fell out of the sharded update)")
        self.last_losses = losses
        for i, k in enumerate(keys):
            self._record(k, float(np.mean(losses[:, i])))
        self._n_updates += self.n_epochs

    def _learn_loop(self, total_timesteps, log_interval, reward_target, log_name=None, log_to_file=False):
        """algorithms.py:261-308 / 504-543 / 715-756.  With log_to_file (or when no logger was passed) the run is logged
        through ppx's own logger module, which writes the reference's CSV schema (logger.py:13-52, :222-246)."""
        if log_to_file or self.logger is None:
            from . import logger as ppx_logger
            ppx_logger.configure(log_name or type(self).__name__, str(self.env_id), log_to_file)
            self.logger = ppx_logger
        start, iteration = time.time(), 0
        while self.num_timesteps < total_timesteps:
            self.collect_samples()
            iteration += 1
            if log_interval is not None and iteration % log_interval == 0:
                self._record("time/total timesteps", self.num_timesteps)
                if len(self.ep_info_buffer) > 0 and len(self.ep_info_buffer[0]) > 0:
                    self._record("rollout/ep_rew_mean", np.mean([e["r"] for e in self.ep_info_buffer]))
                    self._record("rollout/num_episodes", self.num_episodes)
                self._record("time/total_time", time.time() - start)
                if self.logger is not None and hasattr(self.logger, "dump"):
                    self.logger.dump(step=self.num_timesteps)
            self.train()
            if reward_target is not None and len(self.ep_info_buffer) > 0 and \
                    np.mean([e["r"] for e in self.ep_info_buffer]) > reward_target:
                break
        return self


class PPO(BaseAlgorithm):
    """algorithms.py:121-308."""

    def __init__(self, *, env_id=None, lr=3e-4, nstep=128, batch_size=128, n_epochs=10, gamma=0.99, gae_lam=0.95,
                 clip_range=0.2, ent_coef=.01, vf_coef=1, max_grad_norm=0.2, hidden_size=128, sim_hash=False,
                 sil=False, env=None, device="cuda", logger=None, hash_bits=16):
        super().__init__(env_id, lr, nstep, batch_size, n_epochs, gamma, gae_lam, clip_range, ent_coef, vf_coef,
                         max_grad_norm, env=env, device=device, logger=logger)
        if sil:
            raise NotImplementedError("self-imitation is dead code in the reference (SURVEY §2 rows 16-17)")
        self.policy = Policy(self.env, hidden_size, device=self.device)
        self.rollout = RolloutStorage(nstep, self.num_envs, self.env.observation_space, self.env.action_space,
                                      gae_lam=gae_lam, gamma=gamma, sim_hash=sim_hash, device=self.device,
                                      hash_bits=hash_bits)
        self._reset_env()
        self.sim_hash = sim_hash
        self.sil = sil

    def collect_samples(self):
        """algorithms.py:166-198."""
        assert self.last_obs is not None
        if self.device_env:
            return self._collect_device()
        self.rollout.reset()
        for _ in range(self.nstep):
            actions, values, log_probs = self.policy.act(self.last_obs)
            obs, rewards, dones, infos = self.env.step(actions.cpu().numpy())
            if any(dones):
                self.num_episodes += sum(dones)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            A = self.action_converter.action_output
            self.rollout.add(self.last_obs, actions.reshape(self.num_envs, A), rewards, values, dones,
                             log_probs.reshape(self.num_envs, A))
            self.last_obs = obs
        self.rollout.compute_returns_and_advantages(values, dones=dones)
        return True

    def _collect_device(self):
        """collect_samples for an env on the GPU, line for line: act_into (forward + one launch writing the step's rows),
        env.step, record_step (one launch) -- no host sync; SimHash once over the whole rollout.  The env's returned
        tensors are never read after the next step() (envs commonly reuse their output buffers)."""
        ro = self.rollout
        ro.reset()
        stats = self._episode_log_begin()
        for _ in range(self.nstep):
            p = ro.pos
            actions, values = self.policy.act_into(self.last_obs, ro)
            obs, rewards, dones, infos = self.env.step(actions)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            ro.record_step(rewards, dones, self._episodes_dev)
            if stats is not None:
                self._episode_log_step(stats, p)
            self.last_obs = obs
        if stats is not None:
            self._episode_log_end()
        if ro.do_hash:
            ro.sim_hash_recorded()
        ro.compute_returns_and_advantages(values, dones=ro.masks[-1])
        return True

    def train(self):
        """algorithms.py:200-259."""
        ro = self.rollout
        rng = self._begin_train(ro)
        total, Bg, n_mb = self._train_geometry(ro)
        bufs = ro._minibatch_buffers(-(-Bg // D.world_size()) if self.shard_shuffle == "global" else Bg)
        fuse = self._fuse_adam_ok()
        step = 0
        for ep in range(self.n_epochs):
            # one graph per EPOCH (the device step cursor finds each minibatch's index slice): the launches of its
            # minibatches follow each other without the ~3 us a graph boundary costs
            mbs = list(self._epoch_minibatches(ro, rng, ep, self.n_epochs))

            def fn(mbs=mbs):
                for opts, lo, b, bt, key, src in mbs:
                    ok = self._gather_with_stats(ro, self._perm_all[lo:], bufs, opts=opts, B=b, sources=src)
                    self._policy_step(bufs, b, self._losses_buf.data_ptr(), B_total=bt, stats_ready=ok, stats_global=src is not None,
                                      row_dev=self._cursor.data_ptr(), fuse_adam=fuse)
                    self._policy_optim_step()
            self._graph_call(("ppo",) + tuple(mb[4] for mb in mbs), fn)
            step += len(mbs)
        ro.generator_ready = True
        self._rng_close(rng)
        self._finish_train(step, ("train/total_loss", "train/policy_gradient_loss", "train/value_loss",
                                  "train/entropy_loss"))

    def learn(self, total_timesteps, log_interval, reward_target=None, log_to_file=False):
        name = "PPO_SimHash" if self.sim_hash else "PPO"                       # algorithms.py:270-275
        return self._learn_loop(total_timesteps, log_interval, reward_target, name, log_to_file)


class PPO_RND(BaseAlgorithm):
    """algorithms.py:310-543."""

    def __init__(self, *, env_id=None, lr=3e-4, nstep=128, batch_size=128, n_epochs=10, gamma=0.99, int_gamma=0.99,
                 gae_lam=0.95, clip_range=0.2, ent_coef=.01, vf_coef=0.5, int_vf_coef=0.5, max_grad_norm=0.2,
                 hidden_size=128, int_hidden_size=128, int_lr=3e-4, rnd_start=1e+3, env=None, device="cuda",
                 logger=None):
        super().__init__(env_id, lr, nstep, batch_size, n_epochs, gamma, gae_lam, clip_range, ent_coef, vf_coef,
                         max_grad_norm, env=env, device=device, logger=logger)
        self.policy = Policy(self.env, hidden_size, intrinsic_model=True, device=self.device)
        self.rnd = RndNetwork(self.state_dim, hidden_size=int_hidden_size, device=self.device)
        self.rollout = IntrinsicStorage(nstep, self.num_envs, self.env.observation_space, self.env.action_space,
                                        gae_lam=gae_lam, gamma=gamma, int_gamma=int_gamma, device=self.device)
        self.int_lr = int_lr
        self.rnd_start = rnd_start
        self.int_vf_coef = int_vf_coef
        self._reset_env()
        self.int_rew_rms = RunningMeanStd(device=self.device, sharded=True)
        self.normalize = True
        self.last_dones = np.array([0 for _ in range(self.num_envs)])
        self._rnd_loss = torch.zeros(1, dtype=torch.float64, device=self.device)

    def rnd_bonus(self, obs):
        """The bonus lines of collect_samples after warm-up (algorithms.py:394-398) for one env step:
        normalise -> (pred-target)^2 -> int_rew_rms.update -> divide.  obs [N,D]; returns [N] f32 CUDA."""
        o = _dev(obs, torch.float32, self.device)
        r = self.rnd.int_reward(o, rms=self.obs_rms)
        return self._normalize_int_rewards(r.view(1, -1)).view(-1)

    def _normalize_int_rewards(self, r):
        """int_rew_rms.update(step batch) + divide (algorithms.py:396-398), step by step in t order, for r [T, N].  Sharded:
        a step's batch is the rewards of ALL W*N envs, so the raw rewards are all-gathered into global env order first
        (T*N*W floats) and every rank runs the identical merge -- moments and divisors equal the 1-GPU ones bit for bit."""
        W, rk = D.world_size(), D.rank()
        T, N = r.shape
        if W == 1:
            L.call("ppx_rnd_normalize_rollout", r.data_ptr(), T, N, self.int_rew_rms.mean_dev.data_ptr(),
                   self.int_rew_rms.var_dev.data_ptr(), self.int_rew_rms.count_dev.data_ptr(), L.stream())
            return r
        full = D.interleave_env_shards(D.all_gather_cat(r.contiguous())).contiguous()          # [T, W*N]
        L.call("ppx_rnd_normalize_rollout", full.data_ptr(), T, W * N, self.int_rew_rms.mean_dev.data_ptr(),
               self.int_rew_rms.var_dev.data_ptr(), self.int_rew_rms.count_dev.data_ptr(), L.stream())
        return full[:, rk * N:(rk + 1) * N].contiguous()

    def rnd_bonus_rollout(self, next_obs):
        """Same arithmetic for a whole rollout at once: next_obs [T,N,D] -> [T,N].  Exact because obs_rms is
        frozen after warm-up and the int-reward moments are merged step by step in t order on device."""
        o = _dev(next_obs, torch.float32, self.device)
        T, N = o.shape[0], o.shape[1]
        r = self.rnd.int_reward(o.reshape(T * N, -1), rms=self.obs_rms)
        return self._normalize_int_rewards(r.view(T, N))

    def collect_samples(self):
        """algorithms.py:367-407."""
        assert self.last_obs is not None
        if self.device_env:
            return self._collect_device()
        self.rollout.reset()
        for _ in range(self.nstep):
            actions, values, int_values, log_probs = self.policy.act(self.last_obs)
            obs, rewards, dones, infos = self.env.step(actions.cpu().numpy())
            if any(dones):
                self.num_episodes += sum(dones)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            A = self.action_converter.action_output
            if (self.num_timesteps / self.num_envs) < self.rnd_start:
                int_rewards = torch.zeros(self.num_envs, device=self.device)
                self.obs_rms.update(self.env.unnormalize_obs(self.last_obs))
            else:
                int_rewards = self.rnd_bonus(obs)
            self.rollout.add(self.last_obs, actions.reshape(self.num_envs, A), rewards, int_rewards, values,
                             int_values, dones, log_probs.reshape(self.num_envs, A))
            self.last_obs = obs
            self.last_dones = dones
        mean_int = self.rollout.compute_returns_and_advantages(values, int_values, dones)
        self._mean_int_reward = mean_int                            # logged lazily (rollout/mean_int_reward, buffer.py:335)
        return True

    def _collect_device(self):
        """collect_samples for an env on the GPU (see PPO._collect_device).  The warm-up statistics read the observation
        from the rollout row, not from the env's (possibly reused) tensor."""
        ro = self.rollout
        ro.reset()
        stats = self._episode_log_begin()
        for _ in range(self.nstep):
            p = ro.pos
            actions, values, int_values = self.policy.act_into(self.last_obs, ro)
            obs, rewards, dones, infos = self.env.step(actions)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            if (self.num_timesteps / self.num_envs) < self.rnd_start:
                int_rewards = None                                  # zeros
                self.obs_rms.update(self.env.unnormalize_obs(ro.observations[p]))
            else:
                int_rewards = self.rnd_bonus(obs)
            ro.record_step(rewards, int_rewards, dones, self._episodes_dev)
            if stats is not None:
                self._episode_log_step(stats, p)
            self.last_obs = obs
            self.last_dones = ro.masks[p]
        if stats is not None:
            self._episode_log_end()
        self._mean_int_reward = ro.compute_returns_and_advantages(values, int_values, ro.masks[-1])
        return True

    def train_rnd(self, obs, B_total=0):
        """algorithms.py:487-502 on a gathered minibatch of raw observations [B,D]."""
        x = normalize_obs(obs, self.obs_rms, out=self._scratch.get("rnd_nobs", obs.numel())[:obs.numel()].view(obs.shape))
        self.rnd.train_step(x, self._rnd_loss, B_total)
        self._sync_grads(self.rnd.bank)
        self.rnd.bank.adam_step(self.int_lr, self.max_grad_norm)

    def train(self):
        """algorithms.py:409-485."""
        ro = self.rollout
        rng = self._begin_train(ro, randn_per_minibatch=True)
        total, Bg, n_mb = self._train_geometry(ro)
        bufs = ro._minibatch_buffers(-(-Bg // D.world_size()) if self.shard_shuffle == "global" else Bg)
        fuse = self._fuse_adam_ok()
        step = 0
        self.rnd_trained_steps = 0
        for ep in range(self.n_epochs):
            for opts, lo, b, bt, key, src in self._epoch_minibatches(ro, rng, ep, self.n_epochs):
                def fn(opts=opts, lo=lo, b=b, bt=bt, src=src):
                    ok = self._gather_with_stats(ro, self._perm_all[lo:], bufs, dual=True, opts=opts, B=b, sources=src)
                    self._policy_step(bufs, b, self._losses_buf.data_ptr(), dual=True, int_vf_coef=self.int_vf_coef,
                                      B_total=bt, stats_ready=ok, stats_global=src is not None, row_dev=self._cursor.data_ptr(),
                                      fuse_adam=fuse)
                    self._policy_optim_step()
                self._graph_call(("rnd_policy",) + key, fn)
                if rng.next() < 0.25:                               # algorithms.py:468, same host RNG stream
                    self._graph_call(("rnd_pred",) + key, lambda b=b, bt=bt: self.train_rnd(bufs['observations'][:b], bt))
                    self.rnd_trained_steps += 1
                step += 1
        ro.generator_ready = True
        self._rng_close(rng)
        self._finish_train(step, ("train/total_loss", "train/policy_gradient_loss", "train/value_loss",
                                  "train/entropy_loss", "train/intrinsic_loss"))

    def learn(self, total_timesteps, log_interval, reward_target=None, log_to_file=False):
        return self._learn_loop(total_timesteps, log_interval, reward_target, "PPO_RND", log_to_file)


class PPO_ICM(BaseAlgorithm):
    """algorithms.py:546-756."""

    def __init__(self, *, env_id=None, lr=3e-4, int_lr=3e-4, nstep=128, batch_size=128, n_epochs=10, gamma=0.99,
                 gae_lam=0.95, clip_range=0.2, ent_coef=.01, vf_coef=0.5, max_grad_norm=0.2, hidden_size=128,
                 int_hidden_size=32, int_rew_integration=0.05, beta=0.2, policy_weight=1, env=None, device="cuda",
                 logger=None):
        super().__init__(env_id, lr, nstep, batch_size, n_epochs, gamma, gae_lam, clip_range, ent_coef, vf_coef,
                         max_grad_norm, env=env, device=device, logger=logger)
        self.int_rew_integration = int_rew_integration
        self.policy = Policy(self.env, hidden_size, device=self.device)
        # the reference builds this buffer WITHOUT gamma -> 0.99 always (algorithms.py:591)
        self.rollout = RolloutStorage(nstep, self.num_envs, self.env.observation_space, self.env.action_space,
                                      gae_lam=gae_lam, device=self.device)
        self.intrinsic_module = IntrinsicCuriosityModule(self.state_dim, self.action_converter,
                                                         hidden_size=int_hidden_size, device=self.device)
        self.int_lr = int_lr
        self._reset_env()
        self.policy_weight = policy_weight
        self.beta = 0.2                                             # hard-wired, algorithms.py:600
        self._icm_loss = torch.zeros(1, dtype=torch.float64, device=self.device)

    def icm_bonus(self, last_obs, obs, actions, rewards):
        """algorithms.py:629-630: r = (1-eta) r + eta * clamp(mean_f((fwd(phi(s),a) - phi(s'))^2), -5, 5).
        Returns (blended rewards [N] f32 CUDA, raw int_rewards [N])."""
        r = _dev(rewards, torch.float32, self.device).clone()
        ri = self.intrinsic_module.int_reward(last_obs, obs, actions, rewards=r, eta=self.int_rew_integration)
        return r, ri

    def collect_samples(self):
        """algorithms.py:603-649."""
        assert self.last_obs is not None
        if self.device_env:
            return self._collect_device()
        self.rollout.reset()
        ri_means = []
        for _ in range(self.nstep):
            actions, values, log_probs = self.policy.act(self.last_obs)
            obs, rewards, dones, infos = self.env.step(actions.cpu().numpy())
            if any(dones):
                self.num_episodes += sum(dones)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            rewards, ri = self.icm_bonus(self.last_obs, obs, actions, rewards)
            ri_means.append(ri.mean())
            A = self.action_converter.action_output
            self.rollout.add(self.last_obs, actions.reshape(self.num_envs, A), rewards, values, dones,
                             log_probs.reshape(self.num_envs, A))
            self.last_obs = obs
        self._mean_int_reward = torch.stack(ri_means).mean()
        self.rollout.compute_returns_and_advantages(values, dones=dones)
        return True

    def _collect_device(self):
        """collect_samples for an env on the GPU (see PPO._collect_device).  The bonus reads s and a from the rollout rows
        (the env may reuse its observation tensor and modify the actions it was given)."""
        ro = self.rollout
        ro.reset()
        stats = self._episode_log_begin()
        ri_means = []
        for _ in range(self.nstep):
            p = ro.pos
            actions, values = self.policy.act_into(self.last_obs, ro)
            obs, rewards, dones, infos = self.env.step(actions)
            self.num_timesteps += self.num_envs
            self.update_info_buffer(infos)
            rewards, ri = self.icm_bonus(ro.observations[p], obs, ro.actions[p], rewards)
            ri_means.append(ri.mean())
            ro.record_step(rewards, dones, self._episodes_dev)
            if stats is not None:
                self._episode_log_step(stats, p)
            self.last_obs = obs
        if stats is not None:
            self._episode_log_end()
        self._mean_int_reward = torch.stack(ri_means).mean()
        ro.compute_returns_and_advantages(values, dones=ro.masks[-1])
        return True

    def train(self):
        """algorithms.py:651-713.  Sharded ("global"): the shuffled-consecutive pairing of :684 (rows i, i+1 of the
        GLOBAL minibatch) is kept exactly -- rank r evaluates the pairs that start in its slice [lo, lo+b) and gathers
        ONE halo row (the first row of the next rank's slice) for the last of them; the ICM losses are means over the
        bg-1 global pairs, its gradients are summed over the ranks before its Adam step."""
        ro = self.rollout
        W = D.world_size()
        if W > 1 and self.shard_shuffle != "global":
            raise NotImplementedError("sharded PPO_ICM.train needs shard_shuffle='global' (the pairing spans the global minibatch)")
        rng = self._begin_train(ro)
        total, Bg, n_mb = self._train_geometry(ro)
        bufs = ro._minibatch_buffers((-(-Bg // W) if W > 1 else Bg) + 1)
        fuse = self._fuse_adam_ok()
        icm_row = self._icm_loss
        step = 0
        for ep in range(self.n_epochs):
            for opts, lo, b, bt, key, src in self._epoch_minibatches(ro, rng, ep, self.n_epochs):
                halo = 1 if (W > 1 and lo + b < bt) else 0          # pairs starting in [lo, lo+b): the last one needs row lo+b
                pairs_total = (bt if W > 1 else b) - 1

                def fn(opts=opts, lo=lo, b=b, bt=bt, src=src, halo=halo, pairs_total=pairs_total):
                    ok = self._gather_with_stats(ro, self._perm_all[lo:], bufs, opts=opts, B=b + halo, sources=src)
                    self._policy_step(bufs, b, self._losses_buf.data_ptr(), policy_weight=float(self.policy_weight),
                                      B_total=bt, stats_ready=ok, stats_global=src is not None, row_dev=self._cursor.data_ptr(),
                                      row_hold=True, fuse_adam=fuse)
                    icm_row.zero_()
                    self.intrinsic_module.train_step(bufs['observations'][:b + halo], bufs['actions'][:b + halo], self.beta,
                                                     icm_row, pairs_total=pairs_total)
                    self._policy_optim_step()                                   # only policy grads are clipped (:697)
                    if W > 1:
                        D.all_reduce_sum_(self.intrinsic_module.bank.grad)
                        D.all_reduce_sum_(icm_row)
                    self.intrinsic_module.bank.adam_step(self.int_lr, 0.0)
                    # total = pw*(...) + icm_loss (:692): the ICM loss lands in column 5 of the row the policy step left open
                    L.call("ppx_loss_row_commit", self._losses_buf.data_ptr(), self._cursor.data_ptr(), icm_row.data_ptr(), 5, 1,
                           L.stream())
                self._graph_call(("icm",) + key, fn)
                step += 1
        ro.generator_ready = True
        self._rng_close(rng)
        keys = ("train/total_loss", "train/policy_gradient_loss", "train/value_loss", "train/entropy_loss")
        self._finish_train(step, keys)
        self._record("train/icm_loss", float(np.mean(self.last_losses[:, 5])))

    def learn(self, total_timesteps, log_interval=5, reward_target=None, log_to_file=False):
        return self._learn_loop(total_timesteps, log_interval, reward_target, "PPO_ICM", log_to_file)
