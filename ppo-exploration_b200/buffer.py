"""Device-resident rollout buffers with the reference's call surface.

Mirrors buffer.py of the reference: BaseBuffer (:13-109), RolloutStorage (:111-267),
IntrinsicStorage (:271-394).  Same constructor arguments, method names, attribute names and
RolloutSample field order; the arrays are torch CUDA tensors in the reference's [T,N,...] layout and
the arithmetic (GAE scan, SimHash counts, shuffle-gather) runs in libppx.so.

Deliberate differences (documented in DESIGN.md):
  * arrays are allocated once and zeroed on reset() instead of re-allocated (buffer.py:153-161);
  * get() does not rewrite the attributes into the env-major flat layout (buffer.py:241-245): the
    gather kernel decodes flat index -> (t, n) on the fly.  `flat(name)` returns the flat view;
  * masks are uint8 (the reference stores int64 ones/zeros);
  * the hash width k is a constructor argument (`hash_bits`, default 16 = buffer.py:137).
The shuffle indices come from the same `np.random.permutation(T*N)` draw as the reference
(buffer.py:239), so a seeded run visits identical minibatches.
"""
import atexit
import ctypes as C
import os
import queue
import threading
import time
import weakref
from collections import namedtuple

import numpy as np
import torch

from . import _lib as L


def _dev(x, dtype, device):
    """numpy / torch (any device) -> contiguous CUDA tensor of `dtype`."""
    if isinstance(x, torch.Tensor):
        return x.detach().to(device=device, dtype=dtype, non_blocking=True).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x)).to(device=device, dtype=dtype, non_blocking=True)


def np_permutation(n):
    """np.random.permutation(n) (the draw of buffer.py:239), bit-exact and ~3x faster: libppx replays numpy's
    legacy MT19937 shuffle from numpy's own global state and hands the advanced state back."""
    st = np.random.get_state()
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = C.c_int(int(st[2]))
    out = np.empty(int(n), np.int64)
    L.call("ppx_np_permutation", key.ctypes.data, C.byref(pos), int(n), out.ctypes.data)
    np.random.set_state((st[0], key, pos.value, st[3], st[4]))
    return out


_live_streams = weakref.WeakSet()


class _Task:
    """Handle of a function running on a pooled worker thread; join() like a Thread's."""

    def __init__(self, fn, args):
        self.fn, self.args, self.done = fn, args, threading.Event()

    def join(self, timeout=None):
        self.done.wait(timeout)

    def is_alive(self):
        return not self.done.is_set()


class _WorkerPool:
    """Host worker threads that outlive the streams they serve.  A learner opens one HostRngStream per train() call (and
    one speculative stream per call); starting and retiring three OS threads each time is not free for the GPU -- the
    address-space changes of thread stacks (mmap / madvise in a process with pinned CUDA mappings) showed up as one
    ~0.3 ms stall of the running kernels per pass on the bench host (tools/trace_sharded.py).  Idle workers are re-used;
    the pool only grows when every worker is busy (e.g. two learners with parked speculative streams)."""

    def __init__(self):
        self.lock = threading.Lock()
        self.idle = []

    def submit(self, fn, *args):
        task = _Task(fn, args)
        with self.lock:
            box = self.idle.pop() if self.idle else None
        if box is None:
            box = queue.SimpleQueue()
            threading.Thread(target=self._loop, args=(box,), daemon=True).start()
        box.put(task)
        return task

    def _loop(self, box):
        while True:
            task = box.get()
            try:
                task.fn(*task.args)
            finally:
                task.done.set()
                with self.lock:
                    self.idle.append(box)


_workers = _WorkerPool()


def _stop_streams_at_exit():
    """Worker threads must not be inside torch / CUDA calls while the interpreter finalises."""
    for st in list(_live_streams):
        st.cancel()
    for st in list(_live_streams):
        st.t1.join(timeout=2.0)
        for t in st.t2:
            t.join(timeout=2.0)


atexit.register(_stop_streams_at_exit)


def rng_states_equal(a, b):
    """Equality of two np.random.get_state() tuples (legacy MT19937)."""
    return (a[0] == b[0] and int(a[2]) == int(b[2]) and int(a[3]) == int(b[3]) and float(a[4]) == float(b[4])
            and np.array_equal(a[1], b[1]))


class DevicePartners:
    """A permutation delivered as its Fisher-Yates partner list (pinned int32 [n] in acceptance order: entry r = partner
    of position n-1-r): the swaps are applied on the device (ppx_np_shuffle_apply_device, acceptance_order=1).

    The pinned buffer comes from a small per-size pool shared by the streams of this process (`_PartnerPool`): a consumer
    that has queued its H2D copy calls `release(event)` with an event recorded after the copy; the buffer is handed out
    again once that event has completed.  A consumer that never releases simply keeps its buffer (the pool allocates a
    new one) until the object is collected."""
    __slots__ = ("j", "ready", "_slot", "__weakref__")

    def __init__(self, j, slot=None):
        self.j = j
        self.ready = None                 # CUDA event: the permutation is staged on the device (set by a stream's uploader)
        self._slot = slot

    def release(self, event=None):
        if self._slot is not None:
            self._slot[1] = event if event is not None else True
            self._slot = None


class _PartnerPool:
    """Pinned int32 partner buffers, re-used across permutations and passes.  Why: a permutation's partner list is
    written once by the draw thread (4 bytes per draw) and read once by the H2D DMA; cycling through a few buffers that
    stay in the host's last-level cache instead of a fresh 4-16 MB block per epoch took the stream from 0.70 to 0.46-0.55 ns
    per draw on the bench host (bare draw loop into one warm buffer: 0.43; tools/host_rng_prof.py)."""

    def __init__(self):
        self.lock = threading.Lock()
        self.slots = {}                                         # n -> [[tensor, state, owner weakref], ...]
        # state: None = handed out, True = free, a CUDA event = free once it has completed

    def take(self, n):
        with self.lock:
            ring = self.slots.setdefault(n, [])
            pick = None
            for slot in ring:
                owner = slot[2]() if slot[2] is not None else None
                if slot[1] is None and owner is not None:
                    continue                                    # in use and its consumer is alive
                if slot[1] is not None and slot[1] is not True and not slot[1].query():
                    continue                                    # the copy out of it has not finished yet
                pick = slot
                break
            if pick is None:
                pick = [torch.empty(n, dtype=torch.int32, pin_memory=torch.cuda.is_available()), None, None]
                ring.append(pick)
            pick[1] = None
            dp = DevicePartners(pick[0], pick)
            pick[2] = weakref.ref(dp)
            return dp


_partner_pool = _PartnerPool()


def device_shuffle_default():
    """Apply the shuffle's swaps on the GPU (shuffle_dev.cu: 58 us per 524 288 on the copy stream, against 0.9 ms on a host
    core)?  Yes unless PPX_SHUFFLE_DEVICE=0: the host then only draws (0.3 ms per permutation), so a pass no longer depends
    on how many cores the ranks of a node have to share (8 ranks on 16 cores) or on a noisy host.  The host-side swaps
    remain for the sharded "global" shuffle (which needs the permutation on the host) and for n > 2^24."""
    return os.environ.get("PPX_SHUFFLE_DEVICE", "1") != "0"


def _apply_workers():
    """Stage-2 threads of a HostRngStream: 2 (measured on the bench host: 50 -> 66M transitions/s at C2; 3-4 workers gain
    nothing more, the draw stage and the GIL hand-offs then pace the stream), 1 when the ranks of this node have to share
    the host cores.  PPX_SHUFFLE_WORKERS overrides."""
    env = os.environ.get("PPX_SHUFFLE_WORKERS")
    if env:
        return max(1, int(env))
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 4
    ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    return max(1, min(2, cores // ranks - 2))


class HostRngStream:
    """Replays a fixed script of draws of the numpy legacy RNG in worker threads, in order, so the host shuffle
    (buffer.py:239) and RND's per-minibatch randn() (algorithms.py:468) overlap the GPU work while consuming exactly
    the reference's random stream.  script items: ('perm', n) | ('randn',).

    The stream works on a PRIVATE RandomState seeded with `state` (default: a snapshot of the global np.random state)
    and never touches the global one; the caller commits `final_state()` with np.random.set_state once the script has
    been consumed.  That makes a stream safe to start speculatively (before the caller knows it will be needed) and to
    cancel.  Two pipelined stages (both release the GIL inside libppx): stage 1 (one thread) owns the RNG -- it draws
    the Fisher-Yates partner sequence of each permutation and the scalar randn()s; stage 2 (`workers` threads, dealt the
    permutations round-robin: only the DRAWS of successive permutations are sequential, their swaps are independent)
    applies the swaps into a pinned buffer, running behind stage 1's published progress inside the permutation being
    drawn.  Results come out in script order; at most `ahead` items are in flight or waiting."""

    def __init__(self, script, state=None, ahead=None, workers=None, device_apply=False, uploader=None):
        self.script = list(script)
        self.device_apply = bool(device_apply)                  # 'perm' items come out as DevicePartners (n <= 2^24)
        # uploader(k, partners) -> CUDA event or None: called ON THE DRAW THREAD for the k-th permutation of the script as
        # soon as it is drawn; it queues the H2D copy + the device-side swaps, sets partners.ready and returns the event
        # that marks the end of the copy.  Before the draw thread would go idle (queue full, script done) it waits on the
        # last such event: the core that just wrote the partner list stays awake while the DMA reads it (a vCPU that goes
        # idle with the list dirty in its cache made that one 2 MB copy take 380 us instead of 45 on the bench host --
        # once per pass, after the last permutation).
        self.uploader = uploader
        self.profile, self.t_birth = [], time.perf_counter()    # per staged permutation: (start, wait+setup, draw, publish+stage) seconds
        nw = int(workers) if workers is not None else _apply_workers()
        self.nw = max(1, nw)
        if ahead is None:
            # a stream that stages its permutations itself may run through its whole script (the staging set holds every
            # epoch; a speculative stream then prepares the whole next pass while this one computes); device_apply without
            # an uploader has no stage 2: two finished permutations in hand are enough
            ahead = max(2, len(self.script)) if uploader is not None else (2 if self.device_apply else self.nw + 2)
        # results are delivered in script order through `q`: stage 1 enqueues one slot [event, value] per item BEFORE
        # it dispatches the work, the stage-2 worker that owns the item fills it
        self.q = queue.Queue(maxsize=max(1, int(ahead)))
        self.mids = [queue.Queue(maxsize=2) for _ in range(self.nw)]
        self.err = None
        self.cancelled = False
        self._final = None
        self.rs = np.random.RandomState()
        self.rs.set_state(np.random.get_state() if state is None else state)
        script = self.script
        self._jbufs = {}                                        # rotating partner buffers (<= ahead + 1 in flight per size)
        _live_streams.add(self)
        # stage 2 is only needed when some permutation of the script is applied on the host
        need2 = any(op[0] == 'perm' and not (self.device_apply and 2 <= int(op[1]) <= (1 << 24)) for op in script)
        self.nw2 = self.nw if need2 else 0
        self.t2 = [_workers.submit(self._apply, w) for w in range(self.nw2)]
        self.t1 = _workers.submit(self._draw, list(script))

    def _put(self, qq, item):
        while not self.cancelled:
            try:
                qq.put(item, timeout=0.05)
                return True
            except queue.Full:
                continue
        return False

    def _draw(self, script):
        """Stage 1 (one thread, owns the RNG): draws in script order; permutations are handed round-robin to the
        stage-2 workers -- the swaps of different permutations are independent, only the draws are sequential."""
        k = 0
        kperm = -1
        pending = None
        try:
            for op in script:
                if self.cancelled:
                    break
                slot = [threading.Event(), None]
                t_item = time.perf_counter()
                if pending is not None and self.q.full():       # about to block: see `uploader`
                    pending.synchronize()
                    pending = None
                if not self._put(self.q, slot):
                    break
                if op[0] == 'perm':
                    n = int(op[1])
                    kperm += 1
                    st = self.rs.get_state()
                    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
                    pos = C.c_int(int(st[2]))
                    if self.device_apply and 2 <= n <= (1 << 24):
                        # draws only: the partner list goes to the device, which applies the swaps (shuffle_dev.cu)
                        dp = _partner_pool.take(n)
                        prog = np.zeros(1, np.int64)
                        t0 = time.perf_counter()
                        L.call("ppx_np_shuffle_draws32_stream", key.ctypes.data, C.byref(pos), n, dp.j.data_ptr(), prog.ctypes.data)
                        t1 = time.perf_counter()
                        self.rs.set_state((st[0], key, pos.value, st[3], st[4]))
                        if self.uploader is not None and not self.cancelled:
                            pending = self.uploader(kperm, dp)
                        slot[1] = dp
                        slot[0].set()
                        t2 = time.perf_counter()
                        self.profile.append((t_item - self.t_birth, t0 - t_item, t1 - t0, t2 - t1))
                        continue
                    small = n <= 0x7fffffff
                    nbuf = self.q.maxsize + 2
                    pool = self._jbufs.setdefault(n, [[(np.empty(max(n, 1), np.int32 if small else np.int64),
                                                        np.zeros(1, np.int64)) for _ in range(nbuf)], 0])
                    j, prog = pool[0][pool[1] % nbuf]
                    pool[1] += 1
                    mid = self.mids[k % self.nw]
                    k += 1
                    if small:
                        # streaming: hand the buffer to stage 2 first, it runs behind the published progress counter
                        prog[0] = 0
                        if not self._put(mid, ('perm', j, n, prog, slot)):
                            break
                        try:
                            L.call("ppx_np_shuffle_draws32_stream", key.ctypes.data, C.byref(pos), n, j.ctypes.data,
                                   prog.ctypes.data)
                        except Exception:
                            prog[0] = 1 << 62                   # never leave stage 2 spinning on a failed draw
                            raise
                    else:
                        L.call("ppx_np_shuffle_draws", key.ctypes.data, C.byref(pos), n, j.ctypes.data)
                        if not self._put(mid, ('perm', j, n, None, slot)):
                            break
                    self.rs.set_state((st[0], key, pos.value, st[3], st[4]))
                else:
                    slot[1] = float(self.rs.randn())
                    slot[0].set()
            else:
                self._final = self.rs.get_state()
        except Exception as e:
            self.err = e
        self._put(self.q, None)
        for mid in self.mids:
            self._put(mid, None)
        if pending is not None:
            pending.synchronize()

    def _apply(self, w):
        """Stage 2 worker w: applies the swaps of the permutations dealt to it into a pinned buffer."""
        scratch32 = None
        mid = self.mids[w]
        try:
            while not self.cancelled:
                try:
                    item = mid.get(timeout=0.05)
                except queue.Empty:
                    continue
                if item is None:
                    break
                _, j, n, prog, slot = item
                out = torch.empty(n, dtype=torch.int64, pin_memory=torch.cuda.is_available())
                if prog is not None:
                    if scratch32 is None or scratch32.size < n:
                        scratch32 = np.empty(max(n, 1), np.int32)
                    L.call("ppx_np_shuffle_apply32_stream", j.ctypes.data, n, prog.ctypes.data,
                           scratch32.ctypes.data, out.data_ptr())
                else:
                    L.call("ppx_np_shuffle_apply", j.ctypes.data, n, out.data_ptr())
                slot[1] = out
                slot[0].set()
        except Exception as e:
            self.err = e
            self.cancelled = True                               # unblock everything; next() reports the error

    def next(self):
        slot = self.q.get()
        if slot is None:
            raise self.err if self.err is not None else RuntimeError("HostRngStream: script exhausted")
        while not slot[0].wait(timeout=0.05):
            if self.err is not None:
                raise self.err
        return slot[1]

    def final_state(self):
        """RNG state after the whole script (blocks until stage 1 has drawn everything)."""
        self.t1.join()
        if self.err is not None:
            raise self.err
        return self._final

    def cancel(self):
        """Abandon the stream (a speculative stream whose snapshot no longer matches the global RNG)."""
        self.cancelled = True

    def drain(self):
        self.t1.join()
        for t in self.t2:
            t.join()


class BaseBuffer(object):
    """buffer.py:13-109 (the parts the rollout path uses)."""

    def __init__(self, buffer_size, observation_space, action_space, n_envs=1, device=None):
        self.buffer_size = buffer_size
        self.observation_space = observation_space
        self.obs_shape = tuple(observation_space.shape)
        self.action_space = action_space
        self.pos = 0
        self.full = False
        self.n_envs = n_envs
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("ppx buffers live on a CUDA device; there is no CPU path")
        self.action_dim = 1 if action_space.__class__.__name__ == "Discrete" else action_space.shape[0]

    @staticmethod
    def swap_and_flatten(arr):
        """[T,N,...] -> [T*N,...] env-major, trailing dim added to 2-D input (buffer.py:40-52)."""
        shape = tuple(arr.shape)
        if len(shape) < 3:
            shape = shape + (1,)
        return arr.transpose(0, 1).reshape(shape[0] * shape[1], *shape[2:])

    def size(self):
        return self.buffer_size if self.full else self.pos

    def reset(self):
        self.pos = 0
        self.full = False


class CountTable:
    """Persistent SimHash count table (buffer.py:136) living in device memory."""

    def __init__(self, capacity=1 << 20):
        h = C.c_void_p()
        L.call("ppx_count_table_create", int(capacity), C.byref(h))
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                L.call("ppx_count_table_destroy", self._h)
                self._h = None
        except Exception:
            pass

    def clear(self):
        L.call("ppx_count_table_clear", self._h, L.stream())

    def update_codes(self, codes):
        """Sequential-semantics count update on packed uint64 codes -> uint32 counts."""
        counts = torch.empty(codes.numel(), dtype=torch.int32, device=codes.device)
        L.call("ppx_count_table_update", self._h, codes.data_ptr(), codes.numel(), counts.data_ptr(), L.stream())
        return counts

    def update_codes_owned(self, codes, W, rank):
        """Sharded table: `codes` is the globally ordered code list (identical on every rank); this rank updates only the
        codes it owns (hash(code) % W == rank) and returns their counts, 0 elsewhere (sum over ranks = all counts)."""
        counts = torch.empty(codes.numel(), dtype=torch.int32, device=codes.device)
        L.call("ppx_count_table_update_owned", self._h, codes.data_ptr(), codes.numel(), counts.data_ptr(), int(W), int(rank),
               L.stream())
        self.sharded = True
        return counts

    def __len__(self):
        n = C.c_uint64()
        L.call("ppx_count_table_size", self._h, C.byref(n))
        return int(n.value)

    def items(self):
        """{code: count} copied to the host (synchronous; tests and checkpointing)."""
        n = len(self)
        keys = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
        counts = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
        got = C.c_uint64()
        L.call("ppx_count_table_dump", self._h, keys.data_ptr(), counts.data_ptr(), n, C.byref(got))
        k = keys[:n].cpu().numpy().view(np.uint64)
        c = counts[:n].cpu().numpy()
        mine = {int(a): int(b) for a, b in zip(k, c)}
        if getattr(self, "sharded", False):                     # sharded table: the reference's dict is the union of the ranks' parts
            from . import dist as D
            if D.world_size() > 1:
                import torch.distributed as tdist
                parts = [None] * D.world_size()
                tdist.all_gather_object(parts, mine)
                mine = {}
                for p in parts:
                    mine.update(p)
        return mine

    def capacity(self):
        c = C.c_uint64()
        L.call("ppx_count_table_capacity", self._h, C.byref(c))
        return int(c.value)

    def state_dict(self):
        """This rank's part of the table for a checkpoint: the keys (uint64 codes as int64 bit patterns) and counts, sorted
        by key on the host so that the file does not depend on the dump's atomic order, the capacity and the `sharded`
        flag.  Synchronous."""
        n = len(self)
        keys = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
        counts = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
        got = C.c_uint64()
        L.call("ppx_count_table_dump", self._h, keys.data_ptr(), counts.data_ptr(), n, C.byref(got))
        k = keys[:n].cpu().numpy().view(np.uint64)
        order = np.argsort(k, kind="stable")
        return {"keys": torch.from_numpy(k[order].view(np.int64).copy()), "counts": counts[:n].cpu()[torch.from_numpy(order)],
                "capacity": self.capacity(), "sharded": bool(getattr(self, "sharded", False))}

    def load_state_dict(self, sd):
        """Replace the table by the one `state_dict()` described: a new table at the saved capacity (so growth happens at
        the same calls as on the original), filled by one insert kernel (ppx_count_table_load).  Synchronous."""
        keys, counts = sd["keys"], sd["counts"]
        if keys.dtype != torch.int64 or counts.dtype != torch.int32 or keys.dim() != 1 or keys.shape != counts.shape:
            raise ValueError("count table state: keys must be int64 [n] and counts int32 [n]")
        h = C.c_void_p()
        L.call("ppx_count_table_create", int(sd["capacity"]), C.byref(h))
        try:
            if keys.numel():
                k, c = keys.to("cuda"), counts.to("cuda")
                L.call("ppx_count_table_load", h, k.data_ptr(), c.data_ptr(), keys.numel(), L.stream())
        except BaseException:
            L.call("ppx_count_table_destroy", h)
            raise
        L.call("ppx_count_table_destroy", self._h)
        self._h = h
        self.sharded = bool(sd["sharded"])


class RolloutStorage(BaseBuffer):
    """buffer.py:111-267."""

    def __init__(self, buffer_size, n_envs, obs_space, action_space, gae_lam=0.95, gamma=0.99, sim_hash=False,
                 device=None, hash_bits=16, table_capacity=1 << 20):
        super().__init__(buffer_size, obs_space, action_space, n_envs=n_envs, device=device)
        self.gae_lam = gae_lam
        self.gamma = gamma
        self.generator_ready = False
        self._alloc()
        self.reset()
        # same global-RNG draw, at the same point, as buffer.py:137 (made whether or not hashing is on)
        self.A = np.random.randn(hash_bits, self.obs_shape[0])
        self._A_dev = None
        self.do_hash = bool(sim_hash)
        self.beta = 0.1 if sim_hash else None
        self.count_table = CountTable(table_capacity) if sim_hash else None
        self.RolloutSample = namedtuple('RolloutSample', ['observations', 'actions', 'old_values', 'old_log_probs',
                                                          'advantages', 'returns'])
        self._fields = [('observations', 'observations'), ('actions', 'actions'), ('old_values', 'values'),
                        ('old_log_probs', 'action_log_probs'), ('advantages', 'advantages'), ('returns', 'returns')]
        self._mb = {}
        self._load_stream, self._load_done = None, None     # load_rollout(overlap=True)
        self._rewards_f64, self._staged = None, False       # record_step: f64 rewards awaiting the SimHash bonus

    # ------------------------------------------------------------------ storage
    def _alloc(self):
        T, N, dev = self.buffer_size, self.n_envs, self.device
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)
        self.observations = z(T, N, *self.obs_shape)
        self.actions = z(T, N, self.action_dim, dt=torch.float64)            # f64, buffer.py:154
        self.rewards = z(T, N)
        self.int_rewards = z(T, N)
        self.values = z(T, N)
        self.returns = z(T, N)
        self.action_log_probs = z(T, N, self.action_dim)
        self.masks = torch.ones(T, N, dtype=torch.uint8, device=dev)         # ones, buffer.py:160
        self.advantages = z(T, N)

    def _zero(self):
        for name in ('observations', 'actions', 'rewards', 'int_rewards', 'values', 'returns', 'action_log_probs',
                     'advantages'):
            getattr(self, name).zero_()
        self.masks.fill_(1)

    def reset(self):
        """buffer.py:149-163 (zeroed in place instead of re-allocated)."""
        self._zero()
        self.generator_ready = False
        super().reset()

    def add(self, obs, action, reward, value, mask, log_prob):
        """buffer.py:165-186: write row `pos`; SimHash bonus first when enabled."""
        self.await_load()
        p, dev = self.pos, self.device
        obs_d = _dev(obs, torch.float32, dev).reshape(self.n_envs, *self.obs_shape)
        self.observations[p].copy_(obs_d)
        if self.do_hash:
            reward = self.sim_hash(obs_d, reward)
        self.actions[p].copy_(_dev(action, torch.float64, dev).reshape(self.n_envs, self.action_dim))
        self.rewards[p].copy_(_dev(reward, torch.float32, dev).reshape(self.n_envs))
        self.masks[p].copy_(_dev(mask, torch.uint8, dev).reshape(self.n_envs))
        self.values[p].copy_(_dev(value, torch.float32, dev).reshape(self.n_envs))
        self.action_log_probs[p].copy_(_dev(log_prob, torch.float32, dev).reshape(self.n_envs, self.action_dim))
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True

    def record_step(self, reward, done, episodes):
        """The rest of add() (buffer.py:165-186) for a step whose observation, action, log-prob and value rows were written
        by Policy.act_into: rewards and masks at row `pos` in ONE launch (ppx_rollout_record_step), and the number of
        nonzero dones added to `episodes` (int64 CUDA [1]).  reward: f32 / f64 [N] (CUDA or numpy); done: bool / uint8 [N]
        (CUDA or numpy).  No SimHash here: `sim_hash_recorded()` applies the bonus to the whole rollout afterwards."""
        self._record(reward, done, episodes, None, None)

    def _record(self, reward, done, episodes, int_reward, int_row):
        self.await_load()
        p, N, dev = self.pos, self.n_envs, self.device
        if isinstance(reward, torch.Tensor) and reward.is_cuda and reward.dtype in (torch.float32, torch.float64):
            r = reward.reshape(N).contiguous()
        else:
            f64 = (reward.dtype == torch.float64) if isinstance(reward, torch.Tensor) else np.asarray(reward).dtype == np.float64
            r = _dev(reward, torch.float64 if f64 else torch.float32, dev).reshape(N)
        f64 = r.dtype == torch.float64
        stage = None
        if f64 and self.do_hash:
            if self._rewards_f64 is None:
                self._rewards_f64 = torch.empty(self.buffer_size, N, dtype=torch.float64, device=dev)
            stage = self._rewards_f64[p]
        if p == 0:
            self._staged = stage is not None
        elif self._staged != (stage is not None):
            raise RuntimeError("record_step: the reward dtype changed within a rollout")
        if not isinstance(done, torch.Tensor):
            done = torch.as_tensor(np.ascontiguousarray(done))
        d = done.to(dev, non_blocking=True) if done.dtype in (torch.bool, torch.uint8) else _dev(done, torch.uint8, dev)
        d = d.reshape(N).contiguous()
        ir = None if int_reward is None else _dev(int_reward, torch.float32, dev).reshape(N)
        L.call("ppx_rollout_record_step", r.data_ptr(), int(f64), d.data_ptr(), L.ptr(ir), N, self.rewards[p].data_ptr(),
               L.ptr(stage), self.masks[p].data_ptr(), L.ptr(int_row), episodes.data_ptr(), L.stream())
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True

    def sim_hash_recorded(self):
        """The SimHash bonus (buffer.py:188-200) of a rollout filled through record_step, applied once to the whole rollout
        in the reference's order (t-major, env-minor) through sim_hash_sharded: on one GPU the per-step updates of add()
        bit for bit, sharded the global count table.  f64 rewards get the bonus in f64 and are rounded to f32 once, as in
        add()."""
        if self._staged:
            self.sim_hash_sharded(rewards=self._rewards_f64)
            self.rewards.copy_(self._rewards_f64)
        else:
            self.sim_hash_sharded()

    def load_rollout(self, overlap=False, **arrays):
        """Bulk fill from [T,N,...] host or device arrays (one H2D copy per field) and mark full.
        overlap=True: only what the count bonus reads (observations, rewards) is copied on the caller's stream; the other
        fields go up on a side stream UNDER the bonus kernels, and the methods of this class that read them
        (compute_returns_and_advantages, gather_into / get, flat, add) wait for that copy first.  Code that reads the
        arrays directly (`ro.values`, ...) on its own stream must call `await_load()` itself, hence opt-in."""
        dt = {'actions': torch.float64, 'masks': torch.uint8}

        def put(name, a):
            dst = getattr(self, name)
            dst.copy_(_dev(a, dt.get(name, torch.float32), self.device).reshape(dst.shape))
        self.await_load()
        first = ('observations', 'rewards')
        late = [k for k in arrays if k not in first] if overlap else []
        for name, a in arrays.items():
            if name not in late:
                put(name, a)
        if late:
            if self._load_stream is None:
                self._load_stream = torch.cuda.Stream(device=self.device)
            cur = torch.cuda.current_stream()
            self._load_stream.wait_stream(cur)                  # earlier readers of these arrays were queued on the caller's stream
            with torch.cuda.stream(self._load_stream):
                for name in late:
                    put(name, arrays[name])
                self._load_done = torch.cuda.Event()
                self._load_done.record(self._load_stream)
        self.pos, self.full = self.buffer_size, True
        self.generator_ready = False

    def await_load(self):
        """Make the caller's stream wait for the side-stream part of the last load_rollout(overlap=True)."""
        if self._load_done is not None:
            torch.cuda.current_stream().wait_event(self._load_done)
            self._load_done = None

    # ------------------------------------------------------------------ SimHash
    def _A(self):
        if self._A_dev is None or self._A_dev_src is not self.A:
            self._A_dev = torch.as_tensor(np.ascontiguousarray(self.A, dtype=np.float64)).to(self.device)
            self._A_dev_src = self.A
        return self._A_dev

    def sim_hash(self, obs, rewards):
        """buffer.py:188-200.  Mutates and returns `rewards` (numpy in -> numpy out, tensor in -> tensor).
        A 3-D obs [T,N,D] with rewards [T,N] applies the bonus for a whole rollout in one launch, in the
        reference's order (t-major, env-minor)."""
        A = self._A()
        k, D = A.shape
        obs_d = _dev(obs, torch.float32, self.device).reshape(-1, D)
        n = obs_d.shape[0]
        is_np = not isinstance(rewards, torch.Tensor)
        f64 = (rewards.dtype == np.float64) if is_np else (rewards.dtype == torch.float64)
        if is_np or not rewards.is_cuda:
            r_d = _dev(rewards, torch.float64 if f64 else torch.float32, self.device).reshape(n).clone()
        else:
            r_d = rewards if f64 else rewards  # in place on the caller's CUDA tensor
            if r_d.dtype not in (torch.float32, torch.float64) or not r_d.is_contiguous():
                raise RuntimeError("sim_hash: rewards must be a contiguous f32/f64 tensor")
        L.call("ppx_simhash_update", self.count_table._h, A.data_ptr(), obs_d.data_ptr(), int(k), int(D), int(n),
               float(self.beta), r_d.data_ptr(), int(f64), None, None, L.stream())
        if is_np:
            rewards[...] = r_d.cpu().numpy().reshape(rewards.shape)
            return rewards
        if not rewards.is_cuda:
            rewards.copy_(r_d.cpu().reshape(rewards.shape))
            return rewards
        return rewards

    def sim_hash_sharded(self, obs=None, rewards=None):
        """buffer.py:188-200 for a rollout whose env columns are sharded over the ranks (SURVEY §8e rows 2-3): this
        rank holds columns [rank*N, (rank+1)*N) of the global [T, W*N] rollout.  Codes are computed locally; the
        count table is global and its update order-dependent (t-major, env-minor over ALL envs), so the packed codes
        are all-gathered into that order and the table is SHARDED by code: rank hash(code) % W owns a code, resolves its
        occurrences in the global order and keeps its count; the counts come back through one all-reduce and every rank
        applies those of its own columns -- bit-identical to one GPU holding all envs, per-rank work independent of W
        except for the linear partition pass.  Mutates and returns `rewards` ([T,N] CUDA f32; default: the stored rollout)."""
        from . import dist as D
        obs = self.observations if obs is None else obs
        rewards = self.rewards if rewards is None else rewards
        W, r = D.world_size(), D.rank()
        if W == 1:
            return self.sim_hash(obs, rewards)
        T, N = obs.shape[0], obs.shape[1]
        if not (isinstance(rewards, torch.Tensor) and rewards.is_cuda and rewards.dtype in (torch.float32, torch.float64)
                and rewards.is_contiguous()):
            raise RuntimeError("sim_hash_sharded: rewards must be a contiguous f32 / f64 CUDA tensor [T, N]")
        codes = self.sim_hash_codes(obs).view(T, N)
        allc = D.interleave_env_shards(D.all_gather_cat(codes)).reshape(-1)          # [T, W*N] in global env order
        # bucket-owner ranks: every rank walks the same ordered list but resolves only the codes it owns (1/W of the
        # order-dependent work, table sharded by hash(code) % W); one all-reduce returns every count to every rank
        counts = self.count_table.update_codes_owned(allc, W, r)
        D.all_reduce_sum_(counts)
        counts = counts.view(T, W, N)[:, r].contiguous()
        L.call("ppx_simhash_bonus", counts.data_ptr(), T * N, float(self.beta), rewards.data_ptr(),
               int(rewards.dtype == torch.float64), L.stream())
        return rewards

    def sim_hash_codes(self, obs):
        """packed uint64 codes (bit b = sign bit b of buffer.py:194) as an int64 CUDA tensor."""
        A = self._A()
        k, D = A.shape
        obs_d = _dev(obs, torch.float32, self.device).reshape(-1, D)
        codes = torch.empty(obs_d.shape[0], dtype=torch.int64, device=self.device)
        L.call("ppx_simhash_codes", A.data_ptr(), obs_d.data_ptr(), int(k), int(D), obs_d.shape[0], codes.data_ptr(),
               L.stream())
        return codes

    # ------------------------------------------------------------------ GAE
    def compute_returns_and_advantages(self, last_value, dones):
        """buffer.py:203-230."""
        self.await_load()
        lv = _dev(last_value, torch.float32, self.device).reshape(self.n_envs)
        d = _dev(dones, torch.uint8, self.device).reshape(self.n_envs)
        L.call("ppx_gae", self.rewards.data_ptr(), self.values.data_ptr(), self.masks.data_ptr(), lv.data_ptr(),
               d.data_ptr(), float(self.gamma), float(self.gae_lam), self.buffer_size, self.n_envs,
               self.advantages.data_ptr(), self.returns.data_ptr(), L.stream())

    # ------------------------------------------------------------------ shuffle-gather
    def flat(self, name):
        """env-major flat view of a stored array, shaped like the reference's flattened attribute."""
        self.await_load()
        return self.swap_and_flatten(getattr(self, name))

    def _minibatch_buffers(self, B):
        """Persistent gather destinations for minibatches of up to B samples (stable addresses)."""
        key = int(B)
        if key not in self._mb:
            bufs = {}
            for field, src in self._fields:
                s = getattr(self, src)
                bufs[field] = torch.empty((B,) + tuple(s.shape[2:]), dtype=s.dtype, device=self.device)
            self._mb[key] = bufs
        return self._mb[key]

    def gather_into(self, idx_dev, bufs, stats=None, opts=None, sources=None, B=None):
        """One fused launch: every RolloutSample field for the flat indices `idx_dev` (int64, CUDA).  stats: optional list
        of (field, device pointer to 2 doubles) -- {mean, unbiased std} of that gathered f32 [B] field (the advantage
        normalisation statistics) computed by the same launch."""
        self.await_load()
        B = idx_dev.numel() if B is None else int(B)
        n = len(self._fields)
        srcs = (C.c_void_p * n)()
        dsts = (C.c_void_p * n)()
        rb = (C.c_int * n)()
        n_envs = self.n_envs
        for i, (field, src) in enumerate(self._fields):
            s = getattr(self, src)
            if B > bufs[field].shape[0]:
                raise RuntimeError(f"gather_into: {B} rows do not fit the {bufs[field].shape[0]}-row minibatch buffer '{field}'")
            srcs[i] = s.data_ptr() if sources is None else sources[src].data_ptr()
            dsts[i] = bufs[field].data_ptr()
            rb[i] = int(s[0, 0].numel() * s.element_size()) if s.dim() > 2 else s.element_size()
        if opts is not None and opts.n_shard > 0:
            n_envs = sources[self._fields[0][1]].shape[0] * opts.n_shard     # sources: [W, T, n_shard, ...]
        if stats or opts is not None:
            names = [f for f, _ in self._fields]
            stats = stats or []
            sf = (C.c_int * max(1, len(stats)))(*[names.index(f) for f, _ in stats])
            so = (C.c_void_p * max(1, len(stats)))(*[p for _, p in stats])
            L.call("ppx_gather_minibatch_stats", srcs, dsts, rb, n, idx_dev.data_ptr(), B, self.buffer_size, n_envs,
                   sf, so, len(stats), C.byref(opts) if opts is not None else None, L.stream())
            return
        L.call("ppx_gather_minibatch", srcs, dsts, rb, n, idx_dev.data_ptr(), B, self.buffer_size, n_envs,
               L.stream())

    def _sample_from(self, bufs, B):
        out = []
        for field, src in self._fields:
            t = bufs[field][:B]
            if field in ('advantages', 'int_advantages'):
                t = t.reshape(B, 1)                                       # 2-D arrays gain a trailing dim
            out.append(t)
        return self.RolloutSample(*out)

    def permutation(self):
        """The epoch's shuffle: the reference's own host draw (buffer.py:239), uploaded once."""
        idx = np_permutation(self.buffer_size * self.n_envs)
        return torch.as_tensor(idx).to(self.device, non_blocking=True)

    def get(self, batch_size=None):
        """buffer.py:233-254: generator of RolloutSample minibatches (CUDA tensors; each sample owns
        fresh storage, like the reference's torch.tensor copies)."""
        self.await_load()
        assert self.full, ''
        total = self.buffer_size * self.n_envs
        idx = self.permutation()
        self.generator_ready = True
        if batch_size is None:
            batch_size = total
        start = 0
        while start < total:
            sl = idx[start:start + batch_size]
            B = sl.numel()
            bufs = {f: torch.empty((B,) + tuple(getattr(self, s).shape[2:]), dtype=getattr(self, s).dtype,
                                   device=self.device) for f, s in self._fields}
            self.gather_into(sl, bufs)
            yield self._sample_from(bufs, B)
            start += batch_size


class IntrinsicStorage(RolloutStorage):
    """buffer.py:271-394: two reward streams (RND)."""

    def __init__(self, buffer_size, n_envs, obs_space, action_space, gae_lam=0.95, gamma=0.99, int_gamma=0.99,
                 device=None):
        super().__init__(buffer_size, n_envs, obs_space, action_space, gae_lam, gamma, device=device)
        self.int_gamma = int_gamma
        self.RolloutSample = namedtuple('RolloutSample', ['observations', 'actions', 'old_values', 'int_values',
                                                          'old_log_probs', 'advantages', 'int_advantages', 'returns',
                                                          'int_returns'])
        self._fields = [('observations', 'observations'), ('actions', 'actions'), ('old_values', 'values'),
                        ('int_values', 'int_values'), ('old_log_probs', 'action_log_probs'),
                        ('advantages', 'advantages'), ('int_advantages', 'int_advantages'), ('returns', 'returns'),
                        ('int_returns', 'int_returns')]

    def _alloc(self):
        super()._alloc()
        T, N, dev = self.buffer_size, self.n_envs, self.device
        for name in ('int_values', 'int_returns', 'int_advantages'):
            setattr(self, name, torch.zeros(T, N, dtype=torch.float32, device=dev))

    def _zero(self):
        super()._zero()
        for name in ('int_values', 'int_returns', 'int_advantages'):
            getattr(self, name).zero_()

    def add(self, obs, action, reward, int_reward, value, int_value, mask, log_prob):
        """buffer.py:305-318."""
        self.await_load()
        p, dev = self.pos, self.device
        self.int_rewards[p].copy_(_dev(int_reward, torch.float32, dev).reshape(self.n_envs))
        self.int_values[p].copy_(_dev(int_value, torch.float32, dev).reshape(self.n_envs))
        super().add(obs, action, reward, value, mask, log_prob)

    def record_step(self, reward, int_reward, done, episodes):
        """RolloutStorage.record_step with the intrinsic-reward row (buffer.py:305-318) in the same launch; int_reward None
        writes zeros (RND's warm-up)."""
        self._record(reward, done, episodes, int_reward, self.int_rewards[self.pos])

    def compute_returns_and_advantages(self, last_value, last_int_value, dones):
        """buffer.py:321-362.  Returns mean(int_rewards) as a 0-d CUDA tensor (the value the reference
        logs at :335) so the caller can record it without forcing a sync here."""
        self.await_load()
        lv = _dev(last_value, torch.float32, self.device).reshape(self.n_envs)
        liv = _dev(last_int_value, torch.float32, self.device).reshape(self.n_envs)
        d = _dev(dones, torch.uint8, self.device).reshape(self.n_envs)
        L.call("ppx_gae_dual", self.rewards.data_ptr(), self.values.data_ptr(), self.masks.data_ptr(), lv.data_ptr(),
               d.data_ptr(), float(self.gamma), float(self.gae_lam), self.int_rewards.data_ptr(),
               self.int_values.data_ptr(), liv.data_ptr(), float(self.int_gamma), self.buffer_size, self.n_envs,
               self.advantages.data_ptr(), self.returns.data_ptr(), self.int_advantages.data_ptr(),
               self.int_returns.data_ptr(), L.stream())
        return self.int_rewards.mean()


def discount_with_dones(rewards, dones, gamma, device="cuda"):
    """SilModule.discount_with_dones (sil_module.py:99-105) over [T] or [T,N] columns, f64."""
    r = _dev(np.asarray(rewards, dtype=np.float64), torch.float64, device)
    d = _dev(np.asarray(dones), torch.uint8, device)
    shape = r.shape
    r2 = r.reshape(shape[0], -1).contiguous()
    d2 = d.reshape(shape[0], -1).contiguous()
    out = torch.empty_like(r2)
    L.call("ppx_discount", r2.data_ptr(), d2.data_ptr(), float(gamma), r2.shape[0], r2.shape[1], out.data_ptr(),
           L.stream())
    return out.reshape(shape)
