"""ES-NSRA step on the GPU with the reference's method names.

Mirrors EvolutionStrategy of evolution_strategies.py (:100-384) for the parts on the learner hot
path: _get_population (:172-182), _get_weights_try (:137-145), _update_weights (:217-239), get_kNN
(:264-281), the novelty lines (:318-325) and calc_noveltiy_distribution (:283-290), plus the policy forward
of episode evaluation (FeedForwardNetwork.predict :48-61) batched over the population
(`predict_population`, SURVEY §8f.4).  For a batched env that lives on the GPU, `evaluate` runs the episode loop of
evaluate / get_behavior_char (:153-170) on the device -- fitness, episode lengths and behaviour characterisations -- and
`run_generation` chains ask -> evaluate -> tell, and `run` is the reference's ES-NSRA loop (:293-384) over a meta-population
of brains with a device behaviour archive (DESIGN.md §3.15).  For an env on the host, the caller steps it with `predict_population` /
`discrete_action` and feeds the fitness vector back through `_update_weights` or `tell`.

Build-side design (SURVEY §0.1): the population is a vector of offsets into ONE resident f32 noise
table instead of P fresh f64 randn tensors; theta is one flat f64 device vector over all layers.
Parity mode: pass a dense eps array ([P, D] float32-representable values, or the reference's nested
list-of-layers population) wherever a population is expected.
"""
import numpy as np
import torch

from . import _lib as L
from . import dist as D


class EvolutionStrategy(object):
    def __init__(self, env_id=None, hidden_sizes=(64, 64), nsr_plateu=1.5, nsr_range=(0, 1), nsr_update=0.05,
                 population_size=50, sigma=0.1, learning_rate=0.01, decay=0.9995, novelty_param=0.5, num_threads=1,
                 obs_dim=None, n_actions=None, device="cuda", noise_table_size=1 << 24, noise_seed=0,
                 fitness_shaping="zscore", novelty_mode="brain"):
        if novelty_mode not in ("brain", "member"):
            raise ValueError(f"novelty_mode must be 'brain' or 'member', got {novelty_mode!r}")
        if obs_dim is None or n_actions is None:
            raise ValueError("pass obs_dim= and n_actions= (the reference reads them from gym.make(env_id), "
                             "evolution_strategies.py:121; the env layer is out of scope here)")
        self.env_id = env_id
        self.device = torch.device(device)
        self.hidden_sizes = list(hidden_sizes)
        sizes = [obs_dim, *hidden_sizes, n_actions]
        self.shapes = [(sizes[i], sizes[i + 1]) for i in range(len(sizes) - 1)]       # :33-35, bias-free
        self.layer_sizes = [a * b for a, b in self.shapes]
        self.D = int(sum(self.layer_sizes))
        # same global-RNG draws as FeedForwardNetwork.__init__ (:34-35)
        w0 = [np.random.randn(*s) for s in self.shapes]
        self.theta = torch.as_tensor(np.concatenate([w.ravel() for w in w0])).to(self.device)
        self.POPULATION_SIZE = population_size
        self.SIGMA = sigma
        self._lr = torch.full((1,), float(learning_rate), dtype=torch.float64, device=self.device)
        self.decay = decay
        self.novelty_param = novelty_param
        self.K = 10
        self.nsr_plateu, self.nsr_range, self.nsr_update = nsr_plateu, list(nsr_range), nsr_update
        self.fitness_shaping = fitness_shaping
        # "brain": the reference's update, brain b's novelty broadcast over the population; "member": NSRA-ES (Conti et al.
        # 2018, Alg. 3), every member's own novelty shaped next to its fitness (DESIGN.md §3.16)
        self.novelty_mode = novelty_mode
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._ws = None
        self._noise = None
        self._noise_size, self._noise_seed = int(noise_table_size), int(noise_seed)
        self._draw = torch.zeros(2, dtype=torch.int64, device=self.device)        # [population draws made so far, ticket word]
        self._px = False                                                          # PeerExchange for the sharded update | None
        self._graphs = {}
        self.update_mode = "single"
        self.thetas = None                                                        # the meta-population of run() [M, D] f64

    # ---- checkpoints (DESIGN.md §3.14) ----
    def save(self, path):
        """Write theta, the device learning rate, the device draw counter, novelty_param and the constructor configuration
        to `path` (one `torch.save` file, loadable with `weights_only=True`).  The noise table is not stored: `load`
        regenerates it from its seed.  After run(), also the run's state at the generation boundary: `thetas`, the
        behaviour archive, the brains' last BCs and returns, the f_b window and best, the generation counter, numpy's global
        RNG state (the brain picks draw from it) and the `state_dict()` of env and brain_env where they have one.  Under
        torch.distributed every rank saves its own file: pass a per-rank path."""
        from .checkpoint import header
        ck = header(type(self).__name__)
        ck.update(
            config=dict(env_id=self.env_id, hidden_sizes=list(self.hidden_sizes), nsr_plateu=self.nsr_plateu,
                        nsr_range=list(self.nsr_range), nsr_update=self.nsr_update, population_size=int(self.POPULATION_SIZE),
                        sigma=float(self.SIGMA), decay=self.decay, obs_dim=int(self.shapes[0][0]),
                        n_actions=int(self.shapes[-1][1]), noise_table_size=self._noise_size, noise_seed=self._noise_seed,
                        fitness_shaping=self.fitness_shaping, novelty_mode=self.novelty_mode),
            K=int(self.K), theta=self.theta.cpu(), lr=self._lr.cpu(), draw=self._draw.cpu(),
            novelty_param=float(self.novelty_param), world_size=D.world_size(), rank=D.rank())
        if self.thetas is not None:
            from .checkpoint import np_rng_state
            env, brain_env = getattr(self, "_run_envs", (None, None))
            state = {name: e.state_dict() for name, e in (("env", env), ("brain_env", brain_env))
                     if e is not None and callable(getattr(e, "state_dict", None))}
            ck["run"] = dict(thetas=self.thetas.cpu(), archive=self.archive.cpu(), bc=self._bc_m.cpu(), f=self._f_m.cpu(),
                             fb_window=list(self._fb_window), best=float(self._best), generation=int(self._generation),
                             numpy_rng=np_rng_state(), envs=state)
        torch.save(ck, path)

    @classmethod
    def load(cls, path, device="cuda", env=None, brain_env=None):
        """The strategy saved at `path` by `save()`: the next ask() / evaluate() / tell() / run_generation() compute what the
        saved object would have.  numpy's global RNG is left as it was (the constructor's draw of initial weights is
        undone) -- unless the file holds a run: then the run's state is restored, numpy's global RNG is set to its state at
        save(), `env` / `brain_env` (fresh ones, as passed to run()) load their saved `state_dict()`, and the next run()
        continues the run.  Captured graphs are captured anew.  ValueError for another format version or world size / rank."""
        from .checkpoint import read, tensor_into
        ck = read(path, cls.__name__)
        W, r = D.world_size(), D.rank()
        if (ck["world_size"], ck["rank"]) != (W, r):
            raise ValueError(f"the checkpoint was saved by rank {ck['rank']} of {ck['world_size']}, this is rank {r} of {W}")
        rng = np.random.get_state()
        es = cls(device=device, **ck["config"])
        np.random.set_state(rng)
        es.K, es.novelty_param = ck["K"], ck["novelty_param"]
        tensor_into(es.theta, ck["theta"], "ES theta")
        tensor_into(es._lr, ck["lr"], "ES learning rate")
        tensor_into(es._draw, ck["draw"], "ES draw counter")
        run = ck.get("run")
        if run is not None:
            from .checkpoint import np_rng_tuple
            M, k = run["bc"].shape
            n = run["archive"].shape[0]
            es.thetas = run["thetas"].to(es.device)
            es._run_buffers(M, k, capacity=max(16, 1 << n.bit_length()))
            es._archive[:n].copy_(run["archive"])
            es._archive_n = n
            es._bc_m.copy_(run["bc"])
            es._f_m.copy_(run["f"])
            es._fb_window, es._best, es._generation = list(run["fb_window"]), run["best"], run["generation"]
            for name, e in (("env", env), ("brain_env", brain_env)):
                if e is not None and name in run["envs"]:
                    e.load_state_dict(run["envs"][name])
            np.random.set_state(np_rng_tuple(run["numpy_rng"]))
        return es

    # ---- state views ----
    @property
    def learning_rate(self):
        return float(self._lr.item())

    @learning_rate.setter
    def learning_rate(self, v):
        self._lr.fill_(float(v))

    @property
    def weights(self):
        return self.get_weights()

    def get_weights(self):
        """list of [in,out] f64 numpy arrays, like FeedForwardNetwork.get_weights (:63-64)."""
        flat = self.theta.cpu().numpy()
        out, o = [], 0
        for s, n in zip(self.shapes, self.layer_sizes):
            out.append(flat[o:o + n].reshape(s).copy())
            o += n
        return out

    def set_weights(self, weights):
        self.theta.copy_(torch.as_tensor(np.concatenate([np.asarray(w, np.float64).ravel() for w in weights])))

    # ---- noise table / population ----
    def noise_table(self):
        if self._noise is None:
            self._noise = torch.empty(self._noise_size, dtype=torch.float32, device=self.device)
            L.call("ppx_noise_fill", self._noise.data_ptr(), self._noise_size, self._noise_seed, L.stream())
        return self._noise

    def _get_population(self, out=None):
        """:172-182.  Returns int64 offsets [P] (multiples of 4, so rows are 16-byte aligned) into the table, drawn on the
        device (Philox keyed by the noise seed, counter = (member, draw number)): no host RNG, no H2D copy, and every rank
        of a sharded run draws the identical population."""
        self.noise_table()
        off = torch.empty(self.POPULATION_SIZE, dtype=torch.int64, device=self.device) if out is None else out
        L.call("ppx_es_offsets", self._noise_seed + 1, self._draw.data_ptr(), self.POPULATION_SIZE, self._noise_size, self.D,
               off.data_ptr(), L.stream())
        return off

    def _as_eps(self, population):
        """-> (noise tensor f32, offsets tensor or None)."""
        if isinstance(population, torch.Tensor) and population.dtype == torch.int64:
            return self.noise_table(), population
        if isinstance(population, list):                             # reference nested list [P][L] of arrays
            population = np.array([np.concatenate([np.asarray(l).ravel() for l in m]) for m in population])
        eps = torch.as_tensor(np.ascontiguousarray(population)).to(self.device)
        if eps.dtype != torch.float32:
            e32 = eps.float()
            if not torch.equal(e32.double(), eps.double()):
                raise ValueError("dense eps must be float32-representable (the device noise is f32)")
            eps = e32
        return eps.contiguous(), None

    def perturb_all(self, population, out_f64=False):
        """theta + sigma*eps for every member: [P, D] CUDA (f32 by default, f64 = reference dtype)."""
        noise, off = self._as_eps(population)
        P = off.numel() if off is not None else noise.shape[0]
        out = torch.empty(P, self.D, dtype=torch.float64 if out_f64 else torch.float32, device=self.device)
        L.call("ppx_es_perturb", self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None,
               float(self.SIGMA), P, self.D, out.data_ptr(), int(out_f64), L.stream())
        return out

    def predict_population(self, population, obs, discrete=False, sigma=None):
        """FeedForwardNetwork.predict (:48-61) for every member at once: member p sees obs[p] and acts with
        theta + sigma*eps_p, formed on the fly from the noise table (the perturbed weights are never materialised).
        obs [P, obs_dim] -> f64 CUDA [P, n_actions]: tanh(logits) for Box (continuous_action :84-89); the raw logits
        with discrete=True (sample them with `discrete_action`, which keeps the reference's host RNG draw)."""
        noise, off = self._as_eps(population)
        P = off.numel() if off is not None else noise.shape[0]
        obs = torch.as_tensor(np.asarray(obs) if not isinstance(obs, torch.Tensor) else obs).to(self.device).double().contiguous()
        sizes = [self.shapes[0][0]] + [sh[1] for sh in self.shapes]
        if tuple(obs.shape) != (P, sizes[0]):
            raise ValueError(f"obs must be [{P}, {sizes[0]}], got {tuple(obs.shape)}")
        out = torch.empty(P, sizes[-1], dtype=torch.float64, device=self.device)
        import ctypes as C
        L.call("ppx_es_forward", self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None,
               float(self.SIGMA if sigma is None else sigma), P, (C.c_int * len(sizes))(*sizes), len(sizes) - 1,
               obs.data_ptr(), 0 if discrete else 1, out.data_ptr(), L.stream())
        return out

    def predict(self, obs, discrete=False):
        """FeedForwardNetwork.predict (:48-61) of the CURRENT weights for one observation (or a batch [n, obs_dim])."""
        obs = np.asarray(obs, dtype=np.float64)
        obs = obs.reshape(1, -1) if obs.ndim == 1 or obs.size == self.shapes[0][0] else obs
        zero = np.zeros((obs.shape[0], self.D), dtype=np.float32)
        return self.predict_population(zero, obs, discrete=discrete, sigma=0.0)

    @staticmethod
    def discrete_action(logits):
        """discrete_action (:81-82) on the host: softmax then one np.random.choice per member (the reference's RNG)."""
        out = []
        for row in np.asarray(logits.cpu() if isinstance(logits, torch.Tensor) else logits, dtype=np.float64):
            p = np.exp(row) / np.sum(np.exp(row))
            out.append(int(np.random.choice(np.arange(row.size), p=p.squeeze())))
        return np.array(out)

    def _get_weights_try(self, w, p):
        """:137-145 for ONE member given as the reference's list of per-layer eps arrays; returns a list of
        f64 numpy arrays.  (`w` is accepted for signature compatibility; theta on device is what is used.)"""
        flat = self.perturb_all([p], out_f64=True)[0].cpu().numpy()
        out, o = [], 0
        for s, n in zip(self.shapes, self.layer_sizes):
            out.append(flat[o:o + n].reshape(s))
            o += n
        return out

    # ---- population sharding (SURVEY §8e): members split across ranks, update replicated ----
    def shard_population(self, population):
        """The contiguous slice of `population` (offsets [P] or dense eps [P,D]) this rank perturbs and evaluates.
        Every rank must hold the same `population` (same noise seed -> `_get_population` draws identical offsets)."""
        W, r = D.world_size(), D.rank()
        P = population.shape[0]
        if P % W:
            raise ValueError(f"population size {P} must be a multiple of the world size {W}")
        return population[r * (P // W):(r + 1) * (P // W)]

    def gather_fitness(self, local_rewards):
        """all-gather of the per-rank fitness slices -> [P] f64 in member order on every rank; each rank then applies
        the identical `_update_weights` from the replicated noise table (no parameter traffic)."""
        r = torch.as_tensor(np.asarray(local_rewards, dtype=np.float64)).to(self.device) \
            if not isinstance(local_rewards, torch.Tensor) else local_rewards.to(self.device, torch.float64)
        W = D.world_size()
        if W == 1:
            return r
        out = torch.empty(W, r.numel(), dtype=torch.float64, device=self.device)
        D.all_gather_into(out, r)
        return out.reshape(-1)

    # ---- update ----
    def _update_weights(self, rewards, population, novelty=None):
        """:217-239.  Asynchronous; `self.update_skipped` reads back the std==0 flag.  `novelty` may be a python float
        (as in the reference) or a 1-element f64 CUDA tensor (e.g. `novelty_batch(...)[1][m:m+1]`), which keeps the
        k-NN result on the device -- no host round trip in the step.
        novelty_mode="member": `novelty` is required, the novelty of every member (f64 [P], global member order, e.g.
        `member_novelty(...)`), and the update is ppx_es_update_member: fitness and novelty each shaped over the P members,
        mixed with novelty_param; z-score skips only when both stds are 0."""
        noise, off = self._as_eps(population)
        P = off.numel() if off is not None else noise.shape[0]
        r = torch.as_tensor(np.asarray(rewards, dtype=np.float64)).to(self.device) if not isinstance(rewards, torch.Tensor) \
            else rewards.to(self.device, torch.float64)
        if self.novelty_mode == "member":
            return self._update_weights_member(r, noise, off, P, novelty)
        need = L.call("ppx_es_update_workspace", P, self.D)
        if self._ws is None or self._ws.numel() * 8 < need:
            self._ws = torch.zeros(need // 8 + 1, dtype=torch.float64, device=self.device)     # holds self re-arming tickets
        nov_dev = None
        if isinstance(novelty, torch.Tensor):
            nov_dev = novelty.to(self.device, torch.float64).reshape(-1)[:1].contiguous()
        W, rk = D.world_size(), D.rank()
        px = self._peer_exchange() if (W > 1 and self.fitness_shaping != "centered_rank" and P % W == 0) else None
        if px is not None:
            # sharded update: identical z-scores everywhere, GEMV over this rank's P/W members only, one fused
            # barrier + rank-ordered sum + apply over NVLink peer memory (theta / lr stay bit-identical replicas)
            self.update_mode = "sharded: partial GEMV over P/W members + fused peer-memory all-reduce of the update"
            L.call("ppx_es_update_sharded", self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None,
                   r.data_ptr(), P, rk * (P // W), P // W, self.D, float(self.SIGMA), float(self.novelty_param),
                   float(novelty) if (novelty is not None and nov_dev is None) else 0.0,
                   nov_dev.data_ptr() if nov_dev is not None else None, int(novelty is not None), float(self.decay),
                   self._lr.data_ptr(), self._status.data_ptr(), self._ws.data_ptr(), self._dtheta.data_ptr(), px.peer_grad,
                   px.peer_flags[2], px.W, px.rank, px.seq[2], px.status_ptr, L.stream())
            return
        self.update_mode = "single" if W == 1 else "replicated"
        L.call("ppx_es_update", self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None,
               r.data_ptr(), P, self.D, float(self.SIGMA), float(self.novelty_param),
               float(novelty) if (novelty is not None and nov_dev is None) else 0.0,
               nov_dev.data_ptr() if nov_dev is not None else None, int(novelty is not None),
               int(self.fitness_shaping == "centered_rank"), float(self.decay), self._lr.data_ptr(),
               self._status.data_ptr(), self._ws.data_ptr(), L.stream())

    def _update_weights_member(self, r, noise, off, P, novelty):
        if novelty is None:
            raise ValueError("novelty_mode='member' updates with the novelty of every member: pass novelty= (f64 [P])")
        nov = torch.as_tensor(np.asarray(novelty, dtype=np.float64)).to(self.device) if not isinstance(novelty, torch.Tensor) \
            else novelty.to(self.device, torch.float64)
        nov = nov.reshape(-1).contiguous()
        if nov.numel() != P or r.numel() != P:
            raise ValueError(f"member mode needs {P} rewards and {P} novelties, got {r.numel()} and {nov.numel()}")
        need = L.call("ppx_es_update_member_workspace", P, self.D)
        if self._ws is None or self._ws.numel() * 8 < need:
            self._ws = torch.zeros(need // 8 + 1, dtype=torch.float64, device=self.device)
        W, rk = D.world_size(), D.rank()
        rank_mode = int(self.fitness_shaping == "centered_rank")
        px = self._peer_exchange() if (W > 1 and not rank_mode and P % W == 0) else None
        common = (self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None, r.data_ptr(),
                  nov.data_ptr(), P)
        tail = (float(self.SIGMA), float(self.novelty_param), rank_mode, float(self.decay), self._lr.data_ptr(),
                self._status.data_ptr(), self._ws.data_ptr())
        if px is not None:
            self.update_mode = "sharded: partial GEMV over P/W members + fused peer-memory all-reduce of the update"
            L.call("ppx_es_update_member", *common, rk * (P // W), P // W, self.D, *tail, self._dtheta.data_ptr(), px.peer_grad,
                   px.peer_flags[2], px.W, px.rank, px.seq[2], px.status_ptr, L.stream())
            return
        self.update_mode = "single" if W == 1 else "replicated"
        L.call("ppx_es_update_member", *common, 0, P, self.D, *tail, None, None, None, 1, 0, None, None, L.stream())

    def _peer_exchange(self):
        if self._px is False:
            self._px = D.peer_exchange_or_none(2 * self.D, self.device, L.call("ppx_p2p_max_params"))
            if self._px is not None:
                self._dtheta = self._px.grad.view(torch.float64)                  # this rank's partial update, peer-visible
        return self._px

    # ---- ask / tell: the two device-side halves of one ES iteration, each replayed as ONE CUDA graph ----
    def _hp_state(self):
        """Every host scalar the ask / tell graphs bake into kernel arguments: a graph is keyed on these, so a run that
        adapts novelty_param (or a caller that changes sigma / decay / K) replays a graph captured with the current values."""
        return (float(self.novelty_param), float(self.SIGMA), float(self.decay), int(self.K), self.fitness_shaping,
                self.novelty_mode)

    def _graph(self, key, fn):
        ent = self._graphs.get(key)
        if ent is None:
            self._graphs[key] = "warm"
            return fn()
        if ent == "warm":
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                out = fn()
            ent = (g, L.launch_count() - n0, out)
            L.extra_launches -= ent[1]
            self._graphs[key] = ent
        ent[0].replay()
        L.extra_launches += ent[1]
        return ent[2]

    def ask(self, archive=None, queries=None):
        """First half of an iteration: draw the population (:172-182), form theta + sigma*eps for THIS rank's members
        (:137-145) and -- as run() does before it evaluates the population (:318-325) -- the novelty of `queries` against
        the behaviour `archive` (k-NN on a forked stream, under the perturbation).  One CUDA graph.  Returns (offsets [P]
        int64, weights [P/W, D] f32, novelties [Q] f64 | None): static buffers, overwritten by the next ask()."""
        W = D.world_size()
        if not hasattr(self, "_ask_off"):
            self.noise_table()
            self._ask_off = torch.empty(self.POPULATION_SIZE, dtype=torch.int64, device=self.device)
            self._side = torch.cuda.Stream(device=self.device)
        key = ("ask", archive.data_ptr() if archive is not None else 0, queries.data_ptr() if queries is not None else 0,
               archive.shape[0] if archive is not None else 0, self._hp_state())

        def fn():
            nov = None
            if archive is not None:
                cur = torch.cuda.current_stream()
                self._side.wait_stream(cur)
                with torch.cuda.stream(self._side):
                    _, nov = self.novelty_batch(archive, queries)
            pop = self._get_population(out=self._ask_off)
            w = self.perturb_all(self.shard_population(pop) if W > 1 else pop)
            if archive is not None:
                torch.cuda.current_stream().wait_stream(self._side)
            return pop, w, nov
        out = self._graph(key, fn)
        self._novelty = out[2]
        return out

    def tell(self, local_rewards, brain=0, local_novelty=None):
        """Second half (:217-239): exchange the fitness of the rank-local members and update the parameters with the
        novelty of meta-population member `brain` computed by the last ask().  `local_rewards` must be a persistent CUDA
        tensor (its address is captured).  novelty_mode="member": `local_novelty` (required; a persistent CUDA f64 tensor
        [P/W], this rank's members, e.g. `member_novelty(archive, bc)`) goes through the same all-gather as the fitness and
        the update is ppx_es_update_member."""
        member = self.novelty_mode == "member"
        if member != (local_novelty is not None):
            raise ValueError("tell(local_novelty=) is required with novelty_mode='member' and rejected with 'brain'")
        if member:
            L.require_cuda(local_novelty, torch.float64, "local_novelty")
            key = ("tell", local_rewards.data_ptr(), local_novelty.data_ptr(), self._hp_state())
        else:
            key = ("tell", local_rewards.data_ptr(), int(brain), self._novelty.data_ptr() if self._novelty is not None else 0,
                   self._hp_state())

        def fn():
            r_all = self.gather_fitness(local_rewards)
            if member:
                self._update_weights(r_all, self._ask_off, novelty=self.gather_fitness(local_novelty))
                return
            nov = self._novelty[brain:brain + 1] if self._novelty is not None else None
            self._update_weights(r_all, self._ask_off, novelty=nov)
        return self._graph(key, fn)

    # ---- episode evaluation on an env that lives on the GPU (INTEGRATION.md §4) ----
    def evaluate(self, env, population=None, *, max_steps, sigma=None, check_every=8, member_lo=None, uniforms=None):
        """evaluate / get_behavior_char (:153-170) with get_action (:75-95) for a batched env on the GPU: env i runs member i
        (global member member_lo + i) for ONE episode.  Per step two libppx launches and no host sync: `ppx_es_act` (the
        forward of the members still running on the env's f32 observations; Box: tanh(logits) f64 [N, A], Discrete: one
        categorical draw int64 [N]; finished members get action 0) and, after env.step, `ppx_es_episode_step`.

        A member's fitness is the f64 sum, in step order, of its rewards up to and including its first done; later rewards,
        dones and behaviours of its env are ignored.  If the env has `behavior()` (CUDA f64 [N, k], the state reached by the
        last step(), before any auto-reset), a member's row is latched at its terminating step.  A member still running after
        `max_steps` steps keeps the sum so far and the behaviour of that step.  Every `check_every` steps the device count of
        running members is copied into pinned memory without blocking, and the loop stops once a copy reads 0; the steps
        issued after the last member ended change nothing, so the results do not depend on `check_every`.

        population: offsets or dense eps as in `predict_population`; default this rank's slice of the last `ask()` (with
        member_lo = rank * P/W), or with sigma=0.0 and no ask() yet, theta itself on every env (the meta-member behaviour of
        :318-325).  The Discrete draw is numpy's RandomState.choice arithmetic on u = a Philox uniform keyed by (noise seed,
        the device draw counter, step, global member), so every rank draws the same action for the same member; `uniforms`
        (CUDA f64 [max_steps, N]) supplies u instead, e.g. numpy's own draws.
        Returns (fitness f64 [N], lengths int64 [N], behaviour f64 [N, k] or None), CUDA buffers that the next evaluate()
        of the same shape overwrites -- `tell(fitness)` replays its captured graph."""
        if max_steps < 1 or check_every < 1:
            raise ValueError(f"max_steps={max_steps} and check_every={check_every} must be >= 1")
        sig = float(self.SIGMA if sigma is None else sigma)
        N = int(env.num_envs)
        if population is None:
            if hasattr(self, "_ask_off"):
                W = D.world_size()
                population = self.shard_population(self._ask_off) if W > 1 else self._ask_off
                if member_lo is None:
                    member_lo = D.rank() * (self.POPULATION_SIZE // W)
            elif sig == 0.0:
                population = torch.zeros(N, dtype=torch.int64, device=self.device)
            else:
                raise ValueError("evaluate() needs a population: call ask() first or pass one")
        noise, off = self._as_eps(population)
        P = off.numel() if off is not None else noise.shape[0]
        if P != N:
            raise ValueError(f"the env runs {N} envs but the population has {P} members (one env per member)")
        discrete, A = self._env_actions(env)
        if uniforms is not None:
            L.require_cuda(uniforms, torch.float64, "uniforms")
            if tuple(uniforms.shape) != (max_steps, N):
                raise ValueError(f"uniforms must be [{max_steps}, {N}], got {tuple(uniforms.shape)}")
        sizes = [self.shapes[0][0]] + [sh[1] for sh in self.shapes]
        import ctypes as C
        sizes_c = (C.c_int * len(sizes))(*sizes)

        def act(t, o, buf):
            L.call("ppx_es_act", self.theta.data_ptr(), noise.data_ptr(), off.data_ptr() if off is not None else None, sig, N,
                   sizes_c, len(sizes) - 1, o.data_ptr(), buf["alive"].data_ptr(), int(discrete), self._noise_seed + 2,
                   self._draw.data_ptr(), t, int(member_lo or 0), uniforms[t].data_ptr() if uniforms is not None else None,
                   buf["actions"].data_ptr(), L.stream())
        return self._episodes(env, "population", A, discrete, max_steps, check_every, act)

    def _env_actions(self, env):
        """(discrete, number of actions) of env.action_space; ValueError if the network has another number of actions."""
        space = env.action_space
        discrete = getattr(space, "n", None) is not None and not getattr(space, "shape", ())
        A = int(space.n) if discrete else int(space.shape[-1])
        if A != self.shapes[-1][1]:
            raise ValueError(f"the env has {A} actions, the network {self.shapes[-1][1]}")
        return discrete, A

    def _episodes(self, env, tag, A, discrete, max_steps, check_every, act):
        """The device episode loop of evaluate() and of run()'s brains: one episode per env, `act(t, obs f32 [N, D0], buffers)`
        launching the forward that writes buffers["actions"], then env.step and `ppx_es_episode_step`.  `tag` keeps the
        buffers of the two loops apart."""
        N = int(env.num_envs)
        obs = env.reset()
        if not (isinstance(obs, torch.Tensor) and obs.is_cuda):
            raise TypeError("evaluate() steps environments that live on the GPU: env.reset() must return a CUDA tensor "
                            f"(got {type(obs).__name__}); for an env returning numpy, loop over predict_population / "
                            "discrete_action on the host")
        buf = self._eval_buffers(tag, N, A, discrete)
        buf["fitness"].zero_()
        buf["lengths"].zero_()
        buf["alive"].fill_(1)
        buf["state"].zero_()
        has_bc = callable(getattr(env, "behavior", None))
        bc_out = None
        st = L.stream()
        d0 = self.shapes[0][0]
        t = 0
        while t < max_steps:
            o = self._device_input(obs, torch.float32, (N, d0), "observations")
            act(t, o, buf)
            obs, rew, done, _ = env.step(buf["actions"])
            rew = self._device_input(rew, None, (N,), "rewards")
            done = self._device_input(done, torch.uint8, (N,), "dones")
            bc = None
            if has_bc:
                bc = env.behavior()
                if not (isinstance(bc, torch.Tensor) and bc.is_cuda):
                    raise TypeError("env.behavior() must return a CUDA tensor [N, k]")
                bc = bc.reshape(N, -1).to(torch.float64).contiguous()
                if bc_out is None:
                    bc_out = self._eval_bc(tag, N, bc.shape[1])
            L.call("ppx_es_episode_step", rew.data_ptr(), int(rew.dtype == torch.float64), done.data_ptr(),
                   bc.data_ptr() if bc is not None else None, bc.shape[1] if bc is not None else 0, N, int(t == max_steps - 1),
                   buf["alive"].data_ptr(), buf["fitness"].data_ptr(), buf["lengths"].data_ptr(),
                   bc_out.data_ptr() if bc is not None else None, buf["state"].data_ptr(), st)
            t += 1
            if t % check_every == 0 and t < max_steps:
                if buf["polled"] and buf["event"].query() and int(buf["host"][0]) == 0:
                    break
                buf["host"].copy_(buf["state"][2:3], non_blocking=True)
                buf["event"].record()
                buf["polled"] = True
        buf["polled"] = False
        self.last_eval_steps = t
        return buf["fitness"], buf["lengths"], bc_out

    def _eval_buffers(self, tag, N, A, discrete):
        if not hasattr(self, "_eval"):
            self._eval = {}
        key = (tag, N, A, discrete)
        if key not in self._eval:
            dev = self.device
            self._eval[key] = dict(
                fitness=torch.zeros(N, dtype=torch.float64, device=dev), lengths=torch.zeros(N, dtype=torch.int64, device=dev),
                alive=torch.ones(N, dtype=torch.uint8, device=dev), state=torch.zeros(3, dtype=torch.int64, device=dev),
                actions=torch.zeros(N, dtype=torch.int64, device=dev) if discrete else
                torch.zeros(N, A, dtype=torch.float64, device=dev),
                host=torch.zeros(1, dtype=torch.int64).pin_memory(), event=torch.cuda.Event(), polled=False)
        return self._eval[key]

    def _eval_bc(self, tag, N, k):
        key = ("bc", tag, N, k)
        if key not in self._eval:
            self._eval[key] = torch.zeros(N, k, dtype=torch.float64, device=self.device)
        return self._eval[key]

    def _device_input(self, x, dtype, shape, name):
        """An env output as a contiguous CUDA tensor of `shape`: dtype None keeps f32 / f64 (other types become f64); uint8
        accepts bool as is.  Numpy arrays are copied up (an env on the GPU returns CUDA tensors)."""
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(np.asarray(x)).to(self.device)
        if dtype is None:
            dtype = x.dtype if x.dtype in (torch.float32, torch.float64) else torch.float64
        if dtype == torch.uint8 and x.dtype == torch.bool:
            x = x.view(torch.uint8)
        elif dtype == torch.uint8 and x.dtype != torch.uint8:
            x = (x != 0).to(torch.uint8)
        x = x.to(dtype).reshape(shape).contiguous()
        if x.device != self.theta.device:
            raise ValueError(f"{name} live on {x.device}, the ES on {self.theta.device}")
        return x

    def run_generation(self, env, *, max_steps, archive=None, queries=None, brain=0, check_every=8):
        """One ES generation on an env that lives on the GPU: ask() -> evaluate() of this rank's members -> tell().  Sharded,
        every rank evaluates its P/W envs and tell() gathers the fitness.  Returns what evaluate() returned.
        novelty_mode="member": ask() -> evaluate() (the env must have behavior()) -> member_novelty(archive, BCs) -> tell();
        `archive` (f64 CUDA [n, k]) is required and `queries` / `brain` are not used."""
        if self.novelty_mode == "member":
            if archive is None:
                raise ValueError("run_generation() with novelty_mode='member' scores the members against archive=")
            self.ask()
            out = self.evaluate(env, max_steps=max_steps, check_every=check_every)
            if out[2] is None:
                raise TypeError("novelty_mode='member' characterises the members by env.behavior() (CUDA f64 [N, k])")
            nov = self._member_nov_buffer(out[2].shape[0])
            self.member_novelty(archive, out[2], out=nov)
            self.tell(out[0], local_novelty=nov)
            return out
        self.ask(archive, queries)
        out = self.evaluate(env, max_steps=max_steps, check_every=check_every)
        self.tell(out[0], brain=brain)
        return out

    def _member_nov_buffer(self, n):
        """The persistent [n] f64 buffer of this rank's member novelties that the captured tell() graph reads."""
        buf = getattr(self, "_member_nov", None)
        if buf is None or buf.numel() != n:
            buf = self._member_nov = torch.zeros(n, dtype=torch.float64, device=self.device)
        return buf

    # ---- the ES-NSRA run loop (evolution_strategies.py:293-384, order of SURVEY §3.4; DESIGN.md §3.15) ----
    def run(self, env, brain_env, iterations, *, max_steps, meta_population_size=2, reward_target=None, log_interval=1,
            log_to_file=False, check_every=8):
        """Train a meta-population of M = meta_population_size parameter vectors (`thetas`, f64 [M, D]) with ES-NSRA for up
        to `iterations` generations.  `env` runs the population (P envs, P/W per rank when sharded), `brain_env` M envs, one
        episode per brain at sigma = 0 (identical on every rank: same seed, env_offset=0); both live on the GPU
        (INTEGRATION.md §4) and brain_env has behavior().  The first run() keeps the constructor's theta as brain 0 and
        draws brains 1..M-1 from numpy's global RNG as the constructor draws theta, runs the brains once and seeds the
        behaviour archive with all M characterisations (BCs).  Each generation then
          1. computes every brain's novelty against the archive (one ppx_knn_novelty launch) and reads it to the host with
             the previous generation's log row -- the generation's one blocking device->host read;
          2. picks brain b with pick_brain (numpy's global RNG), copies thetas[b] into theta and runs ask() -> evaluate(env)
             -> tell() with novelty nu_b and the current novelty_param, then copies theta back into thetas[b];
          3. runs the brains on brain_env (one ppx_es_act_rows + one ppx_es_episode_step launch per step), appends BC_b to the
             archive, and -- once f_b, brain b's episode return, is on the host -- adapts novelty_param every 5 generations,
             logs the row and stops when f_b > reward_target.
        The adaptation is ppx's rule (the reference stores nsr_plateu / nsr_range / nsr_update; its use of them is not
        pinned, oracle/es_nsra.py `nsr_adapt`): with R the best f_b of the last 5 generations and B the best before them,
        novelty_param -= nsr_update (at least nsr_range[0]) if R > B + nsr_plateu, else += nsr_update (at most
        nsr_range[1]); then B = max(B, R).  A later run() (or one after `load`) continues the run.  Logged through
        `ppo_exploration_b200.logger` as ("ES", env_id): iteration, total_time, reward (f_b), brain, novelty_param (the
        weight of the generation's update), learning_rate, fitness_mean, fitness_max, archive_size.
        novelty_mode="member" (NSRA-ES, DESIGN.md §3.16): `env` must have behavior() too.  After evaluate(env), one
        ppx_knn_novelty_many launch scores this rank's members' BCs against the archive as it stands before BC_b is appended
        (M passed by value, so the tell graph is never recaptured as the archive grows), and tell() updates brain b with the
        members' own novelties.  The log gains novelty_mean, the population's mean novelty.  Returns self."""
        import time
        from . import logger as ppx_logger
        M, W = int(meta_population_size), D.world_size()
        if M < 1 or iterations < 0 or max_steps < 1 or check_every < 1 or log_interval < 1:
            raise ValueError("run() needs meta_population_size, max_steps, check_every, log_interval >= 1, iterations >= 0")
        if int(env.num_envs) * W != self.POPULATION_SIZE:
            raise ValueError(f"env runs {int(env.num_envs)} envs per rank; the population of {self.POPULATION_SIZE} needs "
                             f"{self.POPULATION_SIZE // W} on each of {W} rank(s)")
        if int(brain_env.num_envs) != M:
            raise ValueError(f"brain_env runs {int(brain_env.num_envs)} envs, the meta-population has {M} brains")
        if not callable(getattr(brain_env, "behavior", None)):
            raise TypeError("run() characterises the brains by brain_env.behavior() (CUDA f64 [M, k])")
        member = self.novelty_mode == "member"
        if member and not callable(getattr(env, "behavior", None)):
            raise TypeError("run() with novelty_mode='member' characterises the members by env.behavior() (CUDA f64 [N, k])")
        if W > 1 and getattr(brain_env, "env_offset", 0) != 0:
            raise ValueError("every rank must step the same brain_env: build it with env_offset=0")
        if self.thetas is not None and self.thetas.shape[0] != M:
            raise ValueError(f"this run has {self.thetas.shape[0]} brains, not meta_population_size={M}")
        self._env_actions(env)
        self._env_actions(brain_env)
        ppx_logger.configure("ES", str(self.env_id), log_to_file)
        self._run_envs = (env, brain_env)
        if W > 1:
            self._check_rng_replicas()
        if self.thetas is None:
            self._start_run(brain_env, M, max_steps, check_every)
        start = time.time()
        pending = None                                          # (brain, novelty weight) of the generation whose row is on the device
        for _ in range(iterations):
            self._knn_into(self._run_dev[:M])
            vals = self._run_read()
            if pending is not None and self._finish_generation(pending, vals, M, start, log_interval, reward_target):
                pending = None
                break
            b, _ = self.pick_brain([float(v) for v in vals[:M]])
            w = float(self.novelty_param)
            self.theta.copy_(self.thetas[b])
            self.ask()
            if member:
                fit, _, bc_p = self.evaluate(env, max_steps=max_steps, check_every=check_every)
                nov_p = self._member_nov_buffer(bc_p.shape[0])
                L.call("ppx_knn_novelty_many", self._archive.data_ptr(), self._archive_n, bc_p.data_ptr(), bc_p.shape[0],
                       bc_p.shape[1], int(self.K), None, nov_p.data_ptr(), L.stream())
                self.tell(fit, local_novelty=nov_p)
            else:
                nu_b = self._run_dev[M + 4:M + 5]               # tell() mixes in nu_b from a fixed slot: one graph for every brain
                nu_b.copy_(self._run_dev[b:b + 1])
                self._novelty = nu_b
                fit = self.evaluate(env, max_steps=max_steps, check_every=check_every)[0]
                self.tell(fit)
            self.thetas[b].copy_(self.theta)
            bc, f = self._brains(brain_env, max_steps, check_every)
            self._bc_m.copy_(bc)
            self._f_m.copy_(f)
            self._archive_append(bc[b])
            fit_all = self.gather_fitness(fit)
            row = self._run_dev
            row[M].copy_(f[b])
            row[M + 1].copy_(fit_all.mean())
            row[M + 2].copy_(fit_all.max())
            row[M + 3].copy_(self._lr[0])
            if member:
                row[M + 4].copy_(self.gather_fitness(nov_p).mean())
            self._generation += 1
            pending = (b, w)
        if pending is not None:
            self._finish_generation(pending, self._run_read(), M, start, log_interval, reward_target)
        return self

    def _start_run(self, brain_env, M, max_steps, check_every):
        """Brain 0 = theta, brains 1..M-1 drawn layer by layer from numpy's global RNG (the constructor's order), one brain
        loop, the archive seeded with every brain's BC."""
        rest = [np.concatenate([np.random.randn(*s).ravel() for s in self.shapes]) for _ in range(M - 1)]
        self.thetas = torch.empty(M, self.D, dtype=torch.float64, device=self.device)
        self.thetas[0].copy_(self.theta)
        if rest:
            self.thetas[1:].copy_(torch.as_tensor(np.stack(rest)))
        bc, f = self._brains(brain_env, max_steps, check_every)
        self._run_buffers(M, bc.shape[1])
        self._bc_m.copy_(bc)
        self._f_m.copy_(f)
        for m in range(M):
            self._archive_append(bc[m])
        self._fb_window, self._best, self._generation = [], -float("inf"), 0

    def _run_buffers(self, M, k, capacity=16):
        self._archive = torch.empty(capacity, k, dtype=torch.float64, device=self.device)
        self._archive_n = 0
        self._bc_m = torch.empty(M, k, dtype=torch.float64, device=self.device)
        self._f_m = torch.empty(M, dtype=torch.float64, device=self.device)
        self._knn_sums = torch.empty(M, dtype=torch.float64, device=self.device)
        # [nu_0 .. nu_M-1, f_b, fitness mean, fitness max, lr | nu_b]: the first M + 4 are the generation's read; member
        # mode reads one more slot, M + 4 = the population's mean novelty (it has no nu_b)
        self._run_dev = torch.zeros(M + 5, dtype=torch.float64, device=self.device)
        self._run_host = torch.zeros(M + 4 + (self.novelty_mode == "member"), dtype=torch.float64).pin_memory()
        self._run_event = torch.cuda.Event()

    def _archive_append(self, row):
        """One BC row onto the device archive; the host keeps the count, and the capacity doubles when it is full."""
        n = self._archive_n
        if n == self._archive.shape[0]:
            grown = torch.empty(2 * n, self._archive.shape[1], dtype=torch.float64, device=self.device)
            grown[:n].copy_(self._archive)
            self._archive = grown
        self._archive[n].copy_(row)
        self._archive_n = n + 1

    @property
    def archive(self):
        """The behaviour archive of run(): f64 CUDA [n, k] (a view), or None before the first run()."""
        return None if self.thetas is None else self._archive[:self._archive_n]

    def _knn_into(self, nov):
        """nov [M] = the novelty of every brain's last BC against the archive (one launch)."""
        L.call("ppx_knn_novelty", self._archive.data_ptr(), self._archive_n, self._bc_m.data_ptr(), self._bc_m.shape[0],
               self._bc_m.shape[1], int(self.K), self._knn_sums.data_ptr(), nov.data_ptr(), L.stream())

    def _run_read(self):
        """The generation's one blocking read: the device row [novelties, previous f_b, fitness mean / max, lr] into pinned
        memory, then an event wait."""
        self._run_host.copy_(self._run_dev[:self._run_host.numel()], non_blocking=True)
        self._run_event.record()
        self._run_event.synchronize()
        return self._run_host.numpy().copy()

    def _finish_generation(self, pending, vals, M, start, log_interval, reward_target):
        """Host half of the generation whose row `vals` holds: the f_b window, novelty_param, the log row.  True when f_b
        exceeds reward_target."""
        import time
        from . import logger as ppx_logger
        b, w = pending
        fb = float(vals[M])
        self._fb_window.append(fb)
        if len(self._fb_window) == 5:                           # ppx's adaptation rule (docstring of run())
            R = max(self._fb_window)
            if R > self._best + self.nsr_plateu:
                self.novelty_param = float(max(self.nsr_range[0], self.novelty_param - self.nsr_update))
            else:
                self.novelty_param = float(min(self.nsr_range[1], self.novelty_param + self.nsr_update))
            self._best = max(self._best, R)
            self._fb_window = []
        if self._generation % log_interval == 0:
            for key, v in (("time/iteration", self._generation), ("time/total_time", time.time() - start), ("es/reward", fb),
                           ("es/brain", b), ("es/novelty_param", w), ("es/learning_rate", float(vals[M + 3])),
                           ("es/fitness_mean", float(vals[M + 1])), ("es/fitness_max", float(vals[M + 2])),
                           ("es/archive_size", self._archive_n)) + ((("es/novelty_mean", float(vals[M + 4])),)
                                                                    if self.novelty_mode == "member" else ()):
                ppx_logger.record(key, v)
            ppx_logger.dump(step=self._generation)
        return reward_target is not None and fb > reward_target

    def _brains(self, brain_env, max_steps, check_every):
        """One episode per brain on brain_env: row m acts with thetas[m] at sigma = 0 (ppx_es_act_rows; Discrete draws on
        their own Philox key, noise seed + 3).  Returns (BC f64 [M, k], episode return f64 [M])."""
        import ctypes as C
        discrete, A = self._env_actions(brain_env)
        M = self.thetas.shape[0]
        sizes = [self.shapes[0][0]] + [sh[1] for sh in self.shapes]
        sizes_c = (C.c_int * len(sizes))(*sizes)
        noise = self.noise_table()

        def act(t, o, buf):
            L.call("ppx_es_act_rows", self.thetas.data_ptr(), noise.data_ptr(), M, sizes_c, len(sizes) - 1, o.data_ptr(),
                   buf["alive"].data_ptr(), int(discrete), self._noise_seed + 3, self._draw.data_ptr(), t,
                   buf["actions"].data_ptr(), L.stream())
        fit, _, bc = self._episodes(brain_env, "brains", A, discrete, max_steps, check_every, act)
        return bc, fit

    def _check_rng_replicas(self):
        """Sharded run(): every rank must make the same brain picks, so numpy's global RNG must be in the same state on
        every rank (the learners' "global" convention)."""
        digest = D.rng_digest(np.random.get_state())
        seen = D.all_gather_cat(torch.tensor([digest], dtype=torch.int64, device=self.device)).cpu().numpy().ravel()
        if not (seen == seen[0]).all():
            raise RuntimeError("ppx: a sharded ES run() needs numpy's global RNG in the same state on every rank (seed all "
                               "ranks alike and keep rank-dependent draws off np.random); digests: %s" % seen.tolist())

    @property
    def update_skipped(self):
        return bool(self._status.item())

    def centered_ranks(self, rewards):
        r = torch.as_tensor(np.asarray(rewards, dtype=np.float64)).to(self.device)
        ranks = torch.empty(r.numel(), dtype=torch.int64, device=self.device)
        cen = torch.empty(r.numel(), dtype=torch.float64, device=self.device)
        L.call("ppx_rank_center", r.data_ptr(), r.numel(), ranks.data_ptr(), cen.data_ptr(), L.stream())
        return ranks, cen

    # ---- novelty ----
    def novelty_batch(self, archive, queries, K=None):
        """archive [M,dim], queries [Q,dim] -> (knn distance sums [Q], novelties [Q]) f64 CUDA."""
        a = torch.as_tensor(np.concatenate(archive) if isinstance(archive, list) else np.asarray(archive)) \
            if not isinstance(archive, torch.Tensor) else archive
        a = a.to(self.device, torch.float64).contiguous()
        q = (torch.as_tensor(np.asarray(queries)) if not isinstance(queries, torch.Tensor) else queries)
        q = q.to(self.device, torch.float64).reshape(-1, a.shape[1]).contiguous()
        K = self.K if K is None else K
        s = torch.empty(q.shape[0], dtype=torch.float64, device=self.device)
        nov = torch.empty_like(s)
        L.call("ppx_knn_novelty", a.data_ptr(), a.shape[0], q.data_ptr(), q.shape[0], a.shape[1], int(K), s.data_ptr(),
               nov.data_ptr(), L.stream())
        return s, nov

    def member_novelty(self, archive, behaviors, out=None):
        """The novelty of every row of `behaviors` [n, k] against `archive` [M, k] (both f64 CUDA, or array-likes): f64 CUDA
        [n], with ppx_knn_novelty's values bit for bit, one thread per query (ppx_knn_novelty_many; k <= 8).  `out`: an f64
        CUDA [n] buffer to write into."""
        a = archive if isinstance(archive, torch.Tensor) else torch.as_tensor(np.asarray(archive, np.float64))
        a = a.to(self.device, torch.float64).contiguous()
        q = behaviors if isinstance(behaviors, torch.Tensor) else torch.as_tensor(np.asarray(behaviors, np.float64))
        q = q.to(self.device, torch.float64).reshape(-1, a.shape[1]).contiguous()
        if out is None:
            out = torch.empty(q.shape[0], dtype=torch.float64, device=self.device)
        L.require_cuda(out, torch.float64, "out")
        if out.numel() != q.shape[0]:
            raise ValueError(f"out has {out.numel()} entries for {q.shape[0]} behaviours")
        L.call("ppx_knn_novelty_many", a.data_ptr(), a.shape[0], q.data_ptr(), q.shape[0], a.shape[1],
               int(self.K), None, out.data_ptr(), L.stream())
        return out

    def get_kNN(self, archive, bc, n_neighbors):
        """:264-281: summed distance to the n_neighbors nearest archive entries (python float)."""
        s, _ = self.novelty_batch(archive, bc, K=n_neighbors)
        return float(s[0].item())

    def get_novelty_from_bc(self, archive, bc):
        """:318-325 (dup :208-214) given the behaviour characterisation instead of a policy rollout."""
        _, nov = self.novelty_batch(archive, bc)
        return float(nov[0].item())

    def calc_noveltiy_distribution(self, novelties):
        """:283-290 (host; MPS = 2 scalars)."""
        return [round((n / (sum(novelties))), 4) for n in novelties]

    def pick_brain(self, novelties):
        """:327-333: the meta-population member to train next -- probabilities from calc_noveltiy_distribution,
        renormalised (the rounding to 4 digits breaks the unit sum), one np.random.choice draw from the reference's host
        RNG.  Returns (brain_idx, novelty of that member)."""
        probs = np.array(self.calc_noveltiy_distribution(novelties))
        probs /= probs.sum()
        idx = int(np.random.choice(list(range(len(probs))), p=probs))
        return idx, novelties[idx]
