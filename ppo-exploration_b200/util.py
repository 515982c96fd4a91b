"""Device-side helpers mirroring util.py of the reference."""
import numpy as np
import torch

from . import _lib as L


class RunningMeanStd(object):
    """util.py:9-44 with the float64 moments resident on the GPU (no host sync per update).

    `mean`, `var`, `count` properties copy the state to the host on demand (tests, checkpointing)."""

    def __init__(self, epsilon=1e-4, shape=(), device="cuda", sharded=False):
        # sharded (SURVEY §8e row 4): under torch.distributed every rank feeds the rows of ITS env shard; the rows of all
        # ranks are all-gathered in rank (= global env) order first, so the update sees exactly the batch a single GPU
        # holding every env would see and the running moments stay bit-identical replicas
        self.sharded = bool(sharded)
        self.device = torch.device(device)
        self.shape = tuple(shape)
        self.dim = int(np.prod(shape)) if len(shape) else 1
        self.mean_dev = torch.zeros(self.dim, dtype=torch.float64, device=self.device)
        self.var_dev = torch.ones(self.dim, dtype=torch.float64, device=self.device)
        self.count_dev = torch.full((1,), float(epsilon), dtype=torch.float64, device=self.device)

    def update(self, arr):
        """arr: [n, *shape] numpy or tensor (f32 or f64)."""
        if not isinstance(arr, torch.Tensor):
            arr = torch.as_tensor(np.ascontiguousarray(arr))
        if arr.dtype not in (torch.float32, torch.float64):
            arr = arr.float()
        x = arr.to(self.device).reshape(-1, self.dim).contiguous()
        if self.sharded:
            from . import dist as D
            if D.world_size() > 1:
                x = D.all_gather_cat(x).reshape(-1, self.dim)
        L.call("ppx_rms_update", x.data_ptr(), int(x.dtype == torch.float64), x.shape[0], self.dim,
               self.mean_dev.data_ptr(), self.var_dev.data_ptr(), self.count_dev.data_ptr(), None, L.stream())

    def istd(self):
        """1/sqrt(var + 1e-10) (f64, device): the scale of normalize_obs, for kernels that normalise on the fly."""
        if getattr(self, "_istd", None) is None:
            self._istd = torch.empty(self.dim, dtype=torch.float64, device=self.device)
        L.call("ppx_obs_istd", self.var_dev.data_ptr(), self.dim, self._istd.data_ptr(), L.stream())
        return self._istd

    def state_dict(self):
        """The f64 moments as CPU tensors (checkpoints)."""
        return {"mean": self.mean_dev.cpu(), "var": self.var_dev.cpu(), "count": self.count_dev.cpu()}

    def load_state_dict(self, sd):
        from .checkpoint import tensor_into
        for k in ("mean", "var", "count"):
            tensor_into(getattr(self, k + "_dev"), sd[k], f"running statistics '{k}'")

    def set_state(self, mean, var, count):
        self.mean_dev.copy_(torch.as_tensor(np.asarray(mean, dtype=np.float64)).reshape(-1))
        self.var_dev.copy_(torch.as_tensor(np.asarray(var, dtype=np.float64)).reshape(-1))
        self.count_dev.fill_(float(count))

    @property
    def mean(self):
        return self.mean_dev.cpu().numpy().reshape(self.shape)

    @property
    def var(self):
        return self.var_dev.cpu().numpy().reshape(self.shape)

    @property
    def count(self):
        return float(self.count_dev.item())


def normalize_obs(obs, rms, out=None):
    """BaseAlgorithm.normalize_obs (algorithms.py:111-118) on device: f64 math, f32 result
    (the reference casts to f32 at the consumer, models.py:262 / algorithms.py:495)."""
    x = obs.reshape(-1, obs.shape[-1]).contiguous()
    if out is None:
        out = torch.empty_like(x)
    L.call("ppx_normalize_obs", x.data_ptr(), x.shape[0], x.shape[1], rms.mean_dev.data_ptr(), rms.var_dev.data_ptr(),
           out.data_ptr(), L.stream())
    return out
