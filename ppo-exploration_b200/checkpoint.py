"""The checkpoint file format of the learners and of ES (DESIGN.md §3.14).

A checkpoint is one `torch.save` file that loads with `torch.load(path, weights_only=True)`: CPU tensors, Python scalars
and strings, and lists and dicts of these -- no pickled objects.  The top level carries `format`, `version` and the class
name of what was saved.  Under torch.distributed every rank writes its own file.
"""
import numpy as np
import torch

FORMAT = "ppx-checkpoint"
VERSION = 1


def header(cls_name):
    return {"format": FORMAT, "version": VERSION, "class": cls_name}


def read(path, cls_name):
    """The checkpoint at `path`, after checking its format, version and class; ValueError if any does not fit."""
    ck = torch.load(path, map_location="cpu", weights_only=True)
    check(ck, cls_name)
    return ck


def check(ck, cls_name):
    if not isinstance(ck, dict) or ck.get("format") != FORMAT:
        raise ValueError("not a ppx checkpoint (no format tag 'ppx-checkpoint')")
    if ck.get("version") != VERSION:
        raise ValueError(f"checkpoint format version {ck.get('version')!r}; this ppx reads version {VERSION}")
    if ck.get("class") != cls_name:
        raise ValueError(f"the checkpoint holds a {ck.get('class')!r}, not a {cls_name!r}")


# counters added after version 1 was first written, with the value a file without them stands for
_COUNTER_DEFAULTS = {"eval_draws": 0}


def counters(ck):
    """The checkpoint's counters, with the default of every counter the file predates."""
    return dict(_COUNTER_DEFAULTS, **ck["counters"])


def np_rng_state(state=None):
    """numpy's legacy MT19937 state (default: the global `np.random` one) as a uint32 key tensor plus ints and a float."""
    name, key, pos, has_gauss, cached = np.random.get_state() if state is None else state
    if name != "MT19937":
        raise ValueError(f"unsupported numpy bit generator {name!r}")
    return {"key": torch.from_numpy(np.array(key, dtype=np.uint32)), "pos": int(pos), "has_gauss": int(has_gauss),
            "cached_gaussian": float(cached)}


def np_rng_tuple(d):
    """Inverse of `np_rng_state`: a tuple for `np.random.set_state`."""
    key = d["key"]
    if key.dtype != torch.uint32 or key.numel() != 624:
        raise ValueError("numpy RNG state: the key must be 624 uint32 words")
    return ("MT19937", key.numpy().astype(np.uint32), int(d["pos"]), int(d["has_gauss"]), float(d["cached_gaussian"]))


def scalar(v):
    """A Python scalar for a numpy / Python one (the file holds no numpy objects)."""
    return v.item() if isinstance(v, np.generic) else v


def pack(x):
    """An observation / done array as it sits in the learner: a CUDA (or CPU) tensor or a numpy array, or None."""
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        return {"kind": "tensor", "cuda": bool(x.is_cuda), "data": x.detach().cpu().clone()}
    return {"kind": "numpy", "data": torch.from_numpy(np.array(x))}


def unpack(d, device):
    if d is None:
        return None
    if d["kind"] == "numpy":
        return d["data"].numpy().copy()
    return d["data"].to(device) if d["cuda"] else d["data"].clone()


def tensor_into(dst, src, what):
    """dst.copy_(src) after checking shape and dtype (ValueError on a mismatch)."""
    if tuple(src.shape) != tuple(dst.shape) or src.dtype != dst.dtype:
        raise ValueError(f"checkpoint {what}: {tuple(src.shape)} {src.dtype}, expected {tuple(dst.shape)} {dst.dtype}")
    dst.copy_(src)
