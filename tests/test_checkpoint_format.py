"""Host-side pieces of the checkpoint format (no GPU): numpy's RNG state encoding and the header validation."""
import numpy as np
import pytest
import torch

import ppo_exploration_b200 as ppx
from ppo_exploration_b200 import checkpoint as CK


@pytest.mark.parametrize("gauss", [False, True])
def test_numpy_state_round_trip(tmp_path, gauss):
    np.random.seed(1234)
    np.random.permutation(1000)
    if gauss:
        np.random.randn()                                       # leaves a cached gaussian (has_gauss = 1)
    st = np.random.get_state()
    assert st[3] == int(gauss)
    torch.save({"rng": CK.np_rng_state()}, tmp_path / "s.pt")
    d = torch.load(tmp_path / "s.pt", weights_only=True)["rng"]
    assert d["key"].dtype == torch.uint32 and d["key"].numel() == 624
    want = [np.random.randn(7), np.random.permutation(50), np.random.rand(3)]
    np.random.seed(0)                                           # anywhere else
    np.random.set_state(CK.np_rng_tuple(d))
    got = [np.random.randn(7), np.random.permutation(50), np.random.rand(3)]
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


def test_numpy_state_rejects_bad_key():
    d = CK.np_rng_state()
    with pytest.raises(ValueError):
        CK.np_rng_tuple(dict(d, key=d["key"][:100]))
    with pytest.raises(ValueError):
        CK.np_rng_tuple(dict(d, key=d["key"].to(torch.int64)))


def test_header_validation(tmp_path):
    p = tmp_path / "c.pt"
    torch.save(dict(CK.header("PPO"), x=torch.zeros(2)), p)
    assert CK.read(p, "PPO")["x"].shape == (2,)
    with pytest.raises(ValueError, match="not a 'PPO_RND'"):
        CK.read(p, "PPO_RND")
    torch.save(dict(CK.header("PPO"), version=2), p)
    with pytest.raises(ValueError, match="version"):
        CK.read(p, "PPO")
    torch.save({"format": "something-else", "version": 1, "class": "PPO"}, p)
    with pytest.raises(ValueError, match="not a ppx checkpoint"):
        CK.read(p, "PPO")
    torch.save([1, 2, 3], p)
    with pytest.raises(ValueError, match="not a ppx checkpoint"):
        CK.read(p, "PPO")


def test_learner_and_es_check_the_class_first(tmp_path):
    """load() reads and validates the header before it builds anything, so a wrong file fails without a GPU."""
    p = tmp_path / "c.pt"
    torch.save(CK.header("PPO"), p)
    with pytest.raises(ValueError):
        ppx.PPO_ICM.load(p, env=None)
    with pytest.raises(ValueError):
        ppx.EvolutionStrategy.load(p)


def test_pack_unpack_host_arrays():
    for a in (np.arange(6, dtype=np.float32).reshape(2, 3), np.array([True, False, True]), np.zeros(4, dtype=np.int64)):
        d = CK.pack(a)
        b = CK.unpack(d, "cpu")
        assert isinstance(b, np.ndarray) and b.dtype == a.dtype and np.array_equal(a, b)
    t = torch.arange(5, dtype=torch.float64)
    u = CK.unpack(CK.pack(t), "cpu")
    assert isinstance(u, torch.Tensor) and torch.equal(t, u) and u.data_ptr() != t.data_ptr()
    assert CK.pack(None) is None and CK.unpack(None, "cpu") is None
    assert type(CK.scalar(np.float64(1.5))) is float and type(CK.scalar(np.int64(3))) is int and CK.scalar("x") == "x"


def test_tensor_into_checks_shape_and_dtype():
    dst = torch.zeros(3)
    CK.tensor_into(dst, torch.ones(3), "x")
    assert torch.equal(dst, torch.ones(3))
    with pytest.raises(ValueError):
        CK.tensor_into(dst, torch.ones(4), "x")
    with pytest.raises(ValueError):
        CK.tensor_into(dst, torch.ones(3, dtype=torch.float64), "x")
