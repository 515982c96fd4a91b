"""GPU parity: shuffle indices and minibatch gather are bit-exact vs the reference fixtures."""
import numpy as np
import pytest
import torch

from conftest import Golden
from oracle import rollout as OR

pytestmark = pytest.mark.gpu


def test_get_single_golden():
    import ppo_exploration_b200 as ppx
    g = Golden("get_single")
    raw = g.group("raw")
    buf = ppx.RolloutStorage(8, 3, ppx.Box((4,)), ppx.Box((2,)))
    buf.load_rollout(**{k: raw[k] for k in ("observations", "actions", "values", "action_log_probs", "advantages",
                                           "returns", "rewards", "masks")})
    np.random.seed(123)
    for ep in range(2):
        batches = list(buf.get(5))
        assert len(batches) == 5 and batches[-1].observations.shape[0] == 4          # ragged last minibatch
        for bi, b in enumerate(batches):
            for f in b._fields:
                want = g[f"ep{ep}/b{bi}/{f}"]
                got = getattr(b, f).cpu().numpy()
                assert got.shape == want.shape and got.dtype == want.dtype and np.array_equal(got, want), (ep, bi, f)
    assert buf.generator_ready
    assert np.array_equal(buf.flat("values").cpu().numpy(), OR.swap_and_flatten(raw["values"]))


def test_get_dual_golden():
    import ppo_exploration_b200 as ppx
    g = Golden("get_dual")
    raw = g.group("raw")
    buf = ppx.IntrinsicStorage(8, 3, ppx.Box((4,)), ppx.Discrete(3))
    buf.load_rollout(**raw)
    np.random.seed(77)
    for bi, b in enumerate(buf.get(7)):
        assert b._fields == ('observations', 'actions', 'old_values', 'int_values', 'old_log_probs', 'advantages',
                             'int_advantages', 'returns', 'int_returns')
        for f in b._fields:
            want = g[f"b{bi}/{f}"]
            got = getattr(b, f).cpu().numpy()
            assert got.shape == want.shape and np.array_equal(got, want), (bi, f)


def test_get_requires_full():
    import ppo_exploration_b200 as ppx
    buf = ppx.RolloutStorage(4, 2, ppx.Box((3,)), ppx.Box((1,)))
    with pytest.raises(AssertionError):
        next(buf.get(2))


@pytest.mark.parametrize("T,N,D,A,B", [(256, 2048, 8, 2, 131072), (16, 5, 28224, 1, 17), (128, 8, 4, 1, 128)])
def test_gather_vs_oracle_sizes(T, N, D, A, B):
    import ppo_exploration_b200 as ppx
    rs = np.random.RandomState(T)
    buf = ppx.RolloutStorage(T, N, ppx.Box((D,)), ppx.Box((A,)))
    arrs = dict(observations=rs.randn(T, N, D).astype(np.float32), actions=rs.randn(T, N, A),
                values=rs.randn(T, N).astype(np.float32), action_log_probs=rs.randn(T, N, A).astype(np.float32),
                advantages=rs.randn(T, N).astype(np.float32), returns=rs.randn(T, N).astype(np.float32))
    buf.load_rollout(**arrs)
    np.random.seed(5)
    it = buf.get(B)
    b0 = next(it)
    np.random.seed(5)
    perm = OR.epoch_permutation(T, N)
    want = OR.gather_single(arrs, perm[:B])
    for f in b0._fields:
        assert np.array_equal(getattr(b0, f).cpu().numpy(), want[f]), f
    # a permutation gathers every row exactly once: checksum over the whole epoch
    tot = b0.returns.double().sum().item() + sum(b.returns.double().sum().item() for b in it)
    np.testing.assert_allclose(tot, arrs["returns"].astype(np.float64).sum(), rtol=1e-9)


@pytest.mark.parametrize("n", [1, 2, 3, 7, 1000, 4097, 524288, (1 << 21) + 5, 1 << 24, (1 << 24) + 1, (1 << 25) + 3])
def test_device_shuffle_apply_matches_numpy(n):
    """Fisher-Yates swaps resolved in parallel on the device (shuffle_dev.cu) == np.random.permutation, bit for bit;
    the draws (the RNG stream itself) stay on the host and leave numpy's state where numpy would."""
    import ctypes as C
    from ppo_exploration_b200 import _lib as L
    np.random.seed(n % 1000)
    st = np.random.get_state()
    want = np.random.permutation(n)
    after = np.random.get_state()
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = C.c_int(int(st[2]))
    j = np.zeros(n, np.int32)
    L.call("ppx_np_shuffle_draws32", key.ctypes.data, C.byref(pos), n, j.ctypes.data)
    assert np.array_equal(key, after[1]) and pos.value == after[2]
    # the streaming (AVX-512) draw loop leaves the same list in acceptance order: entry r belongs to position n-1-r
    key2 = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos2, acc = C.c_int(int(st[2])), np.zeros(n, np.int32)
    L.call("ppx_np_shuffle_draws32_stream", key2.ctypes.data, C.byref(pos2), n, acc.ctypes.data)
    assert np.array_equal(key2, after[1]) and pos2.value == after[2]
    ws = torch.empty(L.call("ppx_np_shuffle_apply_device_workspace", n), dtype=torch.uint8, device="cuda")
    out = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    for lst, order in ((j, 0), (acc, 1), (j, 0)):            # repeated: the workspace is reusable, the result does not depend on atomic order
        jd = torch.as_tensor(lst).cuda()
        out.fill_(-1)
        L.call("ppx_np_shuffle_apply_device", jd.data_ptr(), n, order, ws.data_ptr(), out.data_ptr(), L.stream())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want)


def _check_train_stages_numpy_permutations(T, N, batch_size, n_epochs, calls):
    """Every PPO.train() call stages each epoch's np.random.permutation(T*N) on the device bit for bit, drawn from the
    global numpy stream as the reference draws it, and leaves numpy's state where those draws leave it."""
    import ppo_exploration_b200 as ppx
    D, A, total = 8, 2, T * N
    np.random.seed(3)
    want = [np.random.permutation(total) for _ in range(calls * n_epochs)]
    after = np.random.get_state()
    env = ppx.SyntheticVecEnv(N, D, ppx.Box((A,)), seed=0)
    m = ppx.PPO(env=env, nstep=T, hidden_size=64, batch_size=batch_size, n_epochs=n_epochs)
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *shape: torch.randn(*shape, generator=g, device="cuda")
    m.rollout.load_rollout(observations=rnd(T, N, D), actions=rnd(T, N, A).double(), rewards=rnd(T, N), values=rnd(T, N),
                           masks=(torch.rand(T, N, generator=g, device="cuda") < 0.05).to(torch.uint8),
                           action_log_probs=-1.0 + 0.1 * rnd(T, N, A))
    m.rollout.compute_returns_and_advantages(torch.zeros(N), torch.zeros(N))
    np.random.seed(3)
    for c in range(calls):
        spec = m._spec[0] if m._spec is not None else None
        m.train()
        assert c == 0 or m._last_rng is spec
        got = m._perm_all.view(n_epochs, total).cpu().numpy()
        for e in range(n_epochs):
            assert np.array_equal(got[e], want[c * n_epochs + e]), (c, e)
    st = np.random.get_state()
    assert np.array_equal(st[1], after[1]) and st[2] == after[2]


def test_train_stages_numpy_permutations():
    """Three train() calls: the 2nd and 3rd run on the stream pre-drawn by the call before."""
    _check_train_stages_numpy_permutations(32, 16, 128, 3, 3)


def test_train_stages_numpy_permutations_above_2_24():
    """2^24 + 4096 indices per epoch, in minibatches of C2's size."""
    _check_train_stages_numpy_permutations(4097, 4096, 131072, 2, 1)
