"""CPU-only checks: the C-ABI library loads and exports every declared symbol; host logic; hygiene."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ppo-exploration_b200")


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "ppx.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ppx_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import ppo_exploration_b200 as ppx
    lib = ppx._lib.load()                                     # dlopen only: no CUDA call, works without a GPU
    syms = _header_symbols()
    assert len(syms) >= 35
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/ppx.h but not exported by libppx.so"
    assert set(syms) == set(ppx._lib.SIGNATURES), set(syms) ^ set(ppx._lib.SIGNATURES)
    out = subprocess.run(["nm", "-D", "--defined-only", ppx._lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (ppx_[a-z0-9_]+)", out))
    assert set(syms) <= exported
    assert ppx._lib.call("ppx_version") == 100
    assert ppx._lib.launch_count() == 0


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", os.path.join(PKG, "libppx.so")], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_product_never_touches_the_oracle_or_cpu_fallbacks():
    bad = []
    for dp, _, fs in os.walk(PKG):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                s = open(os.path.join(dp, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", s, flags=re.M) or "/root/reference" in s:
                    bad.append(f)
    assert not bad, bad
    for f in ("bench.py", "__graft_entry__.py"):
        s = open(os.path.join(ROOT, f)).read()
        assert "/root/reference" not in s.replace('os.path.isdir("/root/reference")', ""), f


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import ppo_exploration_b200 as ppx
    monkeypatch.setattr(ppx._lib, "_lib", None)
    monkeypatch.setattr(ppx._lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ppx._lib.load()


def test_cpu_tensors_are_rejected():
    import torch
    import ppo_exploration_b200 as ppx
    with pytest.raises(RuntimeError, match="CUDA"):
        ppx.RolloutStorage(4, 2, ppx.Box((3,)), ppx.Box((1,)), device="cpu")
    with pytest.raises(ValueError):
        ppx.PPO(env_id="Swimmer-v2")
    with pytest.raises(ValueError):
        ppx.EvolutionStrategy("Swimmer-v2", [64, 64])


def test_spaces_and_synthetic_env():
    import ppo_exploration_b200 as ppx
    env = ppx.SyntheticVecEnv(5, 3, ppx.Discrete(4), seed=2)
    o = env.reset()
    o2, r, d, info = env.step(np.zeros(5))
    assert o.shape == o2.shape == (5, 3) and o.dtype == np.float32 and r.shape == (5,) and d.dtype == bool and len(info) == 5
    assert ppx.ActionConverter(ppx.Discrete(4)).action_output == 1 and ppx.ActionConverter(ppx.Box((3,))).num_actions == 3


def test_swap_and_flatten_matches_reference_layout():
    import torch
    import ppo_exploration_b200 as ppx
    from oracle import rollout as OR
    a = np.arange(24, dtype=np.float32).reshape(4, 3, 2)
    b = np.arange(12, dtype=np.float32).reshape(4, 3)
    for x in (a, b):
        got = ppx.BaseBuffer.swap_and_flatten(torch.tensor(x)).numpy()
        assert np.array_equal(got, OR.swap_and_flatten(x))


def _replay_partners(partners):
    """arange(n) with the Fisher-Yates swaps of a stream's partner list applied on the CPU, in acceptance order (entry r
    is the partner of position n-1-r) as shuffle_dev.cu applies them on the GPU."""
    acc = partners.j.tolist()
    n = len(acc)
    a = list(range(n))
    for r in range(n - 1):
        i, j = n - 1 - r, acc[r]
        a[i], a[j] = a[j], a[i]
    return np.array(a, dtype=np.int64)


def test_host_permutation_is_bit_exact_numpy_replay():
    """libppx's host-side MT19937 shuffle == np.random.permutation, and leaves the global stream in step."""
    from ppo_exploration_b200.buffer import np_permutation, HostRngStream
    for n in (0, 1, 2, 3, 17, 1000, 524288):
        np.random.seed(n)
        want = [np.random.permutation(n) for _ in range(2)] + [np.random.randn(3)]
        np.random.seed(n)
        got = [np_permutation(n) for _ in range(2)] + [np.random.randn(3)]
        assert all(np.array_equal(a, b) for a, b in zip(want, got)), n
    np.random.seed(3)
    want = []
    for _ in range(3):                                       # RND's stream: perm, then one randn per minibatch
        want.append(np.random.permutation(1000))
        want += [np.random.randn() for _ in range(2)]
    tail = np.random.randn()
    np.random.seed(3)
    s = HostRngStream(sum([[('perm', 1000), ('randn',), ('randn',)] for _ in range(3)], []))
    for w in want:
        g = s.next()
        assert np.array_equal(_replay_partners(g), w) if isinstance(w, np.ndarray) else g == w
    s.drain()
    np.random.set_state(s.final_state())                    # the stream works on a private copy; the caller commits
    assert np.random.randn() == tail


def test_vectorised_draw_stream_equals_the_scalar_draws():
    """The AVX-512 block generator / 64-wide acceptance path of ppx_np_shuffle_draws32_stream produces the scalar
    path's partner list (in acceptance order) and leaves the MT19937 state at the same word, across sizes that cross
    several mask ranges and end inside a state block."""
    import ctypes as C
    from ppo_exploration_b200 import _lib as L
    for seed, n in ((1, 70), (2, 4097), (3, 65536), (4, 1 << 20), (5, (1 << 22) + 12345)):
        np.random.seed(seed)
        np.random.rand(seed * 37)                           # start part-way through a state block
        st = np.random.get_state()
        key1, pos1 = np.ascontiguousarray(st[1], dtype=np.uint32).copy(), C.c_int(int(st[2]))
        key2, pos2 = key1.copy(), C.c_int(pos1.value)
        j = np.zeros(n, np.int32)
        acc = np.zeros(n, np.int32)
        L.call("ppx_np_shuffle_draws32", key1.ctypes.data, C.byref(pos1), n, j.ctypes.data)
        L.call("ppx_np_shuffle_draws32_stream", key2.ctypes.data, C.byref(pos2), n, acc.ctypes.data)
        assert np.array_equal(acc[:n - 1], j[:0:-1]), n      # entry r = partner of position n-1-r
        assert pos1.value == pos2.value and np.array_equal(key1, key2), n
        np.random.set_state(st)
        np.random.permutation(n)
        after = np.random.get_state()
        assert int(after[2]) == pos1.value and np.array_equal(after[1], key1), n


def test_speculative_rng_stream_is_exact_and_cancellable():
    """A stream pre-drawn from a snapshot gives the reference's permutations when the global state still equals the
    snapshot; after a foreign draw the snapshot no longer matches (the learner then drops the stream)."""
    from ppo_exploration_b200.buffer import HostRngStream, rng_states_equal
    np.random.seed(11)
    snap = np.random.get_state()
    spec = HostRngStream([('perm', 5000)] * 4, state=snap, ahead=2)      # runs ahead while "the GPU is busy"
    assert rng_states_equal(np.random.get_state(), snap)                 # global stream untouched
    want = [np.random.permutation(5000) for _ in range(4)]
    for w in want:
        assert np.array_equal(_replay_partners(spec.next()), w)
    assert rng_states_equal(spec.final_state(), np.random.get_state())
    snap2 = np.random.get_state()
    spec2 = HostRngStream([('perm', 5000)] * 4, state=snap2, ahead=2)
    np.random.randn()                                                    # somebody else draws
    assert not rng_states_equal(np.random.get_state(), snap2)
    spec2.cancel()
    spec2.drain()


def test_rng_stream_delivers_exact_partner_lists():
    """Permutations come out as Fisher-Yates partner lists in acceptance order (entry r belongs to position n-1-r) and
    the scalar draws in between stay in sequence; replaying the swaps (here on the CPU -- the GPU kernels of
    shuffle_dev.cu are checked in tests/test_gpu_gather.py) gives numpy's permutations, and the final state is numpy's."""
    import torch
    from ppo_exploration_b200.buffer import HostRngStream, DevicePartners, rng_states_equal
    for n in (1, 2, 17, 1000, 70001):
        np.random.seed(n)
        want = []
        for _ in range(3):
            want.append(np.random.permutation(n))
            want.append(np.random.randn())
        after = np.random.get_state()
        np.random.seed(n)
        s = HostRngStream(sum([[('perm', n), ('randn',)] for _ in range(3)], []))
        for w in want:
            g = s.next()
            if isinstance(w, np.ndarray):
                assert isinstance(g, DevicePartners) and g.j.dtype == torch.int32 and g.j.numel() == n
                assert np.array_equal(_replay_partners(g), w), n
            else:
                assert g == w
        s.drain()
        assert rng_states_equal(s.final_state(), after)


def test_committed_bench_lines_carry_the_contract_keys():
    """The bench line the driver parses (profiles/bench_r02_n1.json is a verbatim `python bench.py` output from the B200
    box, profiles/bench_r02_ref.json the reference arm's): every key of the measurement contract is present and typed."""
    import json
    from conftest import ROOT
    line = json.loads([l for l in open(os.path.join(ROOT, "profiles", "bench_r02_n1.json")) if l.startswith("{")][-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in line, k
    assert line["config"]["workload"].startswith("C2") and "model" not in line["config"]
    assert line["scaling"] == "weak" and line["higher_is_better"] is True and line["vs_baseline"] is None and line["dtype"] == "f32"
    assert line["value"] > 0 and line["gpu_launches"] > 0 and abs(line["ms_per_step"] * line["value"] / 1e3 - 524288) < 1
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["value"] < line["value"] and e2e["h2d_bytes_per_step"] > 5e7 and e2e["d2h_bytes_per_step"] > 0
    rf = line["roofline"]
    assert rf["bound"] in ("hbm", "tensor") and rf["unit"] in ("GB/s", "TFLOP/s") and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert rf["traffic"] is None or rf["traffic"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    assert set(line["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    ref = json.loads([l for l in open(os.path.join(ROOT, "profiles", "bench_r02_ref.json")) if l.startswith("{")][-1])
    assert ref["impl"] == "reference" and ref["metric"] == line["metric"] and ref["unit"] == line["unit"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["value"] == ref["value"]


def test_partner_pool_and_worker_pool_reuse():
    """Host plumbing of the shuffle stream: pinned partner buffers are handed out again only once released (or their
    consumer is gone), and worker threads outlive the streams they serve (no thread start / retire per train() call)."""
    import gc
    import threading
    from ppo_exploration_b200 import buffer as BUF
    pool = BUF._PartnerPool()
    a = pool.take(1000)
    b = pool.take(1000)
    assert a.j.data_ptr() != b.j.data_ptr() and len(pool.slots[1000]) == 2           # both in use: two buffers
    a_ptr = a.j.data_ptr()
    a.release()                                                                     # consumer done with it
    c = pool.take(1000)
    assert c.j.data_ptr() == a_ptr and len(pool.slots[1000]) == 2                    # re-used, pool did not grow
    b_ptr = b.j.data_ptr()
    del b
    gc.collect()                                                                    # a consumer that never released but is gone
    d = pool.take(1000)
    assert d.j.data_ptr() == b_ptr and len(pool.slots[1000]) == 2
    assert pool.take(8).j.numel() == 8                                              # sizes do not mix
    # worker threads: two streams in sequence run on the same pooled threads
    np.random.seed(2)
    before = threading.active_count()
    s1 = BUF.HostRngStream([('perm', 100)] * 3)
    p1 = [_replay_partners(s1.next()) for _ in range(3)]
    s1.drain()
    mid = threading.active_count()
    s2 = BUF.HostRngStream([('perm', 100)] * 3)
    p2 = [_replay_partners(s2.next()) for _ in range(3)]
    s2.drain()
    assert before <= mid <= before + 1                                              # one draw thread per stream, at most
    assert threading.active_count() == mid                                          # no new threads for the second stream
    assert all(np.array_equal(x, y) for x, y in zip(p1, p2))                         # both started from the same global state
    np.random.seed(2)
    assert np.array_equal(p1[0], np.random.permutation(100))


def test_bench_dump_array_caps_size_with_a_fixed_sample():
    """bench.py --dump-outputs: a large array shrinks to the same sorted sample in every call, without a draw from the
    global numpy stream (the learner's shuffles draw from it); small arrays keep their shape; f64 stays f64, the rest
    becomes f32."""
    import torch
    import bench
    np.random.seed(4)
    state = np.random.get_state()
    big = torch.arange(3 * (bench.DUMP_MAX_BYTES // 4) + 7, dtype=torch.float32)
    a, b = bench.dump_array(big), bench.dump_array(big)
    assert a.dtype == np.float32 and a.nbytes == bench.DUMP_MAX_BYTES and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.array_equal(a, big.numpy()[a.astype(np.int64)])
    after = np.random.get_state()
    assert np.array_equal(state[1], after[1]) and state[2] == after[2]
    assert bench.dump_array(np.zeros((40, 8))).dtype == np.float64
    assert bench.dump_array(torch.zeros(5, 3, dtype=torch.uint8)).shape == (5, 3)
    assert bench.dump_array(torch.zeros(bench.DUMP_MAX_BYTES // 4, dtype=torch.float64)).nbytes == bench.DUMP_MAX_BYTES
