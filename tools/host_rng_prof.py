"""Diagnostic: rate of the host-side numpy-replay draws on this box -- the bare C call, and through HostRngStream
(thread hand-offs, pinned allocations, numpy state round trips included)."""
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from ppo_exploration_b200 import _lib as L
from ppo_exploration_b200.buffer import HostRngStream

torch.cuda.init()
for n in (524288, 1 << 20, 1 << 21, 1 << 22):
    np.random.seed(1)
    st = np.random.get_state()
    key, pos = np.ascontiguousarray(st[1], dtype=np.uint32).copy(), C.c_int(int(st[2]))
    acc = torch.empty(n, dtype=torch.int32, pin_memory=True)
    best = 1e9
    for _ in range(5):
        t0 = time.perf_counter()
        L.call("ppx_np_shuffle_draws32_stream", key.ctypes.data, C.byref(pos), n, acc.data_ptr())
        best = min(best, time.perf_counter() - t0)
    line = f"n={n}: bare draws {best * 1e3:.3f} ms = {best / n * 1e9:.3f} ns/draw"
    for rep in range(3):
        s = HostRngStream([('perm', n)] * 10)
        t0 = time.perf_counter()
        for _ in range(10):
            s.next().release()                          # as the learner does once the H2D copy is queued
        dt = time.perf_counter() - t0
        s.drain()
    line += f" | HostRngStream 10 perms {dt * 1e3:.3f} ms = {dt / (10 * n) * 1e9:.3f} ns/draw"
    print(line)
