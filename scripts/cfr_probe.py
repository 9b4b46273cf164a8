"""CFR kernel time (zero net: the iteration is the CFR kernel alone) for root waves and for self-play waves."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import rebel_b200 as rb

D, F, K = 1, 6, 8192
H = F ** D
b = np.random.RandomState(1).rand(K, 2, H); b /= b.sum(-1, keepdims=True)
S = rb.WaveSolver(D, F, K, net_mode=rb.NET_ZERO)
S.begin(np.full(K, -1, np.int32), np.zeros(K, np.int32), b)
for _ in range(3):
    S.reset(); S.run(256); S.sync()
tot, _ = S.last_run_ms()
print("root wave: CFR us per iteration", tot / 256 * 1e3, flush=True)
S.selfplay_create(np.arange(K, dtype=np.uint32) * 1000000 + 7)
for _ in range(8):
    S.selfplay_wave()
S.sync()
S.selfplay_wave(); S.sync()
tot, _ = S.last_run_ms()
print("self-play wave: CFR us per iteration", tot / 1024 * 1e3, "rows", S.leaf_rows, flush=True)
