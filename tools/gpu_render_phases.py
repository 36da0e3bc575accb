"""Render-kernel phase cycles (profiling variant libprocgen_b200_phase.so, -DPG_PHASE_TIMING).
usage: PROCGEN_B200_LIB=.../libprocgen_b200_phase.so python tools/gpu_render_phases.py game mode envs desync"""
import ctypes as C
import os
import struct
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from procgen_b200 import ProcgenGym3Env

game, mode, n, desync = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4])
env = ProcgenGym3Env(n, game, distribution_mode=mode, num_levels=0, rand_seed=0)
off = env._lib.pgb200_debug_phase_offset()
assert off >= 0, "needs the PG_PHASE_TIMING build"
g = torch.Generator(device="cuda").manual_seed(0)
acts = torch.randint(0, 15, (64, n), device="cuda", dtype=torch.int32, generator=g)
for t in range(desync):
    env.act(acts[t % 64])
env.observe()
torch.cuda.synchronize()
buf = (C.c_ubyte * 1024)()
acc = []
for e in range(0, n, max(1, n // 512)):
    env._lib.pgb200_debug_read_env(env._h, int(e), buf, None, 0)
    acc.append(struct.unpack_from("<12I", bytes(buf), off))
a = np.array(acc, dtype=np.float64)
# render_kernel's phase counters (thread 0 of the CTA; ids 1-4 belong to the logic kernel's reset phases):
# 0 stage (bulk copies of the frame record and tiles), 5 compose, 6 consumer + pack, 7 store; compose split
# as warp 0 (row owner 0) sees it: 8 gather (cells over background), 9 paint (entity + overlay blits)
phases = [(0, "stage"), (5, "compose"), (8, "  gather (warp 0)"), (9, "  paint (warp 0)"), (6, "consumer+pack"), (7, "store")]
tot = a[:, [0, 5, 6, 7]].sum(1).mean()
print(f"{game} {mode}: mean cycles per frame {tot:.0f}")
for i, nm in phases:
    print(f"  {nm:22s} mean {a[:, i].mean():8.0f}  p90 {np.percentile(a[:, i], 90):8.0f}  {100 * a[:, i].mean() / tot:5.1f}%")
env.close()
