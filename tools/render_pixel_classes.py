#!/usr/bin/env python
"""Pixel-class census of the render kernel's gather, counted on the host debug build (the same
env_setup_frame / compose_rows the device runs, as loops): after a rollout that desynchronises the envs,
the share of frame pixels that take each path of the gather.

  tile opaque     one tile cell, opaque texel (no background fetch)
  tile under      one tile cell whose texel is not opaque, or an empty cell: the background is fetched
  strip           overlap strip pixel: two cell columns and / or rows cover it (2 or 4 candidate cells)
  general solid   one cell that is a solid-colour general blit (CELL_GENERAL)
  general other   one cell that is another general blit (clipped walk, adjusted rect, no tile room)
  no cell         no cell column or row covers it: background only
  painted         (overlapping the classes above) inside the box of an entity or overlay blit

usage: python tools/render_pixel_classes.py [--envs 64] [--steps 300] [--json OUT] [case ...]
       case = game[:mode][:whole]   (whole = center_agent=False); default: coinrun easy and a few grid games
Needs no GPU."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

CLASSES = ["tile opaque", "tile under", "strip", "general solid", "general other", "no cell"]
PAINTED = 0x80
DEFAULT_CASES = ["coinrun:easy", "coinrun:easy:whole", "maze:hard", "heist:hard", "climber:hard", "chaser:hard", "ninja:hard"]


def census(lib_path, game, mode, whole, envs, steps, seed=0):
    """Pixel-class shares (fractions of all frame pixels) over `envs` envs after `steps` random steps."""
    from oracle.ref_env import RefVecEnv, default_pack, mt19937_actions

    kw = dict(center_agent=False) if whole else {}
    env = RefVecEnv(envs, game, distribution_mode=mode, num_levels=0, start_level=0, rand_seed=seed, lib_path=lib_path,
                    resource_root=default_pack(), **kw)
    try:
        acts = mt19937_actions(seed, envs, steps)
        for t in range(steps):
            env.act(acts[t])
        lib = env.lib
        lib.pgb200_debug_pixel_classes.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        lib.pgb200_debug_pixel_classes.restype = C.c_int
        buf = np.zeros((envs, 64 * 64), np.uint8)
        for e in range(envs):
            rc = lib.pgb200_debug_pixel_classes(C.c_void_p(env.h), e, buf[e].ctypes.data_as(C.c_void_p))
            if rc != 0:
                raise RuntimeError("pgb200_debug_pixel_classes failed: the census needs the host debug build")
    finally:
        env.close()
    cls = buf & 0x7F
    out = {name: float((cls == i).mean()) for i, name in enumerate(CLASSES)}
    out["painted"] = float(((buf & PAINTED) != 0).mean())
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("cases", nargs="*", default=DEFAULT_CASES)
    ap.add_argument("--envs", type=int, default=64)
    ap.add_argument("--steps", type=int, default=300, help="random steps before the census (desynchronises the envs)")
    ap.add_argument("--json", help="also write the table as JSON lines here")
    args = ap.parse_args(argv)
    from procgen_b200 import build as B

    lib_path = B.build_hostsim()
    rows = []
    print(f"{'case':26s} " + " ".join(f"{c:>13s}" for c in CLASSES + ["painted"]))
    for case in args.cases:
        parts = case.split(":")
        game, mode = parts[0], parts[1] if len(parts) > 1 else "hard"
        whole = len(parts) > 2 and parts[2] == "whole"
        r = census(lib_path, game, mode, whole, args.envs, args.steps)
        rows.append(dict(game=game, mode=mode, center_agent=not whole, envs=args.envs, steps=args.steps, shares=r))
        label = f"{game} {mode}" + (" whole" if whole else "")
        print(f"{label:26s} " + " ".join(f"{100 * r[c]:12.2f}%" for c in CLASSES + ["painted"]), flush=True)
    if args.json:
        with open(args.json, "w") as fh:
            for row in rows:
                fh.write(json.dumps(row) + "\n")
    return rows


if __name__ == "__main__":
    main()
