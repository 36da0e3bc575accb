"""The render kernel's gather on the views where its rare paths are common, run in the host debug build
with the device's row ownership and checked in lockstep against the oracle: the whole-world views of the
scrolling games (center_agent=False: cells of 1-3 pixels, one-pixel overlap strips of two cell columns or
rows everywhere), and solid-colour general cells (chaser's orbs, monochrome assets). Plus the pixel-class
census of tools/render_pixel_classes.py, which reads the same frame records."""
import os
import sys

import pytest

from helpers import make_pair, run_lockstep

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name,mode,seed", [("coinrun", "easy", 7), ("coinrun", "hard", 3), ("ninja", "hard", 5),
                                            ("climber", "easy", 11), ("caveflyer", "hard", 2)])
def test_whole_world_strips_bit_exact(ref_lib, hostsim_lib, name, mode, seed):
    ref, dut = make_pair(hostsim_lib, 8, name, distribution_mode=mode, num_levels=0, start_level=0, rand_seed=seed,
                         center_agent=False)
    run_lockstep(ref, dut, 150, seed=seed)
    ref.close()
    dut.close()


@pytest.mark.parametrize("name,extra", [("chaser", {}), ("maze", dict(use_monochrome_assets=True)),
                                        ("coinrun", dict(use_monochrome_assets=True, center_agent=False))])
def test_general_cells_bit_exact(ref_lib, hostsim_lib, name, extra):
    ref, dut = make_pair(hostsim_lib, 8, name, distribution_mode="hard", num_levels=0, start_level=0, rand_seed=4, **extra)
    run_lockstep(ref, dut, 150, seed=4)
    ref.close()
    dut.close()


def test_pixel_class_census(hostsim_lib):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import render_pixel_classes as rpc
    finally:
        sys.path.pop(0)
    classes = rpc.CLASSES
    centred = rpc.census(hostsim_lib, "coinrun", "easy", False, envs=4, steps=20)
    assert abs(sum(centred[c] for c in classes) - 1.0) < 1e-9
    assert centred["strip"] > 0.01, centred  # cells of 4.9 pixels: one-pixel overlaps every few columns / rows
    assert centred["tile opaque"] + centred["tile under"] > 0.5, centred
    assert 0 < centred["painted"] < 1
    mono = rpc.census(hostsim_lib, "maze", "hard", False, envs=4, steps=20)
    assert abs(sum(mono[c] for c in classes) - 1.0) < 1e-9
