"""Pins the oracle (reference sources compiled in place + raster restatement) before it is trusted:
known-answer values recorded from the unmodified reference logic (SURVEY §8c) and the committed
golden fixtures in tests/golden/."""
import hashlib
import os

import numpy as np
import pytest

from oracle.ref_env import RefVecEnv, mt19937_actions

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_mt19937_known_answers():
    # std::mt19937 seed 0 -> 2357136044, 2546248239, 3071714933 (SURVEY §8c)
    rs = np.random.RandomState(0)
    assert list(rs.randint(0, 2 ** 32, size=3, dtype=np.uint32)) == [2357136044, 2546248239, 3071714933]


def test_initial_level_seeds(ref_lib, asset_pack):
    env = RefVecEnv(8, "coinrun", distribution_mode="easy", num_levels=200, start_level=0, rand_seed=0)
    rew, ob, first = env.observe()
    assert list(env.info["level_seed"]) == [71, 106, 137, 26, 171, 23, 156, 72]
    assert first.all() and (rew == 0).all()
    env.close()


@pytest.mark.parametrize("name,mode,n,steps,expect", [
    ("coinrun", "easy", 64, 1000, (360.0, 95, 36)),
    ("coinrun", "hard", 4, 500, (0.0, 1, 0)),
    ("bigfish", "hard", 64, 1000, (128.0, 525, 0)),
    ("maze", "hard", 64, 1000, (600.0, 143, 60)),
    ("heist", "hard", 64, 1000, (120.0, 66, 12)),
    # the other twelve games, N=32, T=1500 (SURVEY §8c "further KATs")
    ("bossfight", "hard", 32, 1500, (50.0, 1117, 4)),
    ("caveflyer", "hard", 32, 1500, (100.0, 113, 10)),
    ("chaser", "hard", 32, 1500, (286.96, 442, 0)),
    ("climber", "hard", 32, 1500, (131.0, 91, 10)),
    ("dodgeball", "hard", 32, 1500, (284.0, 435, 0)),
    ("fruitbot", "hard", 32, 1500, (-752.0, 1280, 0)),
    ("jumper", "hard", 32, 1500, (140.0, 97, 14)),
    ("leaper", "hard", 32, 1500, (280.0, 297, 28)),
    ("miner", "hard", 32, 1500, (164.0, 137, 0)),
    ("ninja", "hard", 32, 1500, (220.0, 187, 22)),
    ("plunder", "hard", 32, 1500, (334.0, 115, 0)),
    ("starpilot", "hard", 32, 1500, (505.0, 568, 0)),
])
def test_aggregate_known_answers(ref_lib, asset_pack, name, mode, n, steps, expect):
    """(sum reward, episode starts, level completes) under the §8c action recipe."""
    env = RefVecEnv(n, name, distribution_mode=mode, num_levels=200, start_level=0, rand_seed=0)
    acts = mt19937_actions(0, n, steps)
    tot, starts, comp = 0.0, 0, 0
    env.observe()
    for t in range(steps):
        env.act(acts[t])
        rew, ob, first = env.observe()
        tot += float(rew.sum())
        starts += int(first.sum())
        comp += int(env.info["prev_level_complete"].sum())
    env.close()
    assert (round(tot, 2), starts, comp) == expect


@pytest.mark.parametrize("fixture", sorted(f for f in os.listdir(GOLDEN) if f.endswith(".npz")) if os.path.isdir(GOLDEN) else [])
def test_oracle_reproduces_golden(ref_lib, asset_pack, fixture):
    g = np.load(os.path.join(GOLDEN, fixture), allow_pickle=False)
    kw = dict(distribution_mode=str(g["mode"]), num_levels=int(g["num_levels"]), start_level=0, rand_seed=int(g["rand_seed"]))
    env = RefVecEnv(int(g["num"]), str(g["env_name"]), **kw)
    acts = g["actions"]
    env.observe()
    for t in range(acts.shape[0]):
        env.act(acts[t])
        rew, ob, first = env.observe()
        assert np.array_equal(rew, g["rew"][t])
        assert np.array_equal(first, g["first"][t])
        assert np.array_equal(env.info["level_seed"], g["level_seed"][t])
        assert hashlib.sha256(ob["rgb"].tobytes()).hexdigest() == str(g["rgb_sha256"][t])
    assert np.array_equal(ob["rgb"], g["last_rgb"])
    env.close()


# The raster restatement against a REAL Qt raster engine (Qt 6.6.3, whose libraries ship with Nsight
# Compute): tests/golden/qt6/make_qt6_golden.py drew every case below with oracle/_ref/libenv_ref_qt6.so
# and stored what Qt drew, so these comparisons need no Qt installation. Frames are stored as one
# 64-bit digest per step plus the pixels in which Qt differed from the restatement when recorded.
QT6_GOLDEN = os.path.join(GOLDEN, "qt6", "qt6_raster.npz")
QT6_FRAME_CASES = {}
for _name, _mode in [("coinrun", "hard"), ("bigfish", "hard"), ("maze", "hard"), ("jumper", "easy"), ("jumper", "hard"),
                     ("fruitbot", "hard"), ("starpilot", "hard")]:
    QT6_FRAME_CASES[f"raster_{_name}_{_mode}"] = (_name, _mode, 8, 150, 0, dict(rand_seed=3))
for _name, _mode in [("jumper", "easy"), ("jumper", "hard"), ("jumper", "memory"), ("coinrun", "hard"), ("caveflyer", "hard"),
                     ("climber", "hard"), ("ninja", "easy")]:
    QT6_FRAME_CASES[f"world_{_name}_{_mode}"] = (_name, _mode, 4, 120, 2, dict(rand_seed=5, center_agent=False))
QT6_FRAME_CASES["rotated_heist_hard"] = ("heist", "hard", 8, 200, 0, dict(rand_seed=3))


def digest64(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest()[:8], np.uint64)[0]


def qt6_case_frames(key, lib_path=None):
    """The rgb batch after every step of one QT6_FRAME_CASES entry, drawn by the oracle at lib_path."""
    name, mode, n, steps, act_seed, kw = QT6_FRAME_CASES[key]
    env = RefVecEnv(n, name, distribution_mode=mode, num_levels=0, lib_path=lib_path, **kw)
    acts = mt19937_actions(act_seed, n, steps)
    for t in range(steps):
        env.act(acts[t])
        yield env.observe()[1]["rgb"]
    env.close()


def _pixels_differing_from_qt6(key):
    """(differing pixels, all pixels) of the restatement against the recorded Qt 6.6.3 frames."""
    g = np.load(QT6_GOLDEN, allow_pickle=False)
    digests, patch = g[key + "_digest"], g[key + "_patch"]
    bad = tot = 0
    for t, rgb in enumerate(qt6_case_frames(key)):
        rows = patch[patch[:, 0] == t]
        qt = rgb.copy()
        qt[rows[:, 1], rows[:, 2], rows[:, 3]] = rows[:, 4:]
        assert digest64(qt) == digests[t], f"{key} step {t}: restatement differs from Qt 6.6.3 beyond the recorded pixels"
        d = (rgb != qt).any(-1)
        bad += int(d.sum())
        tot += d.size
    return bad, tot


def test_raster_restatement_matches_real_qt6(ref_lib, asset_pack):
    """Zero differing pixels from Qt 6.6.3 for the un-rotated draw paths (scaled blits, tiling, fillRect)
    and for jumper's compass (drawEllipse, drawLine)."""
    for key in QT6_FRAME_CASES:
        if key.startswith("raster_"):
            bad, tot = _pixels_differing_from_qt6(key)
            assert bad == 0, f"{key}: {bad} of {tot} pixels differ from Qt 6.6.3"


def test_whole_world_view_restatement_matches_real_qt6(ref_lib, asset_pack):
    """center_agent=False (basic-abstract-game.cpp:819-838): cells of 1 to 3.2 px, and jumper's compass disc on
    the two further non-integer rects whose rows were captured from Qt 6.6.3 — restatement == real Qt 6."""
    for key in QT6_FRAME_CASES:
        if key.startswith("world_"):
            bad, tot = _pixels_differing_from_qt6(key)
            # caveflyer's ship rotates: the coverage budget of test_rotated_raster_restatement_close_to_real_qt6 applies
            assert bad <= (1e-5 * tot if "caveflyer" in key else 0), f"{key}: {bad} of {tot} pixels differ from Qt 6.6.3"


def test_rotated_raster_restatement_close_to_real_qt6(ref_lib, asset_pack):
    """Rotated sprites (heist): the restatement follows Qt's two transformed-image paths. Texels are
    exact; coverage of small quads differs from Qt 6.6.3 only at exact 45-degree headings (26.6
    scan-converter ties). Budget: <= 1e-5 of all pixels (measured 3e-6)."""
    bad, tot = _pixels_differing_from_qt6("rotated_heist_hard")
    assert bad <= 1e-5 * tot, f"{bad} of {tot} pixels differ from Qt 6.6.3"


def ellipse_and_line_draws(lib):
    """drawEllipse (midpoint algorithm on integer rects, pen / no pen / translucent brush, clipped by
    the device edge) and drawLine(int...) with a cosmetic pen, through the shim's test hooks of lib:
    yields (case, image) in a fixed order."""
    import ctypes as C

    bg = 0xff102030

    def ell(x, y, w, h, col, pw):
        dst = np.full((64, 64), bg, np.uint32)
        lib.shim_test_draw_ellipse(dst.ctypes.data_as(C.c_void_p), 64, 64, C.c_double(x), C.c_double(y), C.c_double(w), C.c_double(h), *col, pw)
        return dst

    def line(x1, y1, x2, y2, pw):
        dst = np.full((64, 64), bg, np.uint32)
        lib.shim_test_draw_line(dst.ctypes.data_as(C.c_void_p), 64, 64, x1, y1, x2, y2, 252, 186, 3, pw)
        return dst

    for x in range(-3, 60, 9):
        for y in range(-3, 60, 11):
            for w in range(1, 20, 2):
                for h in (1, 2, 3, 8, 16, w):
                    for col, pw in (((168, 166, 158, 255), 1), ((255, 255, 255, 120), -1), ((252, 186, 3, 255), 0)):
                        yield ("ellipse", x, y, w, h, col, pw), ell(x, y, w, h, col, pw)
    # jumper's four compass discs (jumper.cpp:138-141): all but hard mode's centred one sit on non-integer rects
    unit = np.float32(64) / np.float32(12)
    easy = (float(np.float32(8.75) * unit), float(np.float32(.25) * unit), float(np.float32(3) * unit))
    world_easy = (53.60000228881836, 0.800000011920929, 9.600000381469727)   # center_agent=False, tests/tools/qt6_compass_mask.py
    world_hard = (60.400001525878906, 0.4000000059604645, 3.200000047683716)
    for rect in ((easy[0], easy[1], easy[2], easy[2]), (55.0, 1.0, 8.0, 8.0), world_easy + world_easy[2:], world_hard + world_hard[2:]):
        yield ("compass", rect), ell(*rect, (168, 166, 158, 255), 1)
    # every needle the compass can draw and more: all integer offsets within 9 px of in-bounds centres
    for cx, cy in ((54, 9), (59, 5), (20, 40), (10, 10)):
        for dx in range(-9, 10):
            for dy in range(-9, 10):
                if not (0 <= cx + dx < 64 and 0 <= cy + dy < 64):
                    continue
                for pw in (0, 1):
                    yield ("line", cx, cy, dx, dy, pw), line(cx, cy, cx + dx, cy + dy, pw)


def scaled_blit_and_fill_draws(lib):
    """Rules S and F on random rects, with positions and sizes deliberately placed on exact halves
    and quarters (qRound ties; Qt 6 rounds negative ties away from zero): yields (case, image)."""
    import ctypes as C

    rng = np.random.RandomState(7)
    srcs = [(np.arange(sw * sh, dtype=np.uint32).reshape(sh, sw)) | 0xff000000 for sw, sh in ((8, 8), (64, 64), (17, 17), (480, 270), (128, 64))]

    def draw(src, x, y, w, h):
        sh, sw = src.shape
        dst = np.zeros((64, 64), np.uint32)
        lib.shim_test_draw_image(dst.ctypes.data_as(C.c_void_p), 64, 64, src.ctypes.data_as(C.c_void_p), sw, sh, 0, C.c_double(x), C.c_double(y),
                                 C.c_double(w), C.c_double(h), C.c_double(0), C.c_double(1.0), 0)
        return dst

    def fill(x, y, w, h):
        dst = np.zeros((64, 64), np.uint32)
        lib.shim_test_fill_rect(dst.ctypes.data_as(C.c_void_p), 64, 64, C.c_double(x), C.c_double(y), C.c_double(w), C.c_double(h), 200, 100, 50)
        return dst

    def rnd():
        k = rng.randint(4)
        if k == 0:
            return float(rng.randint(-40, 100)) / 2
        if k == 1:
            return float(rng.randint(-80, 200)) / 4
        return rng.uniform(-20, 70)

    for _ in range(1500):
        x, y = rnd(), rnd()
        w = abs(rnd()) + 0.1 if rng.randint(2) else float(rng.randint(1, 80)) / 2
        h = abs(rnd()) + 0.1 if rng.randint(2) else float(rng.randint(1, 80)) / 2
        if rng.randint(3) == 0:
            w *= 4
            h *= 4
        src = srcs[rng.randint(len(srcs))]
        if w == src.shape[1] and h == src.shape[0]:
            continue  # 1:1 draws take Qt's unscaled path, which no in-scope draw call reaches
        yield ("blit", x, y, w, h, src.shape), draw(src, x, y, w, h)
        yield ("fill", x, y, w, h), fill(x, y, w, h)


def _assert_draws_match_qt6(key, draws):
    import ctypes as C

    from oracle.ref_env import REF_LIB

    expect = np.load(QT6_GOLDEN, allow_pickle=False)[key + "_digest"]
    got = [(case, digest64(img)) for case, img in draws(C.CDLL(REF_LIB))]
    assert len(got) == len(expect), f"{key}: {len(got)} draws, {len(expect)} recorded"
    for (case, d), e in zip(got, expect):
        assert d == e, f"{key}: {case} differs from Qt 6.6.3"


def test_ellipse_and_line_restatement_match_real_qt6(ref_lib, asset_pack):
    """Every ellipse and line case of ellipse_and_line_draws identical to Qt 6.6.3."""
    _assert_draws_match_qt6("ellipse_line", ellipse_and_line_draws)


def test_scaled_blit_and_fill_sweep_match_real_qt6(ref_lib, asset_pack):
    """Every blit and fill of scaled_blit_and_fill_draws identical to Qt 6.6.3."""
    _assert_draws_match_qt6("blit_fill", scaled_blit_and_fill_draws)
