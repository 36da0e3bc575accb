"""Asset pack: the reference's PNG sprites/backgrounds decoded once into a single binary file.

The reference decodes 779 sprite PNGs to ARGB32_Premultiplied and 6 background groups to RGB32 at
process start (resources.cpp:19-28, 813-815, 943-953) from ``procgen/data/assets``.  The package
never reads the reference tree: ``build_pack`` decodes every PNG with PIL to straight RGBA8 —
which equals Qt's ``QImage(path)`` decode for the 8-bit RGBA / palette+tRNS / RGB files the
reference ships (SURVEY §8a) — and writes one zlib-compressed record per image.  Those decoded
images are stored in the repository as data, in tests/golden/assets/ (``export_images``: the
images' RGBA8 bytes in pack order, xz-compressed and cut into parts of under 1 MB, plus their
names, sizes and groups), and ``__graft_entry__.build()`` assembles the pack from there
(``build_pack_from_images``), so that a checkout needs nothing outside it.  The pack itself is a
built artefact (git-ignored).

File layout (little endian):
  header   : magic "PGB2PACK", u32 version, u32 count, u64 manifest_off, u64 manifest_len
  entries  : count x { char name[112]; u32 w; u32 h; u64 off; u32 csize; u32 reserved }
  payloads : zlib(RGBA8 straight alpha, row-major, w*h*4 bytes)
  manifest : JSON {"groups": {group: [relpath, ...]}, "sprites": [relpath, ...]}

Group membership and order matter: ``background_index = randn(len(group))``
(basic-abstract-game.cpp:767) indexes these lists, and ``platform_backgrounds`` gets every
space background appended (resources.cpp:949-953).
"""
from __future__ import annotations

import json
import os
import re
import struct
import zlib

import numpy as np

MAGIC = b"PGB2PACK"
VERSION = 1
_HDR = struct.Struct("<8sIIQQ")
_ENT = struct.Struct("<112sIIQII")

DEFAULT_PACK = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "assets.pack")
REFERENCE_ROOT = "/root/reference/procgen"
IMAGES_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "assets")
_PART_BYTES = 1000 * 1000


def _parse_resource_lists(resources_cpp: str):
    """Pull the sprite list and background groups out of resources.cpp (names only)."""
    text = open(resources_cpp).read()
    start = text.index("auto sprite_paths")
    end = text.index("for (const auto& sprite_path")
    sprites = re.findall(r'"([^"]+\.png)"', text[start:end])
    gstart = text.index("auto group_to_paths")
    gend = text.index("for (auto const &pair")
    body = text[gstart:gend]
    groups = {}
    for m in re.finditer(r'"(\w+_backgrounds)",\s*\{(.*?)\},\s*\}', body, re.S):
        groups[m.group(1)] = re.findall(r'"([^"]+\.png)"', m.group(2))
    # resources.cpp:949-953: space backgrounds double as platform backgrounds
    groups["platform_backgrounds"] = groups["platform_backgrounds"] + groups["space_backgrounds"]
    return sprites, groups


def build_pack(out_path: str = DEFAULT_PACK, reference_root: str = REFERENCE_ROOT, verbose: bool = False) -> str:
    """Decodes the reference's PNGs into a pack (only where the reference tree is present)."""
    from PIL import Image

    assets_dir = os.path.join(reference_root, "data", "assets")
    sprites, groups = _parse_resource_lists(os.path.join(reference_root, "src", "resources.cpp"))
    names = list(dict.fromkeys(sprites + [p for g in groups.values() for p in g]))
    images = []
    for i, name in enumerate(names):
        images.append((name, np.asarray(Image.open(os.path.join(assets_dir, name)).convert("RGBA"), dtype=np.uint8)))
        if verbose and i % 100 == 0:
            print(f"[assets] {i}/{len(names)} {name}")
    return _write_pack(out_path, images, {"groups": groups, "sprites": sprites})


def _write_pack(out_path, images, manifest):
    entries = []
    payloads = []
    off = _HDR.size + _ENT.size * len(images)
    for name, arr in images:
        h, w = arr.shape[:2]
        comp = zlib.compress(arr.tobytes(), 6)
        entries.append((name.encode(), w, h, off, len(comp), 0))
        payloads.append(comp)
        off += len(comp)
    manifest = json.dumps(manifest).encode()
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    tmp = out_path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(_HDR.pack(MAGIC, VERSION, len(images), off, len(manifest)))
        for e in entries:
            f.write(_ENT.pack(*e))
        for p in payloads:
            f.write(p)
        f.write(manifest)
    os.replace(tmp, out_path)
    return out_path


def export_images(pack_path: str = DEFAULT_PACK, out_dir: str = IMAGES_DIR) -> None:
    """Stores the decoded images of a pack in out_dir: index.json and images.xz.NN."""
    import hashlib
    import lzma

    pack = AssetPack(pack_path)
    names = list(pack.index)
    raw = b"".join(pack.rgba(n).tobytes() for n in names)
    data = lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME)
    os.makedirs(out_dir, exist_ok=True)
    for f in os.listdir(out_dir):
        os.remove(os.path.join(out_dir, f))
    for i in range(0, len(data), _PART_BYTES):
        with open(os.path.join(out_dir, f"images.xz.{i // _PART_BYTES:02d}"), "wb") as f:
            f.write(data[i:i + _PART_BYTES])
    index = {"images": [[n, *pack.size(n)] for n in names], "manifest": pack.manifest,
             "sha256": hashlib.sha256(raw).hexdigest()}
    with open(os.path.join(out_dir, "index.json"), "w") as f:
        json.dump(index, f)


def build_pack_from_images(out_path: str = DEFAULT_PACK, images_dir: str = IMAGES_DIR) -> str:
    """The pack, from the images stored in the repository (see export_images)."""
    import hashlib
    import lzma

    with open(os.path.join(images_dir, "index.json")) as f:
        index = json.load(f)
    parts = sorted(p for p in os.listdir(images_dir) if p.startswith("images.xz."))
    raw = lzma.decompress(b"".join(open(os.path.join(images_dir, p), "rb").read() for p in parts))
    if hashlib.sha256(raw).hexdigest() != index["sha256"]:
        raise RuntimeError(f"{images_dir}: stored images are damaged (sha256 mismatch)")
    images = []
    off = 0
    for name, w, h in index["images"]:
        images.append((name, np.frombuffer(raw, np.uint8, w * h * 4, off).reshape(h, w, 4)))
        off += w * h * 4
    return _write_pack(out_path, images, index["manifest"])


class AssetPack:
    """Random-access reader (decompresses lazily, caches)."""

    def __init__(self, path: str = DEFAULT_PACK):
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"asset pack {path} missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        self.path = path
        with open(path, "rb") as f:
            magic, ver, count, moff, mlen = _HDR.unpack(f.read(_HDR.size))
            if magic != MAGIC or ver != VERSION:
                raise ValueError("bad asset pack header")
            self.index = {}
            for _ in range(count):
                name, w, h, off, csize, _r = _ENT.unpack(f.read(_ENT.size))
                self.index[name.rstrip(b"\0").decode()] = (w, h, off, csize)
            f.seek(moff)
            self.manifest = json.loads(f.read(mlen))
        self.groups = self.manifest["groups"]
        self._cache = {}

    def size(self, name):
        w, h, _, _ = self.index[name]
        return w, h

    def rgba(self, name) -> np.ndarray:
        """Straight-alpha RGBA8 array [h, w, 4]."""
        if name not in self._cache:
            w, h, off, csize = self.index[name]
            with open(self.path, "rb") as f:
                f.seek(off)
                raw = zlib.decompress(f.read(csize))
            self._cache[name] = np.frombuffer(raw, dtype=np.uint8).reshape(h, w, 4)
        return self._cache[name]


def byte_mul(c: np.ndarray, a: np.ndarray) -> np.ndarray:
    """Qt's BYTE_MUL per 8-bit channel: (c*a + ((c*a)>>8) + 0x80) >> 8."""
    t = c.astype(np.uint32) * a.astype(np.uint32)
    return ((t + (t >> 8) + 0x80) >> 8).astype(np.uint32)


def to_argb32_premultiplied(rgba: np.ndarray) -> np.ndarray:
    """u32 [h, w] 0xAARRGGBB premultiplied == QImage::convertToFormat(Format_ARGB32_Premultiplied)
    (resources.cpp:21, 814)."""
    r, g, b, a = (rgba[..., i] for i in range(4))
    return ((a.astype(np.uint32) << 24) | (byte_mul(r, a) << 16) | (byte_mul(g, a) << 8) | byte_mul(b, a)).astype(np.uint32)


def to_rgb32(rgba: np.ndarray) -> np.ndarray:
    """u32 [h, w] 0xFFRRGGBB == convertToFormat(Format_RGB32): colour kept, alpha forced to 255
    (resources.cpp:946)."""
    r, g, b = (rgba[..., i].astype(np.uint32) for i in range(3))
    return (np.uint32(0xFF000000) | (r << 16) | (g << 8) | b).astype(np.uint32)
