"""Shared helpers for the parity tests."""
import glob
import hashlib
import os

import numpy as np

from raytracing_b200 import scene_io

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")

_scene_cache = {}


def scene(name):
    if name not in _scene_cache:
        _scene_cache[name] = scene_io.load_scene(name)
    return _scene_cache[name]


def golden_files():
    return sorted(glob.glob(os.path.join(GOLDEN, "golden_*.npz.xz")))


def load_golden(path):
    g = scene_io.load_npz_xz(path)
    base = os.path.basename(path)[len("golden_"):]
    # file name: golden_<scene>_<w>x<h>_b<mb>[_wf][_<tag>].npz.xz
    stem = base.replace(".npz.xz", "")
    parts = stem.split("_")
    size = max(i for i, p in enumerate(parts) if "x" in p and p.replace("x", "").isdigit())
    g["scene_name"] = "_".join(parts[:size])
    return g


def bits(a):
    """Bit pattern of a float32 array for exact comparisons.  NaNs are canonicalised first: the payload/sign of a NaN
    produced by an invalid operation is not specified by IEEE 754 (x86 gives 0xFFC00000, sm_100a 0x7FFFFFFF)."""
    u = np.ascontiguousarray(a, dtype="<f4").copy().view("<u4")
    u[(u & 0x7FFFFFFF) > 0x7F800000] = 0x7FC00000
    return u


def digest(*arrays):
    """SHA-256 (first 128 bits, in hex) over arrays: float arrays as their bit patterns (see bits), others as stored.  Stands in for a stored
    output in the bit-exact comparisons with the reference (tests/golden/ref)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.asarray(a)
        h.update(bits(a).tobytes() if a.dtype.kind == "f" else np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:32]


def synthetic_sampler_tables(seed=20260923):
    """Seeded stand-ins for the blue-noise sampler's tables (same shapes and value ranges as the reference's
    utils/blue_noise_sampler.hpp, which is reference data and not committed here): any tables exercise the same lookups."""
    rng = np.random.default_rng(seed)
    return (rng.integers(0, 256, 65536, dtype=np.int32), rng.integers(0, 256, 131072, dtype=np.int32),
            rng.integers(0, 256, 131072, dtype=np.int32))


def fuzz_configs(n=12, seed=77):
    """Seeded random frame configurations (scene, size, bounces, camera pose / lens, white furnace) shared by the
    oracle-vs-reference fuzz on the CPU and the CUDA-vs-oracle fuzz on the GPU."""
    rng = np.random.default_rng(seed)
    names = ["CornellBox", "ShaderBalls", "CornellBox_Dragon"]
    out = []
    for i in range(n):
        name = names[i % 3]
        w, h = int(rng.integers(33, 97)), int(rng.integers(17, 65))
        mb = int(rng.integers(0, 7))
        pos = (float(rng.uniform(-0.8, 0.8)), float(rng.uniform(-1.8, -0.2)), float(rng.uniform(0.2, 1.8)))
        kw = {"position": pos, "yaw": float(rng.uniform(0.9, 2.2)), "pitch": float(rng.uniform(1.0, 2.1))}
        if rng.random() < 0.4:
            kw.update(aperture=float(rng.uniform(0.0, 0.1)), focus_distance=float(rng.uniform(0.5, 4.0)))
        out.append((name, w, h, mb, kw, bool(rng.random() < 0.2)))
    # axis-aligned views: rays with exactly-zero direction components (inv_dir = +-inf in the slab test)
    out.append(("CornellBox", 65, 33, 3, {"position": (0.0, -1.0, 1.0), "yaw": 1.5707963267948966, "pitch": 1.5707963267948966}, False))
    out.append(("ShaderBalls", 64, 48, 4, {"position": (0.0, 0.0, 3.0), "yaw": 0.0, "pitch": 3.14159265}, False))
    return out
