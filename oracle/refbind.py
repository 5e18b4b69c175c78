"""
oracle/refbind.py — TEST INFRASTRUCTURE.  ctypes binding of oracle/_ref/libref.so
(the reference's own kernels + host code compiled for the CPU, see build_ref.py).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")

import sys
sys.path.insert(0, os.path.dirname(HERE))
from raytracing_b200.layouts import (CAMERA_DT, HIT_DT, LIGHT_DT, MATERIAL_DT, NODE_DT, RAY_DT, SCENE_ARRAYS,  # noqa: E402,F401
                                     SCENE_INFO_DT, TEXTURE_DT, TRIANGLE_DT)


def available(libm: bool = False) -> bool:
    return os.path.exists(os.path.join(REF_DIR, "libref_libm.so" if libm else "libref.so"))


from raytracing_b200.camera import default_camera  # noqa: E402,F401

def set_sampler_tables(tables, libm: bool = False):
    """Process-wide: the blue-noise kernels of libref[_libm].so read copies of these (sobol, scrambling, ranking) tables of the
    reference's sizes from now on; None restores the tables the reference compiled in."""
    L = C.CDLL(os.path.join(REF_DIR, "libref_libm.so" if libm else "libref.so"))
    L.ref_set_sampler_tables.argtypes = [C.c_void_p] * 3
    if tables is None:
        L.ref_set_sampler_tables(None, None, None)
        return
    t = [np.ascontiguousarray(x, dtype=np.int32) for x in tables]
    assert [len(x) for x in t] == [65536, 131072, 131072]
    L.ref_set_sampler_tables(*[x.ctypes.data_as(C.c_void_p) for x in t])


class RefRenderer:
    """One reference scene + integrator instance on the CPU."""

    def __init__(self, libm: bool = False):
        path = os.path.join(REF_DIR, "libref_libm.so" if libm else "libref.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing: run python oracle/build_ref.py where /root/reference exists")
        L = self.lib = C.CDLL(path)
        L.ref_open_obj.restype = C.c_void_p
        L.ref_open_obj.argtypes = [C.c_char_p, C.c_char_p, C.c_float, C.c_int, C.c_int]
        L.ref_open_arrays.restype = C.c_void_p
        L.ref_open_arrays.argtypes = [C.c_void_p, C.c_size_t] * 7 + [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.ref_scene_query.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.ref_begin.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        for name in ("ref_set_camera",):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p]
        for name in ("ref_set_max_bounces",):
            getattr(L, name).argtypes = [C.c_void_p, C.c_uint32]
        for name in ("ref_enable_white_furnace", "ref_set_sampler", "ref_enable_denoiser", "ref_set_aov"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int]
        for name in ("ref_request_reset", "ref_integrate", "ref_close"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.ref_set_row_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.ref_sampler_tables.argtypes = [C.POINTER(C.POINTER(C.c_int))] * 3
        L.ref_read.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        self.h = None
        self.width = self.height = 0

    # ---- scene
    def open_obj(self, ref_root: str, obj_rel_path: str, scale=1.0, flip_yz=False, default_light=True):
        self.h = self.lib.ref_open_obj(ref_root.encode(), obj_rel_path.encode(), scale, int(flip_yz), int(default_light))
        if not self.h:
            raise RuntimeError("ref_open_obj failed")
        return self

    def open_arrays(self, scene: dict):
        a = {k: np.ascontiguousarray(scene[k]) for k, _ in SCENE_ARRAYS}
        env = a["env"]
        args = []
        for k in ("triangles", "nodes", "materials", "lights", "textures", "texels", "emissive"):
            args += [a[k].ctypes.data_as(C.c_void_p), a[k].shape[0]]
        self._keep = a
        self.h = self.lib.ref_open_arrays(*args, env.ctypes.data_as(C.c_void_p), int(scene["env_width"]), int(scene["env_height"]),
                                          a["scene_info"].ctypes.data_as(C.c_void_p))
        return self

    def scene(self) -> dict:
        out = {}
        for i, (name, dt) in enumerate(SCENE_ARRAYS):
            p, n, e0, e1 = C.c_void_p(), C.c_size_t(), C.c_uint32(), C.c_uint32()
            self.lib.ref_scene_query(self.h, i, C.byref(p), C.byref(n), C.byref(e0), C.byref(e1))
            nbytes = n.value * dt.itemsize
            buf = (C.c_char * nbytes).from_address(p.value) if nbytes else b""
            out[name] = np.frombuffer(bytes(buf), dtype=dt).copy()
            if name == "env":
                out["env_width"], out["env_height"] = e0.value, e1.value
        return out

    # ---- integrator
    def begin(self, width: int, height: int):
        self.width, self.height = width, height
        self.lib.ref_begin(self.h, width, height)
        return self

    def set_camera(self, cam: np.ndarray):
        c = np.ascontiguousarray(cam)
        self.lib.ref_set_camera(self.h, c.ctypes.data_as(C.c_void_p))

    def set_max_bounces(self, b): self.lib.ref_set_max_bounces(self.h, b)
    def enable_white_furnace(self, e): self.lib.ref_enable_white_furnace(self.h, int(e))
    def set_blue_noise(self, e): self.lib.ref_set_sampler(self.h, int(e))

    def sampler_tables(self):
        """(sobol[65536], scrambling[131072], ranking[131072]) int32 copies of the tables the reference compiled in."""
        ps = [C.POINTER(C.c_int)() for _ in range(3)]
        self.lib.ref_sampler_tables(*[C.byref(p) for p in ps])
        return tuple(np.ctypeslib.as_array(p, shape=(n,)).astype(np.int32) for p, n in zip(ps, (65536, 131072, 131072)))
    def enable_denoiser(self, e): self.lib.ref_enable_denoiser(self.h, int(e))
    def set_aov(self, a): self.lib.ref_set_aov(self.h, int(a))
    def set_row_sample(self, first, step): self.lib.ref_set_row_sample(self.h, first, step)
    def request_reset(self): self.lib.ref_request_reset(self.h)
    def integrate(self): self.lib.ref_integrate(self.h)

    def _read(self, which, dtype, count):
        out = np.zeros(count, dtype=dtype)
        self.lib.ref_read(self.h, which, out.ctypes.data_as(C.c_void_p))
        return out

    def radiance(self): return self._read(0, "<f4", self.width * self.height * 4).reshape(self.height, self.width, 4)
    def resolved(self): return self._read(1, "<f4", self.width * self.height * 4).reshape(self.height, self.width, 4)
    def primary_hits(self): return self._read(2, HIT_DT, self.width * self.height)
    def primary_rays(self): return self._read(3, RAY_DT, self.width * self.height)

    def stats(self) -> dict:
        s = self._read(4, "<u4", 6 * 64).reshape(6, 64)
        return {k: s[i] for i, k in enumerate(("n_ext", "n_miss", "n_hit", "n_shadow", "n_cont", "n_unoccluded"))}

    def sample_count(self): return int(self._read(5, "<u4", 1)[0])
    def aov_albedo(self): return self._read(6, "<f4", self.width * self.height * 4).reshape(self.height, self.width, 4)
    def aov_depth(self): return self._read(7, "<f4", self.width * self.height).reshape(self.height, self.width)
    def aov_normal(self): return self._read(8, "<f4", self.width * self.height * 4).reshape(self.height, self.width, 4)
    def aov_velocity(self): return self._read(9, "<f4", self.width * self.height * 2).reshape(self.height, self.width, 2)

    def close(self):
        if self.h:
            self.lib.ref_close(self.h)
            self.h = None
