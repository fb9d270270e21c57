"""CPU reference of the emissive-MIS light sampling (tests/emissive_oracle.cpp: the oracle's own code plus the extension
mode, which has no GLSL counterpart).  The library is compiled on first use into the temporary directory, keyed by the
hash of its sources, so a read-only checkout works and the oracle itself stays untouched."""
import ctypes as C
import hashlib
import importlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "emissive_oracle.cpp")] + [
    os.path.join(_ROOT, "oracle", f) for f in ("pt_oracle.cpp", "pt_oracle.h", "glsl_math.h")] + [
    os.path.join(_ROOT, "include", "pt_core.h")]
# the oracle's flags (oracle/Makefile): no contraction, no fast math — the emitter table must match the GPU's bit for bit
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wno-subobject-linkage", "-pthread", "-shared"]
LIGHT_SAMPLING = ("reference", "emissive_mis")

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for path in _SOURCES:
            with open(path, "rb") as f:
                h.update(f.read())
        h.update(" ".join(_FLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"pt_emissive_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(path))
            os.close(fd)
            try:
                subprocess.check_call([os.environ.get("CXX", "g++"), *_FLAGS, "-o", tmp, _SOURCES[0]])
                os.replace(tmp, path)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        L = C.CDLL(path)
        vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int32
        L.pto_scene_create_limits.restype = vp
        L.pto_scene_create_limits.argtypes = [vp, u32, C.c_uint64]
        L.pto_scene_destroy.argtypes = [vp]
        L.pto_render.argtypes = [vp, vp, u32, u32, u32, u32, vp, u32, vp, i32, vp]
        L.pto_texture_sample.argtypes = [vp, u32, vp, vp, u32, i32]
        L.ptx_emitters_create.restype = vp
        L.ptx_emitters_create.argtypes = [vp]
        L.ptx_emitters_destroy.argtypes = [vp]
        L.ptx_emitter_table.argtypes = [vp, vp, vp, vp, vp, vp, u32]
        L.ptx_render_frames.argtypes = [vp, vp, vp, u32, u32, u32, u32, u32, vp, u32, vp, i32, vp]
        _lib = L
    return _lib


class EmissiveOracleScene:
    """The oracle's scene with a light-sampling mode: "reference" renders with the oracle's raygen, "emissive_mis" with
    the extension's; render() has the signature of oracle.OracleScene.render."""

    def __init__(self, scene):
        from oracle import oracle

        self._Counters = oracle.Counters
        self._sc = importlib.import_module("path-tracing_b200.scene")
        desc, keep = scene.to_c()
        self._h = lib().pto_scene_create_limits(C.addressof(desc), 4096, 0)
        del keep
        assert self._h, "pto_scene_create failed"
        self._em = lib().ptx_emitters_create(self._h)
        self.mode = "reference"

    def close(self):
        if self._h:
            lib().ptx_emitters_destroy(self._em)
            lib().pto_scene_destroy(self._h)
            self._h = self._em = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_light_sampling(self, mode: str):
        assert mode in LIGHT_SAMPLING, mode
        self.mode = mode

    def emitter_table(self) -> dict:
        n = C.c_uint32(0)
        assert lib().ptx_emitter_table(self._em, C.byref(n), None, None, None, None, 0) == 0
        t = {k: np.zeros(n.value, np.uint32) for k in ("flat_ids", "weights", "alias_threshold", "alias_index")}
        assert lib().ptx_emitter_table(self._em, C.byref(n), *(t[k].ctypes.data for k in t), n.value) == 0
        return t

    def texture_sample(self, slot, uv_ddx_ddy, use_grad=True):
        a = np.ascontiguousarray(uv_ddx_ddy, np.float32).reshape(-1, 6)
        out = np.zeros((a.shape[0], 4), np.float32)
        assert lib().pto_texture_sample(self._h, slot, a.ctypes.data, out.ctypes.data, a.shape[0], 1 if use_grad else 0) == 0
        return out

    def render(self, params, width, height, first_sample, sample_count, accum=None, tiles=None, threads=0):
        if accum is None:
            accum = np.zeros((height, width, 4), np.float32)
        assert accum.dtype == np.float32 and accum.flags.c_contiguous
        p = params.to_c()
        cnt = self._Counters()
        tl = None if tiles is None else np.ascontiguousarray(tiles, self._sc.TILE)
        tiles_ptr, tile_count = (None, 0) if tl is None else (tl.ctypes.data, len(tl))
        if self.mode == "reference":
            rc = lib().pto_render(self._h, C.addressof(p), width, height, first_sample, sample_count, tiles_ptr, tile_count,
                                  accum.ctypes.data, threads, C.addressof(cnt))
        else:
            rc = lib().ptx_render_frames(self._h, self._em, C.addressof(p), width, height, first_sample, sample_count, 1,
                                         tiles_ptr, tile_count, accum.ctypes.data, threads, C.addressof(cnt))
        assert rc == 0, rc
        return accum, cnt.as_dict()
