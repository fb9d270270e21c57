"""ctypes binding of the C ABI (include/pt_core.h) — the Python face of the drop-in boundary.

``Renderer`` mirrors the verbs of the reference's ``Renderer`` facade
(Path-Tracing/Renderer/Renderer.h:42-85) the same way the C++ ``HeadlessRenderer`` does:
``update_scene_data`` / ``on_resize`` / ``set_settings`` / ``render`` / ``read_accumulation``.
There is no CPU fallback: if the CUDA library is missing or no sm_100 device is present the
constructor raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import scene as sc

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# PT_CORE_LIB selects another build of the same library (A/B experiments with kernel variants)
LIB_PATH = os.environ.get("PT_CORE_LIB") or os.path.join(CSRC, "libpt_core.so")

ABI_SYMBOLS = [
    "pt_context_create",
    "pt_context_destroy",
    "pt_last_error",
    "pt_scene_upload",
    "pt_scene_update",
    "pt_texture_upload",
    "pt_set_sampler",
    "pt_render_begin",
    "pt_render_samples",
    "pt_render_frames",
    "pt_accum_device_ptr",
    "pt_readback",
    "pt_postprocess",
    "pt_synchronize",
    "pt_first_hit_aov",
    "pt_trace_closest",
    "pt_trace_occlusion",
    "pt_get_stats",
    "pt_set_traversal_stats",
    "pt_set_kernel_timing",
    "pt_set_tuning",
    "pt_test_input_stride",
    "pt_test_output_stride",
    "pt_test_shading",
    "pt_test_texture",
    "pt_debug_render",
    "pt_set_light_sampling",
    "pt_emitter_table",
]

# pt_light_sampling, include/pt_core.h
LIGHT_SAMPLING = {"reference": 0, "emissive_mis": 1}


class PtError(RuntimeError):
    """Counterpart of PathTracing::error (Path-Tracing/Core/Core.cpp:82-90)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[{status}] {message}")
        self.status = status


KERNEL_CLASSES = ("extend", "shade", "shadow", "finish")


class PostProcessParams(C.Structure):
    """pt_postprocess_params = Renderer::PostProcessSettings (Path-Tracing/Renderer/Renderer.h:68-73) + tone-mapping mode."""

    _fields_ = [("exposure", C.c_float), ("bloom_threshold", C.c_float), ("bloom_intensity", C.c_float), ("tone_mapping", C.c_uint32)]


class SceneUpdateDesc(C.Structure):
    """pt_scene_update_desc."""

    _fields_ = [("instance_transforms", C.c_void_p), ("instance_count", C.c_uint32), ("point_lights", C.c_void_p),
                ("point_light_count", C.c_uint32), ("directional_light", C.c_void_p), ("bone_transforms", C.c_void_p),
                ("bone_count", C.c_uint32)]


class DebugParams(C.Structure):
    """pt_debug_params: render mode + raygen / hit-group flags of the reference's debug pipeline."""

    _fields_ = [("render_mode", C.c_uint32), ("raygen_flags", C.c_uint32), ("hit_group_flags", C.c_uint32)]


DEBUG_MODES = ("color", "world_position", "normal", "texture_coords", "mips", "geometry", "primitive", "instance")
TONE_MAPPING_SDR, TONE_MAPPING_HDR = 0, 1
OUTPUT_RGBA8_SRGB, OUTPUT_RGBAF32 = 0, 1


class Stats(C.Structure):
    _fields_ = [
        ("rays_closest", C.c_uint64),
        ("rays_shadow", C.c_uint64),
        ("samples", C.c_uint64),
        ("hits", C.c_uint64),
        ("box_tests_closest", C.c_uint64),
        ("tri_tests_closest", C.c_uint64),
        ("alpha_tests_closest", C.c_uint64),
        ("box_tests_shadow", C.c_uint64),
        ("tri_tests_shadow", C.c_uint64),
        ("alpha_tests_shadow", C.c_uint64),
        ("texel_fetches", C.c_uint64),
        ("restarts", C.c_uint64),
        ("wavefront_iterations", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("triangle_count", C.c_uint64),
        ("bvh_node_count", C.c_uint64),
        ("bvh_bytes", C.c_uint64),
        ("bvh_build_ms", C.c_float),
        ("scene_upload_ms", C.c_float),
        ("last_render_ms", C.c_float),
        ("kernel_ms", C.c_float * 4),
        ("kernel_launch_count", C.c_uint32 * 4),
        ("node_visit_hist", C.c_uint64 * 8),
        ("warp_iterations", C.c_uint64),
        ("warp_drain_iterations", C.c_uint64),
        ("max_warp_drain_iterations", C.c_uint64),
        ("bvh_reference_count", C.c_uint64),
        ("bvh_max_depth", C.c_uint32),
        ("stack_overflows", C.c_uint32),
    ]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_}
        d["kernel_ms"] = dict(zip(KERNEL_CLASSES, [float(x) for x in self.kernel_ms]))
        d["kernel_launch_count"] = dict(zip(KERNEL_CLASSES, [int(x) for x in self.kernel_launch_count]))
        d["node_visit_hist"] = [int(x) for x in self.node_visit_hist]
        return d


def build(verbose: bool = False) -> str:
    """Compiles every CUDA source for sm_100a with the committed Makefile (nvcc cross-compiles)."""
    subprocess.check_call(["make", "-C", CSRC, "-j4", "libpt_core.so"], stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def write_png(path: str, rgba8: np.ndarray):
    """Minimal PNG writer (8-bit RGBA, zlib, no filtering) — the reference uses stb_image_write."""
    import struct
    import zlib

    h, w = rgba8.shape[:2]
    raw = np.concatenate([np.zeros((h, 1), np.uint8), np.ascontiguousarray(rgba8, np.uint8).reshape(h, w * 4)], 1).tobytes()

    def chunk(tag: bytes, data: bytes) -> bytes:
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0)) +
                chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


def write_hdr(path: str, rgba: np.ndarray):
    """Radiance .hdr (RGBE, flat scanlines) of a float image — the reference writes OutputFormat::Hdr with
    stbi_write_hdr (Path-Tracing/Renderer/OutputSaver.cpp:240-245); same encoding rule: shared exponent of the
    largest component, mantissas truncated."""
    rgb = np.ascontiguousarray(rgba[..., :3], np.float32)
    h, w = rgb.shape[:2]
    m = rgb.max(-1)
    mant, exp = np.frexp(m)  # m = mant * 2^exp, mant in [0.5, 1)
    scale = np.where(m < 1e-32, 0.0, mant * 256.0 / np.where(m < 1e-32, 1.0, m))
    out = np.zeros((h, w, 4), np.uint8)
    out[..., :3] = (rgb * scale[..., None]).astype(np.uint8)
    out[..., 3] = np.where(m < 1e-32, 0, exp + 128).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n" + f"-Y {h} +X {w}\n".encode() + out.tobytes())


def write_tga(path: str, rgba8: np.ndarray):
    """Uncompressed 32-bit TGA, top-left origin (OutputFormat::Tga, stbi_write_tga without RLE)."""
    import struct

    h, w = rgba8.shape[:2]
    bgra = np.ascontiguousarray(rgba8[..., [2, 1, 0, 3]], np.uint8)
    with open(path, "wb") as f:
        f.write(struct.pack("<BBBHHBHHHHBB", 0, 0, 2, 0, 0, 0, 0, 0, w, h, 32, 0x28) + bgra.tobytes())


def write_exr(path: str, rgba: np.ndarray):
    """OpenEXR 2.0 scanline file, uncompressed, 32-bit float channels A, B, G, R — the headless float output the task names
    beside PNG (the reference's own float format is .hdr; EXR keeps all 32 bits and the alpha).  One chunk per scanline:
    y, byte count, then the channels in alphabetical order, each a row of little-endian floats."""
    import struct

    img = np.ascontiguousarray(rgba, np.float32)
    h, w = img.shape[:2]

    def attr(name: str, typ: str, data: bytes) -> bytes:
        return name.encode() + b"\0" + typ.encode() + b"\0" + struct.pack("<i", len(data)) + data

    chlist = b"".join(c.encode() + b"\0" + struct.pack("<iBBBBii", 2, 0, 0, 0, 0, 1, 1) for c in "ABGR") + b"\0"
    box = struct.pack("<iiii", 0, 0, w - 1, h - 1)
    header = (attr("channels", "chlist", chlist) + attr("compression", "compression", b"\0") + attr("dataWindow", "box2i", box) +
              attr("displayWindow", "box2i", box) + attr("lineOrder", "lineOrder", b"\0") + attr("pixelAspectRatio", "float", struct.pack("<f", 1.0)) +
              attr("screenWindowCenter", "v2f", struct.pack("<ff", 0.0, 0.0)) + attr("screenWindowWidth", "float", struct.pack("<f", 1.0)) + b"\0")
    magic = struct.pack("<ii", 20000630, 2)
    row_bytes = 4 * 4 * w
    first = len(magic) + len(header) + 8 * h
    offsets = b"".join(struct.pack("<Q", first + y * (8 + row_bytes)) for y in range(h))
    planes = img[..., [3, 2, 1, 0]].transpose(0, 2, 1)  # (h, channel A B G R, w)
    with open(path, "wb") as f:
        f.write(magic + header + offsets)
        for y in range(h):
            f.write(struct.pack("<ii", y, row_bytes) + planes[y].tobytes())


def read_exr(path: str) -> np.ndarray:
    """Reads back what write_exr wrote (uncompressed float scanlines, channels A B G R): (h, w, 4) float32 RGBA."""
    import struct

    data = open(path, "rb").read()
    assert struct.unpack_from("<ii", data, 0) == (20000630, 2)
    pos, attrs = 8, {}
    while data[pos] != 0:
        end = data.index(b"\0", pos)
        name = data[pos:end].decode()
        tend = data.index(b"\0", end + 1)
        size = struct.unpack_from("<i", data, tend + 1)[0]
        attrs[name] = data[tend + 5 : tend + 5 + size]
        pos = tend + 5 + size
    pos += 1
    x0, y0, x1, y1 = struct.unpack("<iiii", attrs["dataWindow"])
    w, h = x1 - x0 + 1, y1 - y0 + 1
    assert attrs["compression"] == b"\0"
    out = np.zeros((h, w, 4), np.float32)
    for k in range(h):
        off = struct.unpack_from("<Q", data, pos + 8 * k)[0]
        y, n = struct.unpack_from("<ii", data, off)
        planes = np.frombuffer(data, np.float32, 4 * w, off + 8).reshape(4, w)
        out[y - y0] = planes[[3, 2, 1, 0]].T
    return out


_lib = None


def lib():
    """Loads libpt_core.so.  Raises if it has not been built — the product never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PtError(-2, f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32
    L.pt_context_create.argtypes = [i32, C.POINTER(vp)]
    L.pt_context_destroy.argtypes = [vp]
    L.pt_context_destroy.restype = None
    L.pt_last_error.argtypes = [vp]
    L.pt_last_error.restype = C.c_char_p
    L.pt_scene_upload.argtypes = [vp, vp]
    L.pt_scene_update.argtypes = [vp, vp]
    L.pt_texture_upload.argtypes = [vp, u32, vp]
    L.pt_render_begin.argtypes = [vp, u32, u32]
    L.pt_render_samples.argtypes = [vp, vp, u32, u32, vp, u32]
    L.pt_render_frames.argtypes = [vp, vp, u32, u32, u32, vp, u32]
    L.pt_set_sampler.argtypes = [vp, u32]
    L.pt_set_light_sampling.argtypes = [vp, u32]
    L.pt_emitter_table.argtypes = [vp, vp, vp, vp, vp, vp, u32]
    L.pt_accum_device_ptr.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(vp)]
    L.pt_readback.argtypes = [vp, vp, C.c_size_t]
    L.pt_postprocess.argtypes = [vp, vp, u32, u32, vp, C.c_size_t]
    L.pt_synchronize.argtypes = [vp]
    L.pt_first_hit_aov.argtypes = [vp, vp, u32, u32, vp]
    L.pt_trace_closest.argtypes = [vp, vp, u64, vp]
    L.pt_trace_occlusion.argtypes = [vp, vp, u64, vp]
    L.pt_get_stats.argtypes = [vp, vp]
    L.pt_set_traversal_stats.argtypes = [vp, i32]
    L.pt_set_kernel_timing.argtypes = [vp, i32]
    L.pt_set_tuning.argtypes = [vp, C.c_char_p, u64]
    L.pt_test_input_stride.argtypes = [u32]
    L.pt_test_input_stride.restype = u32
    L.pt_test_output_stride.argtypes = [u32]
    L.pt_test_output_stride.restype = u32
    L.pt_test_shading.argtypes = [vp, u32, vp, vp, u32]
    L.pt_test_texture.argtypes = [vp, u32, vp, vp, u32, i32]
    L.pt_debug_render.argtypes = [vp, vp, vp, u32, u32, vp]
    _lib = L
    return L


class Renderer:
    def __init__(self, cuda_device: int = 0):
        self._L = lib()
        h = C.c_void_p()
        st = self._L.pt_context_create(cuda_device, C.byref(h))
        if st != 0:
            raise PtError(st, (self._L.pt_last_error(None) or b"").decode())
        self._h = h
        self.width = self.height = 0
        self.total_samples = 0
        self.params: sc.RenderParams | None = None

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, st: int):
        if st != 0:
            raise PtError(st, (self._L.pt_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.pt_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- Renderer verbs ---------------------------------------------------------------------
    def update_scene_data(self, scene: sc.SceneData):
        """Renderer::UpdateSceneData for a new scene: upload + GPU BVH build (blocking)."""
        desc, keep = scene.to_c()
        self._check(self._L.pt_scene_upload(self._h, C.addressof(desc)))
        del keep
        self.total_samples = 0
        if self.width:
            self.on_resize(self.width, self.height)

    def update_scene(self, instance_transforms=None, point_lights=None, directional_light=None, bone_transforms=None):
        """The per-frame half of Renderer::UpdateSceneData for animated scenes (Scene::Update's outputs):
        new instance transforms ((N, 12) float32, 3x4 row-major) re-bake the instances and rebuild the BVH;
        point_lights (sc.POINT_LIGHT records) / directional_light (sc.DIRECTIONAL_LIGHT record) rewrite the
        light block; bone_transforms ((B, 12) float32) re-skin the animated geometries (skinning.comp) before the
        rebuild.  The accumulation is not reset — call on_resize() like the reference's `updated` flag."""
        d = SceneUpdateDesc()
        keep = []
        if instance_transforms is not None:
            t = np.ascontiguousarray(instance_transforms, np.float32).reshape(-1, 12)
            keep.append(t)
            d.instance_transforms, d.instance_count = t.ctypes.data, len(t)
        if point_lights is not None:
            pl = np.ascontiguousarray(point_lights, sc.POINT_LIGHT)
            keep.append(pl)
            d.point_lights, d.point_light_count = pl.ctypes.data, len(pl)
        if directional_light is not None:
            dl = np.ascontiguousarray(directional_light, sc.DIRECTIONAL_LIGHT).reshape(1)
            keep.append(dl)
            d.directional_light = dl.ctypes.data
        if bone_transforms is not None:
            bt = np.ascontiguousarray(bone_transforms, np.float32).reshape(-1, 12)
            keep.append(bt)
            d.bone_transforms, d.bone_count = bt.ctypes.data, len(bt)
        self._check(self._L.pt_scene_update(self._h, C.addressof(d)))

    def upload_texture(self, slot: int, tex: sc.Texture):
        px = np.ascontiguousarray(tex.pixels)
        d = sc.CTextureDesc(tex.width, tex.height, tex.format, 1 if tex.srgb else 0, px.ctypes.data, tex.levels)
        self._check(self._L.pt_texture_upload(self._h, slot, C.addressof(d)))

    def on_resize(self, width: int, height: int):
        """Renderer::OnResize / accumulation reset."""
        self._check(self._L.pt_render_begin(self._h, width, height))
        self.width, self.height = width, height
        self.total_samples = 0

    def set_settings(self, params: sc.RenderParams):
        self.params = params

    def render(self, samples: int = 1, tiles=None, params: sc.RenderParams | None = None, first_sample: int | None = None):
        """Renderer::Render with SamplesPerFrame = samples (frames of 1 sample, TotalSamples advancing)."""
        p = (params or self.params).to_c()
        first = self.total_samples if first_sample is None else first_sample
        tl = None if tiles is None else np.ascontiguousarray(tiles, sc.TILE)
        self._check(
            self._L.pt_render_samples(
                self._h, C.addressof(p), first, samples, None if tl is None else tl.ctypes.data, 0 if tl is None else len(tl)
            )
        )
        if first_sample is None:
            self.total_samples += samples

    def render_frames(self, frames: int, samples_per_frame: int, tiles=None, params: sc.RenderParams | None = None,
                      first_sample: int | None = None):
        """Renderer::Render `frames` times with SamplesPerFrame = samples_per_frame (one rng stream and one radiance
        sum per pixel and frame, Renderer.cpp:1688-1700)."""
        p = (params or self.params).to_c()
        first = self.total_samples if first_sample is None else first_sample
        tl = None if tiles is None else np.ascontiguousarray(tiles, sc.TILE)
        self._check(self._L.pt_render_frames(self._h, C.addressof(p), first, frames, samples_per_frame,
                                             None if tl is None else tl.ctypes.data, 0 if tl is None else len(tl)))
        if first_sample is None:
            self.total_samples += frames * samples_per_frame

    def read_accumulation(self, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.height, self.width, 4), np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == self.width * self.height * 4
        self._check(self._L.pt_readback(self._h, out.ctypes.data, out.nbytes))
        return out

    def postprocess(self, exposure: float = 1.0, bloom_threshold: float = 1.0, bloom_intensity: float = 0.1, hdr: bool = False,
                    total_samples: int | None = None) -> np.ndarray:
        """What the reference's "Render" button writes (Renderer::RecordPostProcessCommands +
        RecordSaveOutputCommands + OutputSaver): exposure, bloom, tone mapping and the output-format
        conversion of the accumulated image.  (H, W, 4) uint8 sRGB, or float32 with hdr (the .hdr output,
        not tone-mapped)."""
        p = PostProcessParams(exposure, bloom_threshold, bloom_intensity, TONE_MAPPING_HDR if hdr else TONE_MAPPING_SDR)
        out = np.empty((self.height, self.width, 4), np.float32 if hdr else np.uint8)
        n = self.total_samples if total_samples is None else total_samples
        self._check(self._L.pt_postprocess(self._h, C.addressof(p), int(n), OUTPUT_RGBAF32 if hdr else OUTPUT_RGBA8_SRGB,
                                           out.ctypes.data, out.nbytes))
        return out

    def save_png(self, path: str, **postprocess_args):
        """OutputSaver::WriteImage for OutputFormat::Png (Path-Tracing/Renderer/OutputSaver.cpp:227-253):
        8-bit RGBA, rows top to bottom."""
        write_png(path, self.postprocess(hdr=False, **postprocess_args))

    def save_hdr(self, path: str, **postprocess_args):
        """OutputFormat::Hdr: the chain without the tone curve, written as Radiance RGBE."""
        write_hdr(path, self.postprocess(hdr=True, **postprocess_args))

    def save_tga(self, path: str, **postprocess_args):
        """OutputFormat::Tga: the same 8-bit sRGB image as the PNG."""
        write_tga(path, self.postprocess(hdr=False, **postprocess_args))

    def save_exr(self, path: str, **postprocess_args):
        """The float output (the chain without the tone curve, like .hdr) as an OpenEXR file with all 32 bits per channel."""
        write_exr(path, self.postprocess(hdr=True, **postprocess_args))

    def save_jpg(self, path: str, **postprocess_args):
        """OutputFormat::Jpg (OutputSaver.cpp:237-238: stbi_write_jpg, quality argument 0 = stb's default of 90): the same
        8-bit sRGB image, baseline JPEG of its RGB channels.  Written with Pillow here (the C++ shim uses the reference's
        own stb writer): the files decode to the same picture, the byte streams are not compared."""
        from PIL import Image

        Image.fromarray(self.postprocess(hdr=False, **postprocess_args)[..., :3], "RGB").save(path, "JPEG", quality=90)

    def readback_into(self, host_ptr: int, nbytes: int):
        """pt_readback into caller-owned (e.g. pinned) host memory."""
        self._check(self._L.pt_readback(self._h, host_ptr, nbytes))

    def accum_device_ptr(self):
        ptr, pitch, stream = C.c_void_p(), C.c_size_t(), C.c_void_p()
        self._check(self._L.pt_accum_device_ptr(self._h, C.byref(ptr), C.byref(pitch), C.byref(stream)))
        return ptr.value, pitch.value, stream.value

    def synchronize(self):
        self._check(self._L.pt_synchronize(self._h))

    # -- queries ----------------------------------------------------------------------------
    def first_hit_aov(self, params: sc.RenderParams, width: int, height: int) -> np.ndarray:
        out = np.zeros(width * height, sc.HIT)
        p = params.to_c()
        self._check(self._L.pt_first_hit_aov(self._h, C.addressof(p), width, height, out.ctypes.data))
        return out.reshape(height, width)

    def trace_closest(self, rays: np.ndarray) -> np.ndarray:
        rays = np.ascontiguousarray(rays, sc.RAY)
        out = np.zeros(len(rays), sc.HIT)
        self._check(self._L.pt_trace_closest(self._h, rays.ctypes.data, len(rays), out.ctypes.data))
        return out

    def trace_occlusion(self, rays: np.ndarray) -> np.ndarray:
        rays = np.ascontiguousarray(rays, sc.RAY)
        out = np.zeros(len(rays), np.uint8)
        self._check(self._L.pt_trace_occlusion(self._h, rays.ctypes.data, len(rays), out.ctypes.data))
        return out

    def stats(self) -> dict:
        s = Stats()
        self._check(self._L.pt_get_stats(self._h, C.addressof(s)))
        return s.as_dict()

    def set_traversal_stats(self, enable: bool):
        self._check(self._L.pt_set_traversal_stats(self._h, 1 if enable else 0))

    def set_tuning(self, key: str, value: int):
        """Scheduling knobs (pools, slots, sort_hits, sbuf_mb); results do not depend on them."""
        self._check(self._L.pt_set_tuning(self._h, key.encode(), int(value)))

    def set_sampler(self, max_anisotropy: int):
        """Sampler state (Renderer.cpp:103-112): maximum anisotropy of the material fetches, 1 = isotropic (default) .. 16 (the reference's)."""
        self._check(self._L.pt_set_sampler(self._h, int(max_anisotropy)))

    def set_kernel_timing(self, enable: bool):
        self._check(self._L.pt_set_kernel_timing(self._h, 1 if enable else 0))

    def set_light_sampling(self, mode: str):
        """Light sampling of next-event estimation: "reference" (default: the reference's analytic lights) or
        "emissive_mis" (also the scene's emissive triangles, with multiple importance sampling; DESIGN.md §3g).
        Takes effect at the next render; the accumulation is not reset."""
        if mode not in LIGHT_SAMPLING:
            raise ValueError(f"light sampling must be one of {sorted(LIGHT_SAMPLING)}, not {mode!r}")
        self._check(self._L.pt_set_light_sampling(self._h, LIGHT_SAMPLING[mode]))

    def emitter_table(self) -> dict:
        """The emitter table of the "emissive_mis" mode (built now if out of date): uint32 arrays flat_ids (flattened
        triangle ids), weights (integer selection weights) and the alias entries alias_threshold, alias_index."""
        n = C.c_uint32(0)
        self._check(self._L.pt_emitter_table(self._h, C.byref(n), None, None, None, None, 0))
        t = {k: np.zeros(n.value, np.uint32) for k in ("flat_ids", "weights", "alias_threshold", "alias_index")}
        self._check(self._L.pt_emitter_table(self._h, C.byref(n), *(t[k].ctypes.data for k in t), n.value))
        return t

    def debug_render(self, params: sc.RenderParams, width: int, height: int, mode="color", raygen_flags: int = 0,
                     hit_group_flags: int = 0) -> np.ndarray:
        """One frame of the reference's debug pipeline (Debug/debug*.r*): (H, W, 4) float32."""
        d = DebugParams(DEBUG_MODES.index(mode) if isinstance(mode, str) else int(mode), raygen_flags, hit_group_flags)
        p = params.to_c()
        out = np.zeros((height, width, 4), np.float32)
        self._check(self._L.pt_debug_render(self._h, C.addressof(p), C.addressof(d), width, height, out.ctypes.data))
        return out

    def texture_sample(self, slot: int, uv_ddx_ddy: np.ndarray, use_grad: bool = True) -> np.ndarray:
        """The production sampler on (N, 6) records of uv, dPdx, dPdy -> (N, 4) RGBA (pt_test_texture)."""
        a = np.ascontiguousarray(uv_ddx_ddy, np.float32).reshape(-1, 6)
        out = np.zeros((a.shape[0], 4), np.float32)
        self._check(self._L.pt_test_texture(self._h, slot, a.ctypes.data, out.ctypes.data, a.shape[0], 1 if use_grad else 0))
        return out

    def test_shading(self, mode: int, inputs: np.ndarray) -> np.ndarray:
        """TestRenderer::ExecutePipeline equivalent (Path-Tracing-Tests/TestRenderer.cpp:79-106)."""
        n_in, n_out = self._L.pt_test_input_stride(mode), self._L.pt_test_output_stride(mode)
        inputs = np.ascontiguousarray(inputs, np.float32).reshape(-1, n_in)
        out = np.zeros((inputs.shape[0], n_out), np.float32)
        self._check(self._L.pt_test_shading(self._h, mode, inputs.ctypes.data, out.ctypes.data, inputs.shape[0]))
        return out
