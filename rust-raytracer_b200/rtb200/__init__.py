"""rtb200 — Python host binding of the B200 render path (ctypes over the C ABI in include/rtb200.h).

Mirrors the reference's host-side interface for the path it replaces:
  * ``Config`` / ``Sphere`` / ``Camera`` JSON schema   (reference raytracer/src/config.rs:66-75, sphere.rs:18-23,
    camera.rs:29-36, materials.rs:35-42)  ->  :func:`load_scene`, :class:`Scene`
  * ``render(filename, scene)``                          (reference raytracer/src/raytracer.rs:250-266) -> :func:`render`
The hot path itself lives in ``librtb200.so`` (hand-written sm_100a CUDA). There is no CPU fallback: if the
library or a B200 is missing every render call raises :class:`RtError`.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RTB200_LIB") or os.path.join(os.path.dirname(_HERE), "librtb200.so")   # RTB200_LIB: experimental builds

RT_LAMBERTIAN, RT_METAL, RT_GLASS, RT_TEXTURE, RT_LIGHT = 0, 1, 2, 3, 4
RT_SKY_NONE, RT_SKY_GRADIENT, RT_SKY_TEXTURE = 0, 1, 2
RT_VARIANT_AUTO, RT_VARIANT_FILTERED, RT_VARIANT_EXACT_F64, RT_VARIANT_RETIRED_LANES, RT_VARIANT_BRUTE_FORCE = 0, 1, 2, 3, 4

DEFAULT_SEED = 0x5EED


class RtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rtb200 error {code}: {msg}")
        self.code = code


# ---- ctypes mirrors of include/rtb200.h ---------------------------------------------------------------
class rt_vec3(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]

    def tup(self):
        return (self.x, self.y, self.z)


class rt_camera(C.Structure):
    _fields_ = [("origin", rt_vec3), ("lower_left_corner", rt_vec3), ("horizontal", rt_vec3), ("vertical", rt_vec3)]


class rt_camera_params(C.Structure):
    _fields_ = [("look_from", rt_vec3), ("look_at", rt_vec3), ("vup", rt_vec3), ("vfov_deg", C.c_double), ("aspect", C.c_double)]


class rt_sphere(C.Structure):
    _fields_ = [("center", rt_vec3), ("radius", C.c_double), ("kind", C.c_uint32), ("albedo", C.c_float * 3),
                ("param", C.c_double), ("texture", C.c_int32), ("reserved", C.c_int32)]


class rt_image(C.Structure):
    _fields_ = [("rgb8", C.c_void_p), ("width", C.c_uint64), ("height", C.c_uint64), ("bytes", C.c_uint64)]


class rt_sky(C.Structure):
    _fields_ = [("mode", C.c_uint32), ("reserved", C.c_uint32), ("tex", rt_image)]


class rt_scene(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples_per_pixel", C.c_uint32), ("max_depth", C.c_uint32),
                ("camera", rt_camera), ("sky", rt_sky),
                ("spheres", C.POINTER(rt_sphere)), ("n_spheres", C.c_uint64),
                ("textures", C.POINTER(rt_image)), ("n_textures", C.c_uint64),
                ("seed", C.c_uint64)]


class rt_options(C.Structure):
    _fields_ = [("device", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32), ("band_rows", C.c_uint32),
                ("variant", C.c_uint32), ("flags", C.c_uint32), ("sample_buffer_bytes", C.c_uint64)]


class rt_stats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("samples", C.c_uint64), ("candidates", C.c_uint64),
                ("device_ms", C.c_double), ("trace_ms", C.c_double), ("wall_ms", C.c_double),
                ("kernel_launches", C.c_uint32), ("batches", C.c_uint32),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("clusters", C.c_uint64), ("frames", C.c_uint64),
                ("nodes", C.c_uint64), ("gpus_used", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class rt_kernel_info(C.Structure):
    _fields_ = [("registers", C.c_int32), ("local_bytes", C.c_int32), ("smem_bytes", C.c_uint32), ("grid", C.c_uint32),
                ("block", C.c_uint32), ("ctas_per_sm", C.c_uint32), ("smem_mask", C.c_uint32), ("bvh_nodes", C.c_uint32),
                ("bvh_leaves", C.c_uint32), ("bvh_depth", C.c_uint32), ("pool_slots", C.c_uint32), ("name", C.c_char * 96)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["name"] = d["name"].decode()
        return d


class rt_scene_edit(C.Structure):
    _fields_ = [("camera", C.POINTER(rt_camera)), ("seed", C.POINTER(C.c_uint64)), ("spheres", C.POINTER(rt_sphere)), ("n_spheres", C.c_uint64)]


assert C.sizeof(rt_sphere) == 64

# every symbol include/rtb200.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "rtb200_abi_version", "rtb200_last_error", "rtb200_camera_from_params", "rtb200_shard_rows",
    "rtb200_render_rgb8", "rtb200_render_linear_f32", "rtb200_scene_upload", "rtb200_render_device",
    "rtb200_scene_release", "rtb200_probe_sphere_hit", "rtb200_probe_refract", "rtb200_probe_reflectance",
    "rtb200_probe_sky", "rtb200_probe_get_ray", "rtb200_probe_rng", "rtb200_probe_quantise",
    "rtb200_decode_jpeg_file", "rtb200_free", "rtb200_render_device_async", "rtb200_render_device_wait",
    "rtb200_debug_bvh", "rtb200_probe_sphere_uv", "rtb200_device_count", "rtb200_render_rgb8_multi", "rtb200_scene_kernel_info",
    "rtb200_scene_update", "rtb200_scene_debug_bvh",
]

_lib = None


def lib() -> C.CDLL:
    """Load librtb200.so (built in-tree by `make -C rust-raytracer_b200` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RtError(-2, f"{LIB_PATH} is missing: build it with `make -C rust-raytracer_b200` (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.rtb200_abi_version.restype = C.c_int
    L.rtb200_last_error.restype = C.c_char_p
    L.rtb200_camera_from_params.argtypes = [C.POINTER(rt_camera_params), C.POINTER(rt_camera)]
    L.rtb200_shard_rows.restype = C.c_uint32
    L.rtb200_shard_rows.argtypes = [C.c_uint32, C.c_int32, C.c_int32, C.c_uint32]
    L.rtb200_render_rgb8.argtypes = [C.POINTER(rt_scene), C.POINTER(rt_options), C.c_void_p, C.POINTER(rt_stats)]
    L.rtb200_render_linear_f32.argtypes = [C.POINTER(rt_scene), C.POINTER(rt_options), C.c_void_p, C.POINTER(rt_stats)]
    L.rtb200_scene_upload.argtypes = [C.POINTER(rt_scene), C.POINTER(rt_options), C.POINTER(C.c_void_p)]
    L.rtb200_render_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
    L.rtb200_scene_release.argtypes = [C.c_void_p]
    L.rtb200_render_device_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.rtb200_render_device_wait.argtypes = [C.c_void_p, C.POINTER(rt_stats)]
    L.rtb200_probe_sphere_hit.argtypes = [C.POINTER(rt_vec3), C.c_double, C.POINTER(rt_vec3), C.POINTER(rt_vec3), C.c_double,
                                          C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(rt_vec3),
                                          C.POINTER(rt_vec3), C.POINTER(C.c_int32)]
    L.rtb200_probe_refract.argtypes = [C.POINTER(rt_vec3), C.POINTER(rt_vec3), C.c_double, C.POINTER(rt_vec3)]
    L.rtb200_probe_reflectance.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_double)]
    L.rtb200_probe_sky.argtypes = [C.POINTER(rt_vec3), C.c_uint32, C.POINTER(C.c_float)]
    L.rtb200_probe_get_ray.argtypes = [C.POINTER(rt_camera), C.c_double, C.c_double, C.POINTER(rt_vec3), C.POINTER(rt_vec3)]
    L.rtb200_probe_rng.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_double)]
    L.rtb200_probe_quantise.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    L.rtb200_decode_jpeg_file.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.rtb200_free.argtypes = [C.c_void_p]
    L.rtb200_free.restype = None
    L.rtb200_debug_bvh.argtypes = [C.POINTER(rt_scene), C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.c_void_p, C.c_uint64,
                                   C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    L.rtb200_probe_sphere_uv.argtypes = [C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_double)]
    L.rtb200_device_count.restype = C.c_int
    L.rtb200_render_rgb8_multi.argtypes = [C.POINTER(rt_scene), C.POINTER(rt_options), C.c_int32, C.c_void_p, C.POINTER(rt_stats)]
    L.rtb200_scene_kernel_info.argtypes = [C.c_void_p, C.POINTER(rt_kernel_info)]
    L.rtb200_scene_update.argtypes = [C.c_void_p, C.POINTER(rt_scene_edit)]
    L.rtb200_scene_debug_bvh.argtypes = [C.c_void_p] + L.rtb200_debug_bvh.argtypes[1:]
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise RtError(rc, (lib().rtb200_last_error() or b"").decode("utf-8", "replace"))


def vec3(v) -> rt_vec3:
    if isinstance(v, dict):
        return rt_vec3(float(v["x"]), float(v["y"]), float(v["z"]))
    return rt_vec3(float(v[0]), float(v[1]), float(v[2]))


_camera_backend = None   # bench.py's CPU reference arm installs the oracle's Camera::new here so that it never maps librtb200.so


def set_camera_backend(fn):
    """fn(rt_camera_params*, rt_camera*) -> int replacing rtb200_camera_from_params (None restores the library)."""
    global _camera_backend
    _camera_backend = fn


def camera_from_params(look_from, look_at, vup, vfov: float, aspect: float) -> rt_camera:
    """Camera::new (reference camera.rs:45-77), evaluated by the library's host code."""
    p = rt_camera_params(vec3(look_from), vec3(look_at), vec3(vup), float(vfov), float(aspect))
    out = rt_camera()
    if _camera_backend is not None:
        rc = _camera_backend(C.byref(p), C.byref(out))
        if rc != 0:
            raise RtError(rc, "camera backend failed")
        return out
    _check(lib().rtb200_camera_from_params(C.byref(p), C.byref(out)))
    return out


def shard_rows(height: int, rank: int, world: int, band_rows: int = 1) -> int:
    return int(lib().rtb200_shard_rows(height, rank, world, band_rows))


def shard_row_indices(height: int, rank: int, world: int, band_rows: int = 1) -> np.ndarray:
    y = np.arange(height)
    return y[((y // max(band_rows, 1)) % max(world, 1)) == rank]


def _decode_jpeg(path: str) -> np.ndarray:
    """load_texture_image (reference materials.rs:213-219): the library's own baseline JPEG decoder, so the Python host
    and the C++ CLI stage identical texels."""
    buf = C.c_void_p(); w = C.c_uint64(); h = C.c_uint64()
    rc = lib().rtb200_decode_jpeg_file(os.fsencode(path), C.byref(buf), C.byref(w), C.byref(h))
    if rc != 0:
        raise RtError(rc, f"cannot decode JPEG {path}")
    try:
        arr = np.ctypeslib.as_array(C.cast(buf, C.POINTER(C.c_uint8)), shape=(h.value, w.value, 3)).copy()
    finally:
        lib().rtb200_free(buf)
    return arr


class Scene:
    """Parsed scene = the reference's ``Config`` (config.rs:66-75), flattened into an ``rt_scene``.

    Keeps every buffer the C struct points into alive. Mutating ``width/height/samples_per_pixel/max_depth``
    mirrors how the reference's own tests override a parsed Config (raytracer.rs:272-273, 281-282); call
    :meth:`set_camera` when the aspect ratio changes (aspect is a camera field, camera.rs:26,54).
    """

    def __init__(self):
        self.c = rt_scene()
        self.c.seed = DEFAULT_SEED
        self._spheres = None
        self._tex_arrays: list[np.ndarray] = []
        self._tex_structs = None
        self._sky_array = None
        self.camera_params: Optional[dict] = None
        self.source = None

    # -- construction ---------------------------------------------------------------------------------
    @staticmethod
    def from_config(cfg: dict, base_dir: str = ".", textures: bool = True) -> "Scene":
        sc = Scene()
        sc.source = cfg
        sc.c.width = int(cfg["width"]); sc.c.height = int(cfg["height"])
        sc.c.samples_per_pixel = int(cfg["samples_per_pixel"]); sc.c.max_depth = int(cfg["max_depth"])
        cam = cfg["camera"]
        sc.camera_params = dict(look_from=cam["look_from"], look_at=cam["look_at"], vup=cam["vup"], vfov=cam["vfov"], aspect=cam["aspect"])
        sc.c.camera = camera_from_params(cam["look_from"], cam["look_at"], cam["vup"], cam["vfov"], cam["aspect"])
        # sky: missing/null -> None (black); {"texture": ""} -> gradient; path -> equirect texture (config.rs:49-64, raytracer.rs:137-161)
        sky = cfg.get("sky", None)
        sc.c.sky.mode = RT_SKY_NONE
        if sky is not None:
            tex = sky.get("texture", "")
            if tex in ("", None):
                sc.c.sky.mode = RT_SKY_GRADIENT
            else:
                arr = _decode_jpeg(os.path.join(base_dir, tex))
                sc._sky_array = arr
                sc.c.sky.mode = RT_SKY_TEXTURE
                sc.c.sky.tex = rt_image(arr.ctypes.data, arr.shape[1], arr.shape[0], arr.size)
        objs = cfg.get("objects", [])
        arr_t = rt_sphere * max(len(objs), 1)
        sc._spheres = arr_t()
        tex_structs = []
        for i, o in enumerate(objs):
            s = sc._spheres[i]
            s.center = vec3(o["center"]); s.radius = float(o["radius"]); s.texture = -1
            (kind, body), = o["material"].items()   # externally tagged enum (materials.rs:35-42)
            if kind == "Lambertian":
                s.kind = RT_LAMBERTIAN; s.albedo[:] = [np.float32(a) for a in body["albedo"]]
            elif kind == "Metal":
                s.kind = RT_METAL; s.albedo[:] = [np.float32(a) for a in body["albedo"]]; s.param = float(body["fuzz"])
            elif kind == "Glass":
                s.kind = RT_GLASS; s.param = float(body["index_of_refraction"])
            elif kind == "Texture":
                s.kind = RT_TEXTURE; s.albedo[:] = [np.float32(a) for a in body["albedo"]]; s.param = float(body["h_offset"])
                if not textures:
                    raise ValueError("texture material but textures=False")
                arr = _decode_jpeg(os.path.join(base_dir, body["pixels"]))
                w, h = int(body["width"]), int(body["height"])   # JSON dims, not the file's (materials.rs:208-209)
                if w * h * 3 > arr.size:
                    raise ValueError(f"texture {body['pixels']}: JSON says {w}x{h} but the file holds {arr.shape[1]}x{arr.shape[0]}")
                sc._tex_arrays.append(arr)
                tex_structs.append(rt_image(arr.ctypes.data, w, h, arr.size))
                s.texture = len(tex_structs) - 1
            elif kind == "Light":
                s.kind = RT_LIGHT
            else:
                raise ValueError(f"unknown material {kind}")
        sc.c.spheres = C.cast(sc._spheres, C.POINTER(rt_sphere)); sc.c.n_spheres = len(objs)
        if tex_structs:
            sc._tex_structs = (rt_image * len(tex_structs))(*tex_structs)
            sc.c.textures = C.cast(sc._tex_structs, C.POINTER(rt_image))
        sc.c.n_textures = len(tex_structs)
        return sc

    def set_camera(self, **kw):
        self.camera_params.update(kw)
        p = self.camera_params
        self.c.camera = camera_from_params(p["look_from"], p["look_at"], p["vup"], p["vfov"], p["aspect"])

    def resize(self, width: int, height: int, spp: Optional[int] = None, max_depth: Optional[int] = None, fix_aspect: bool = False):
        self.c.width, self.c.height = int(width), int(height)
        if spp is not None:
            self.c.samples_per_pixel = int(spp)
        if max_depth is not None:
            self.c.max_depth = int(max_depth)
        if fix_aspect:
            self.set_camera(aspect=float(width) / float(height))
        return self

    @property
    def n_spheres(self):
        return int(self.c.n_spheres)

    @property
    def seed(self):
        return int(self.c.seed)

    @seed.setter
    def seed(self, v):
        self.c.seed = int(v)


def read_config(path: str) -> dict:
    """Parse a scene file (plain JSON, or the gzip-compressed copies under scenes/)."""
    if path.endswith(".gz"):
        import gzip

        with gzip.open(path, "rb") as f:
            return json.loads(f.read())
    with open(path, "rb") as f:
        return json.loads(f.read())


def load_scene(path: str, base_dir: Optional[str] = None) -> Scene:
    """serde_json::from_slice::<Config> (reference main.rs:14-15). Texture paths resolve against ``base_dir``
    (the reference resolves them against the process CWD, materials.rs:214)."""
    cfg = read_config(path)
    if base_dir is None:
        base_dir = os.path.dirname(os.path.abspath(path))   # scenes say "data/earth.jpg"
        if not os.path.isdir(os.path.join(base_dir, "data")):
            base_dir = os.path.dirname(base_dir)
    return Scene.from_config(cfg, base_dir)


def bvh_records(scene: "Scene") -> dict:
    """Host-side diagnostic: the hierarchy the closest-hit stage traverses (no GPU needed). See rtb200_debug_bvh."""
    return _bvh_dict(lambda *a: lib().rtb200_debug_bvh(C.byref(scene.c), *a), scene.n_spheres)


def _bvh_dict(debug_bvh, n: int) -> dict:
    """Calls debug_bvh(recentre, info, nodes, cap, leaf_rec, cap, leaf_id, cap, always, cap, flat, cap) twice (sizes, then arrays)."""
    g = (C.c_double * 3)(); info = (C.c_uint32 * 8)()
    _check(debug_bvh(g, info, None, 0, None, 0, None, 0, None, 0, None, 0))
    n_nodes, n_leaves, depth, k, n_always, fpn, n_pairs, _ = (int(x) for x in info)
    nodes = np.zeros(max(n_nodes * fpn, 1), np.float32); rec = np.zeros(max(n_leaves * k * 4, 1), np.float32)
    ids = np.zeros(max(n_leaves * k, 1), np.uint32); always = np.zeros(max(n_always, 1), np.uint32); flat = np.zeros(max(n_pairs * 8, 1), np.float32)
    _check(debug_bvh(g, info, nodes.ctypes.data, nodes.size, rec.ctypes.data, rec.size, ids.ctypes.data, ids.size,
                     always.ctypes.data, always.size, flat.ctypes.data, flat.size))
    nd = nodes[: n_nodes * fpn].reshape(n_nodes, fpn)
    return {"n_nodes": n_nodes, "n_leaves": n_leaves, "depth": depth, "leaf_size": k, "recentre": np.array(g[:]), "n": n,
            "lo": nd[:, :24].reshape(n_nodes, 3, 8), "hi": nd[:, 24:48].reshape(n_nodes, 3, 8), "child": nd[:, 48:56].view(np.uint32),
            "leaf_rec": rec[: n_leaves * k * 4].reshape(n_leaves, k // 2, 2, 4), "leaf_id": ids[: n_leaves * k].reshape(n_leaves, k),
            "always": always[:n_always], "flat": flat[: n_pairs * 8].reshape(n_pairs, 2, 4)}


def make_options(device: int = -1, rank: int = 0, world: int = 1, band_rows: int = 1, variant: int = RT_VARIANT_AUTO,
                 sample_buffer_bytes: int = 0) -> rt_options:
    return rt_options(device, rank, world, band_rows, variant, 0, sample_buffer_bytes)


def render_rgb8(scene: Scene, opts: Optional[rt_options] = None, out: Optional[np.ndarray] = None):
    """Host in, host out: the replacement of reference raytracer.rs:259-263. Returns (uint8 [rows,w,3], stats dict)."""
    rows = scene.c.height if (opts is None or opts.world <= 1) else shard_rows(scene.c.height, opts.rank, opts.world, opts.band_rows)
    if out is None:
        out = np.empty((rows, scene.c.width, 3), dtype=np.uint8)
    st = rt_stats()
    _check(lib().rtb200_render_rgb8(C.byref(scene.c), C.byref(opts) if opts is not None else None, out.ctypes.data, C.byref(st)))
    return out, st.as_dict()


def render_linear(scene: Scene, opts: Optional[rt_options] = None):
    """Per-pixel mean radiance before sqrt/quantisation (float32 [rows,w,3]) and stats."""
    rows = scene.c.height if (opts is None or opts.world <= 1) else shard_rows(scene.c.height, opts.rank, opts.world, opts.band_rows)
    out = np.empty((rows, scene.c.width, 3), dtype=np.float32)
    st = rt_stats()
    _check(lib().rtb200_render_linear_f32(C.byref(scene.c), C.byref(opts) if opts is not None else None, out.ctypes.data, C.byref(st)))
    return out, st.as_dict()


def device_count() -> int:
    return int(lib().rtb200_device_count())


def render_rgb8_multi(scene: Scene, n_gpus: int = 0, opts: Optional[rt_options] = None, out: Optional[np.ndarray] = None):
    """One process, n_gpus devices (0 = all): rtb200_render_rgb8_multi. Returns (uint8 [h,w,3], stats dict)."""
    if out is None:
        out = np.empty((scene.c.height, scene.c.width, 3), dtype=np.uint8)
    st = rt_stats()
    _check(lib().rtb200_render_rgb8_multi(C.byref(scene.c), C.byref(opts) if opts is not None else None, int(n_gpus), out.ctypes.data, C.byref(st)))
    return out, st.as_dict()


class ResidentScene:
    """Scene kept in HBM between frames (rtb200_scene_upload / rtb200_render_device)."""

    def __init__(self, scene: Scene, opts: Optional[rt_options] = None):
        self.scene = scene
        self.opts = opts
        self.h = C.c_void_p()
        _check(lib().rtb200_scene_upload(C.byref(scene.c), C.byref(opts) if opts is not None else None, C.byref(self.h)))
        self.rows = scene.c.height if (opts is None or opts.world <= 1) else shard_rows(scene.c.height, opts.rank, opts.world, opts.band_rows)

    def render(self, dev_rgb8_ptr: int = 0, dev_linear_ptr: int = 0, stream: int = 0) -> dict:
        st = rt_stats()
        _check(lib().rtb200_render_device(self.h, C.c_void_p(dev_rgb8_ptr or None), C.c_void_p(dev_linear_ptr or None),
                                          C.c_void_p(stream or None), C.byref(st)))
        return st.as_dict()

    def render_async(self, dev_rgb8_ptr: int = 0, dev_linear_ptr: int = 0, stream: int = 0):
        """Enqueue a frame without waiting (frame loops); pair with :meth:`wait`."""
        _check(lib().rtb200_render_device_async(self.h, C.c_void_p(dev_rgb8_ptr or None), C.c_void_p(dev_linear_ptr or None), C.c_void_p(stream or None)))

    def wait(self) -> dict:
        st = rt_stats()
        _check(lib().rtb200_render_device_wait(self.h, C.byref(st)))
        return st.as_dict()

    def update(self, spheres=None, camera: Optional[rt_camera] = None, seed: Optional[int] = None):
        """rtb200_scene_update: edit the resident scene for the next frames (None keeps a field). `spheres` is a
        :class:`Scene` (its sphere list) or a ctypes ``rt_sphere`` array with the uploaded count, in the same order."""
        e = rt_scene_edit()
        if spheres is not None:
            if isinstance(spheres, Scene):
                e.spheres, e.n_spheres = spheres.c.spheres, spheres.c.n_spheres
            else:
                e.spheres, e.n_spheres = C.cast(spheres, C.POINTER(rt_sphere)), len(spheres)
        if camera is not None:
            e.camera = C.pointer(camera)
        if seed is not None:
            e.seed = C.pointer(C.c_uint64(int(seed)))
        _check(lib().rtb200_scene_update(self.h, C.byref(e)))

    def bvh_records(self) -> dict:
        """What the closest-hit stage of this handle reads now (after any update), copied back from the device;
        the dict of :func:`bvh_records`. ``flat`` is empty unless the handle renders RT_VARIANT_BRUTE_FORCE."""
        return _bvh_dict(lambda *a: lib().rtb200_scene_debug_bvh(self.h, *a), int(self.scene.c.n_spheres))

    def kernel_info(self) -> dict:
        ki = rt_kernel_info()
        _check(lib().rtb200_scene_kernel_info(self.h, C.byref(ki)))
        return ki.as_dict()

    def release(self):
        if self.h:
            lib().rtb200_scene_release(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


def write_png(path: str, rgb8: np.ndarray):
    """write_image (reference raytracer.rs:33-42): RGB8 PNG."""
    from PIL import Image

    Image.fromarray(np.ascontiguousarray(rgb8, dtype=np.uint8), "RGB").save(path, format="PNG")


def render(filename: str, scene: Scene, opts: Optional[rt_options] = None) -> dict:
    """`pub fn render(filename, scene)` (reference raytracer.rs:250-266): render, print the frame time, write the PNG."""
    img, st = render_rgb8(scene, opts)
    print(f"Frame time: {int(st['wall_ms'])}ms")
    write_png(filename, img)
    return st
