"""Resident scene edits (rtb200_scene_update): camera, seed and sphere edits of an uploaded scene, with the 8-wide BVH refitted
on the device (rtb200_refit.cu).

CPU: a numpy restatement of the refit (same topology, records and node boxes recomputed from a sphere list with directed f32
rounding) reproduces the host builder bit for bit on the builder's own spheres, and keeps every moved sphere inside every
ancestor box. GPU: an edited handle renders exactly what a fresh upload of the edited scene renders, its device records equal
the restatement bit for bit, and refused edits leave the handle unchanged."""
import ctypes as C

import numpy as np
import pytest

import oracle_py as O
import rtb200 as R
from rtb200 import scenes
from synth import _v, mixed_config

f32 = np.float32
EMPTY, LEAF = 0xFFFFFFFF, 0x80000000
U = 2.0 ** -24


# ---- numpy restatement of the refit ----------------------------------------------------------------------------
def _f32_up(x):
    f = x.astype(f32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, f32(np.inf)), f).astype(f32)


def _f32_down(x):
    f = x.astype(f32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, f32(-np.inf)), f).astype(f32)


def _sphere_records(x, y, z, r2):
    """rtbvh::sphere_record for arrays: {x, y, z, nk} in f32, (0, 0, 0, +inf) for spheres outside the f32 frame."""
    c2 = (x * x + y * y) + z * z
    es = 96.0 * U * c2 + 16.0 * U * r2 + 1e-30
    nkd = -(c2 - r2) + es
    rec = np.stack([x.astype(f32), y.astype(f32), z.astype(f32), np.where(np.isfinite(nkd), _f32_up(nkd), f32(np.inf))], axis=1).astype(f32)
    ok = np.isfinite(rec[:, :3]).all(axis=1) & np.isfinite(nkd) & (c2 < 1e30)
    rec[~ok] = [0.0, 0.0, 0.0, np.inf]
    return rec


def _put(pairs, slot, rec):
    """Pair-packed layout {x0,x1,y0,y1},{z0,z1,nk0,nk1}: pairs[slot // 2] gets rec in lane slot & 1."""
    p, k = slot // 2, slot & 1
    pairs[p, 0, k], pairs[p, 0, 2 + k], pairs[p, 1, k], pairs[p, 1, 2 + k] = rec


def _arrays(spheres):
    c = np.array([[s.center.x, s.center.y, s.center.z] for s in spheres], np.float64).reshape(-1, 3)
    r = np.array([s.radius for s in spheres], np.float64)
    return c, r


def refit(b, spheres):
    """The records of topology `b` (a bvh_records dict) for `spheres`: leaf records, flat records and node boxes."""
    c, r = _arrays(spheres)
    g = b["recentre"]
    with np.errstate(all="ignore"):
        cr = c - g
        rec = _sphere_records(cr[:, 0], cr[:, 1], cr[:, 2], r * r)
        out = {k: b[k].copy() for k in ("lo", "hi", "leaf_rec", "flat")}
        for i in range(len(spheres)):
            _put(out["flat"], i, rec[i])
        for leaf in range(b["n_leaves"]):
            for j, i in enumerate(b["leaf_id"][leaf]):
                if i != EMPTY:
                    _put(out["leaf_rec"][leaf], j, rec[i])
        ra = np.abs(r)
        box = np.empty((b["n_nodes"], 8, 2, 3))
        box[:, :, 0], box[:, :, 1] = np.inf, -np.inf
        for node in reversed(range(b["n_nodes"])):          # depth-first emission: children after their parent
            for k, ref in enumerate(b["child"][node]):
                if ref == EMPTY:
                    continue
                if ref & LEAF:
                    ids = b["leaf_id"][int(ref & 0x7FFFFFFF)]
                    ids = ids[ids != EMPTY]
                    lo, hi = (cr[ids] - ra[ids, None]).min(axis=0), (cr[ids] + ra[ids, None]).max(axis=0)
                else:
                    lo, hi = box[int(ref), :, 0].min(axis=0), box[int(ref), :, 1].max(axis=0)
                box[node, k] = lo, hi
                m = 32.0 * U * max(np.abs(lo).max(), np.abs(hi).max()) + 1e-30
                out["lo"][node, :, k], out["hi"][node, :, k] = _f32_down(lo - m), _f32_up(hi + m)
    return out


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _assert_records_equal(got, want, keys=("lo", "hi", "leaf_rec", "flat")):
    for k in keys:
        assert got[k].shape == want[k].shape, k
        assert np.array_equal(_bits(got[k]), _bits(want[k])), k


def _move(spheres, rng, scale=0.3, skip=()):
    """A random motion of every sphere (centre, radius, sign of the radius) except those in `skip`."""
    for i, s in enumerate(spheres):
        if i in skip:
            continue
        s.center.x += float(rng.normal(0, scale)); s.center.y += float(rng.normal(0, scale)); s.center.z += float(rng.normal(0, scale))
        s.radius *= float(rng.uniform(0.5, 1.5)) * (-1.0 if rng.uniform() < 0.05 else 1.0)


def _copy(sc):
    arr = (R.rt_sphere * max(sc.n_spheres, 1))()
    C.memmove(arr, sc.c.spheres, sc.n_spheres * C.sizeof(R.rt_sphere))
    return arr[: sc.n_spheres]


def _rtiow_10k():
    return R.Scene.from_config(scenes._variant(scenes.rtiow_config(50), 32, 24, 1, 4))


CPU_SCENES = {
    "cover": lambda: scenes.cover_scene(64, 48, 1),
    "mixed": lambda: R.Scene.from_config(mixed_config(32, 24, 1, 4, seed=3, n=90)),
    "rtiow10k_breadth_first": _rtiow_10k,
}


@pytest.mark.parametrize("name", sorted(CPU_SCENES))
def test_restatement_reproduces_the_host_builder(name, monkeypatch):
    """Applied to the builder's own spheres, the refit gives the builder's bits (pins the restatement to rtb200_bvh.hpp)."""
    if name == "rtiow10k_breadth_first":
        monkeypatch.setenv("RTB200_BVH_AREA_LEVELS", "2")   # wide levels >= 2 take the breadth-first collapse
    sc = CPU_SCENES[name]()
    b = R.bvh_records(sc)
    if name == "rtiow10k_breadth_first":
        assert b["depth"] >= 3
    _assert_records_equal(refit(b, _copy(sc)), b)


def _subtree(b, ref, out):
    if ref & LEAF:
        ids = b["leaf_id"][int(ref & 0x7FFFFFFF)]
        out.extend(ids[ids != EMPTY].tolist())
        return
    for r in b["child"][int(ref)]:
        if r != EMPTY:
            _subtree(b, int(r), out)


@pytest.mark.parametrize("seed,scale", [(1, 0.05), (2, 0.5), (3, 5.0)])
def test_refit_boxes_hold_the_moved_spheres(seed, scale):
    """Property of the refit on random motions: every sphere's exact box lies inside every ancestor slot's f32 box."""
    sc = R.Scene.from_config(mixed_config(32, 24, 1, 4, seed=seed, n=120))
    b = R.bvh_records(sc)
    sp = _copy(sc)
    _move(sp, np.random.default_rng(seed), scale)
    out = refit(b, sp)
    c, r = _arrays(sp)
    cr, ra = c - b["recentre"], np.abs(r)
    for node in range(b["n_nodes"]):
        for k, ref in enumerate(b["child"][node]):
            if ref == EMPTY:
                continue
            mem = []
            _subtree(b, int(ref), mem)
            lo, hi = out["lo"][node][:, k].astype(np.float64), out["hi"][node][:, k].astype(np.float64)
            assert np.all(lo <= (cr[mem] - ra[mem, None]).min(axis=0)) and np.all(hi >= (cr[mem] + ra[mem, None]).max(axis=0))


# ---- GPU: edited handle == fresh upload of the edited scene -------------------------------------------------------
def _frame(rs, sc):
    import torch
    n = rs.rows * sc.c.width * 3
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    lin = torch.zeros(n, dtype=torch.float32, device="cuda")
    st = rs.render(out.data_ptr(), lin.data_ptr())
    torch.cuda.synchronize()
    return lin.cpu().numpy().reshape(rs.rows, -1, 3), out.cpu().numpy().reshape(rs.rows, -1, 3), st


def _assert_fresh(rs, sc, opts=None, oracle=True):
    """The handle's frame equals a fresh render of `sc` (and the oracle's frame) bit for bit, ray count included."""
    lin, img, st = _frame(rs, sc)
    img_f, st_f = R.render_rgb8(sc, opts)
    lin_f, _ = R.render_linear(sc, opts)
    assert np.array_equal(img, img_f) and np.array_equal(lin, lin_f) and st["rays"] == st_f["rays"]
    if oracle:
        lin_o, img_o, st_o = O.render(sc)
        rows = R.shard_row_indices(sc.c.height, opts.rank, opts.world, opts.band_rows) if opts is not None and opts.world > 1 else slice(None)
        assert np.array_equal(lin, lin_o[rows]) and np.array_equal(img, img_o[rows])
        if opts is None or opts.world == 1:
            assert st["rays"] == st_o["rays"]
    return img


def _light_cfg(n_lights, seed):
    cfg = mixed_config(48, 36, 3, 6, seed=seed, n=30)
    pos = [(0.0, 6.0, 0.0), (-4.0, 3.0, 5.0)]
    for k in range(n_lights):
        cfg["objects"].insert(3 + 5 * k, {"center": _v(*pos[k]), "radius": 1.0 + 0.5 * k, "material": {"Light": {}}})
    return cfg


def _always_cfg():
    cfg = mixed_config(48, 36, 2, 6, seed=5, n=12)
    cfg["objects"].insert(4, {"center": _v(-2e15 - 8.0, 0, 0), "radius": 2e15, "material": {"Lambertian": {"albedo": [0.3, 0.6, 0.9]}}})
    cfg["objects"].insert(7, {"center": _v(float("inf"), 0, 0), "radius": 1.0, "material": {"Metal": {"albedo": [0.9, 0.9, 0.9], "fuzz": 0.0}}})
    return cfg


def _rematerialise(sc, rng):
    """Move, resize and re-materialise the spheres of `sc` in place (Lights stay Lights and may move)."""
    sp = sc._spheres
    _move(sp[: sc.n_spheres], rng, 0.3, skip=(0,))
    for i in range(1, sc.n_spheres):
        s = sp[i]
        if s.kind in (R.RT_LIGHT, R.RT_TEXTURE) or rng.uniform() > 0.3:
            continue
        s.kind = int(rng.choice([R.RT_LAMBERTIAN, R.RT_METAL, R.RT_GLASS]))
        s.albedo[:] = [float(f32(a)) for a in rng.uniform(0.1, 0.9, 3)]
        s.param = 1.5 if s.kind == R.RT_GLASS else float(rng.uniform(0, 0.5))


def _cover():
    return scenes.cover_scene(48, 36, 2, 8)


def _test_scene():
    return R.Scene.from_config(scenes._variant(scenes.test_scene_config(), 64, 48, 3, 8), scenes.SCENES_DIR)


def _edit_textures(sc, rng):
    _rematerialise(sc, rng)
    tex = [i for i in range(sc.n_spheres) if sc._spheres[i].kind == R.RT_TEXTURE]
    assert tex and sc.c.n_textures >= 2
    for i in tex:
        s = sc._spheres[i]
        s.param += 0.25                                   # h_offset
        s.texture = (s.texture + 1) % int(sc.c.n_textures)


GPU_CASES = {
    "cover": (_cover, _rematerialise, None),
    "lights1": (lambda: R.Scene.from_config(_light_cfg(1, 21)), _rematerialise, None),
    "lights2": (lambda: R.Scene.from_config(_light_cfg(2, 23)), _rematerialise, None),
    "textured": (_test_scene, _edit_textures, None),
    "always_list": (lambda: R.Scene.from_config(_always_cfg()), _rematerialise, None),
    "brute_force": (_cover, _rematerialise, lambda: R.make_options(variant=R.RT_VARIANT_BRUTE_FORCE)),
    "exact_f64": (_cover, _rematerialise, lambda: R.make_options(variant=R.RT_VARIANT_EXACT_F64)),
    "shard_1_of_2": (_cover, _rematerialise, lambda: R.make_options(rank=1, world=2, band_rows=4)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GPU_CASES))
def test_update_renders_the_edited_scene(name):
    mk, edit, mk_opts = GPU_CASES[name]
    opts = mk_opts() if mk_opts else None
    s0, s1 = mk(), mk()
    edit(s1, np.random.default_rng(11))
    if name == "always_list":
        s1._spheres[4].center.x -= 1e14; s1._spheres[7].center.y = float("nan")   # always-list spheres may take any valid value
    rs = R.ResidentScene(s0, opts)
    _assert_fresh(rs, s0, opts, oracle=False)
    rs.update(spheres=s1)
    _assert_fresh(rs, s1, opts)
    b0 = R.bvh_records(s0)
    got = rs.bvh_records()
    # device records == the restatement: the hierarchy (tree variant) or the flat records (brute force); exact f64 has neither
    keys = {"brute_force": ("flat",), "exact_f64": ()}.get(name, ("lo", "hi", "leaf_rec"))
    if name in ("brute_force", "exact_f64"):
        assert got["n_nodes"] == 0 and got["n_leaves"] == 0 and len(got["flat"]) == (len(b0["flat"]) if name == "brute_force" else 0)
    else:
        assert len(got["flat"]) == 0
        assert np.array_equal(got["child"], b0["child"]) and np.array_equal(got["leaf_id"], b0["leaf_id"]) and np.array_equal(got["always"], b0["always"])
    _assert_records_equal(got, refit(b0, _copy(s1)), keys)
    rs.update(spheres=s0)                                  # back to the upload's spheres: the upload's records, bit for bit
    _assert_records_equal(rs.bvh_records(), b0, keys)
    _assert_fresh(rs, s0, opts, oracle=False)
    rs.release()


@pytest.mark.gpu
def test_camera_and_seed_edits_and_a_short_animation_on_two_streams():
    import torch
    sc = _cover()
    rs = R.ResidentScene(sc)
    cam = R.camera_from_params([12, 3, 5], [0, 0.5, 0], [0, 1, 0], 25.0, 48 / 36)
    rs.update(camera=cam, seed=7)
    edited = _cover(); edited.c.camera = cam; edited.seed = 7
    _assert_fresh(rs, edited)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    n = sc.c.width * sc.c.height * 3
    outs = [torch.zeros(n, dtype=torch.uint8, device="cuda") for _ in range(2)]
    rng = np.random.default_rng(3)
    for f in range(5):                                    # orbiting camera, bobbing spheres, one frame each
        frame = _cover()
        for i in range(1, frame.n_spheres):
            frame._spheres[i].center.y += 0.2 * np.sin(0.7 * f + i)
        a = 0.3 * f
        frame.c.camera = R.camera_from_params([13 * np.cos(a), 2, 13 * np.sin(a)], [0, 0, 0], [0, 1, 0], 20.0, 48 / 36)
        frame.seed = 100 + f
        rs.update(spheres=frame, camera=frame.c.camera, seed=frame.seed)
        rs.render_async(outs[f & 1].data_ptr(), 0, streams[f & 1].cuda_stream)
        rs.wait()
        ref, _ = R.render_rgb8(frame)
        assert np.array_equal(outs[f & 1].cpu().numpy().reshape(ref.shape), ref), f
    rs.release()


@pytest.mark.gpu
def test_refused_edits_leave_the_handle_unchanged():
    import torch
    L = R.lib()
    sc = R.Scene.from_config(_light_cfg(1, 21))
    light = next(i for i in range(sc.n_spheres) if sc._spheres[i].kind == R.RT_LIGHT)
    rs = R.ResidentScene(sc)
    _, before, _ = _frame(rs, sc)

    def refused(code, spheres=None, **kw):
        with pytest.raises(R.RtError) as e:
            rs.update(spheres=spheres, **kw)
        assert e.value.code == code
        assert np.array_equal(_frame(rs, sc)[1], before)

    sp = _copy(sc)
    _move(sp, np.random.default_rng(1))                    # valid motion everywhere ...
    short = (R.rt_sphere * (sc.n_spheres - 1))(*sp[:-1])
    refused(-1, short)                                     # wrong count
    moved = (R.rt_sphere * sc.n_spheres)(*sp)
    moved[light].kind, moved[light + 1].kind = moved[light + 1].kind, R.RT_LIGHT
    refused(-4, moved)                                     # a Light at another index
    for bad in (1e16, float("nan")):
        far = (R.rt_sphere * sc.n_spheres)(*sp)
        far[sc.n_spheres - 1].center.x = bad              # ... but the last sphere leaves the f32 frame
        refused(-4, far)
    tex = (R.rt_sphere * sc.n_spheres)(*sp)
    tex[sc.n_spheres - 1].kind, tex[sc.n_spheres - 1].texture = R.RT_TEXTURE, 0   # the scene has no textures
    refused(-1, tex)
    out = torch.zeros(rs.rows * sc.c.width * 3, dtype=torch.uint8, device="cuda")
    rs.render_async(out.data_ptr(), 0, 0)
    with pytest.raises(R.RtError) as e:                   # frames in flight read the arrays
        rs.update(seed=9)
    assert e.value.code == -1
    rs.wait()
    assert L.rtb200_scene_update(None, C.byref(R.rt_scene_edit())) == -1
    assert L.rtb200_scene_update(rs.h, None) == -1
    assert np.array_equal(_frame(rs, sc)[1], before)
    rs.release()
