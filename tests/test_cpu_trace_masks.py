"""CPU tests of the filtered traversal of rtc_trace_closest_ex / rtc_trace_any_ex / rtc_trace_count_ex: instance visibility masks
and triangle face culling.

csrc/trace.cuh's FILTER variant is compiled for the host (tests/native/trace_host_ex.cpp th_trace_ex) and held against
  * the oracle's brute force with the same masks and flags (tests/native/oracle_masks.c over oracle/rt_oracle.c), bit for bit;
  * oracle/wide_bvh.inc's traversal with the two tests restated (tests/native/oracle_masks.c), counter for counter, under all
    three triangle schedules;
  * the geometric definition of facing: dot((v1 - v0) x (v2 - v0), d_obj) < 0 in double is front-facing;
  * the unfiltered traversal, when nothing is masked and nothing is culled.
It also checks the new exports and the refusals that need no device."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
from mask_oracle import MaskedScene, product_trace_ex, wide_trace_ex
from oracle import orc
from tweeker_raytracer_b200 import core, host

FLAG_SETS = [0, core.RAY_CULL_BACK_FACING, core.RAY_CULL_FRONT_FACING, core.RAY_CULL_BACK_FACING | core.RAY_CULL_FRONT_FACING]
NEW = ("rtc_scene_set_instance_masks", "rtc_trace_closest_ex", "rtc_trace_any_ex", "rtc_trace_count_ex")


def fuzz_scene(tmp_path, seed):
    """A scene of tests/test_gpu_fuzz.py (same generator and seeds as tests/test_cpu_trace_source.py) on the host: (app, export, oracle)."""
    from test_gpu_fuzz import random_scene
    rng = np.random.default_rng(1000 + seed)
    scene = os.path.join(str(tmp_path), "scene_fuzz.txt")
    random_scene(scene, rng)
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="32 32", samplesSqrt=1), scene, host_only=True)
    geos = [app.geometry(g) for g in range(app.info.numGeometries)]
    insts = [app.instance(i)[:2] for i in range(app.info.numInstances)]
    export, _ = core.host_scene_export(geos, insts)
    return app, export, MaskedScene(H.oracle_scene(app), len(insts))


def soup_scene(seed):
    """Unstructured soup with duplicates, repeated vertices and collinear triangles, instanced five times: identity, mirrored and
    non-uniformly scaled, uniformly scaled, far-translated, and mirrored in one axis only."""
    rng = np.random.default_rng(seed)
    n = 1200
    centre = rng.uniform(-3, 3, size=(n, 1, 3))
    size = np.exp(rng.uniform(np.log(1e-3), np.log(2.0), size=(n, 1, 1)))
    tris = (centre + size * rng.normal(size=(n, 3, 3))).astype(np.float32)
    tris[10:20] = tris[0:10]
    tris[20:30, 1] = tris[20:30, 0]
    tris[30:40, 2] = (tris[30:40, 0] + tris[30:40, 1]) * np.float32(0.5)
    verts = tris.reshape(-1, 3)
    idx = np.arange(3 * n, dtype=np.uint32).reshape(n, 3)
    transforms = [np.array(t, dtype=np.float32) for t in (
        [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0],
        [-0.7, 0.2, 0, 1.5, 0.1, 1.3, 0.3, -0.5, 0, -0.4, 0.6, 2.0],
        [2.5, 0, 0, -1, 0, 2.5, 0, 0.5, 0, 0, 2.5, 1],
        [1, 0, 0, 1000.0, 0, 1, 0, -2000.0, 0, 0, 1, 500.0],
        [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, -1, 0.25])]
    export, _ = core.host_scene_export([(verts, idx)], [(t, 0) for t in transforms])
    attrs = np.zeros(len(verts), dtype=orc.ATTR_DTYPE)
    attrs["vertex"] = verts
    ref = orc.Scene()
    ref.add_geometry(attrs, idx)
    for t in transforms:
        ref.add_instance(t, 0, 0)
    ref.commit()
    ref = MaskedScene(ref, len(transforms))
    rays = np.concatenate([H.random_rays(2500, seed=seed, lo=(-4, -4, -4), hi=(4, 4, 4)),
                           H.random_rays(500, seed=seed + 50, lo=(996, -2004, 496), hi=(1004, -1996, 504))])
    return export, ref, rays


def check_against_oracle(export, ref, rays, masks, rng, label):
    ref.set_instance_masks(0, masks)
    for flags in FLAG_SETS:
        ray_mask = int(rng.integers(0, 256))
        hits, counts, overflows = product_trace_ex(export, rays, masks, ray_mask, flags)
        assert overflows == 0
        want = ref.trace_closest_ex(rays, ray_mask, flags)
        assert H.hits_equal(hits, want), (label, flags, ray_mask)
        model_hits, model_counts = wide_trace_ex(export, rays, masks=masks, ray_mask=ray_mask, flags=flags)
        assert H.hits_equal(hits, model_hits) and counts == model_counts, (label, flags, ray_mask)
        occl, counts_any, _ = product_trace_ex(export, rays, masks, ray_mask, flags, any_hit=True)
        assert np.array_equal(occl["inst"] != 0xffffffff, ref.trace_any_ex(rays, ray_mask, flags).astype(bool)), (label, flags)
        assert counts_any == wide_trace_ex(export, rays, any_hit=True, masks=masks, ray_mask=ray_mask, flags=flags)[1], (label, flags)
        # the occluding candidate any-hit reports is a real, unmasked instance's hit
        found = occl["inst"] != 0xffffffff
        assert np.all(masks[occl["inst"][found]] & ray_mask)


@pytest.mark.parametrize("seed", list(range(8)))
def test_twin_equals_brute_force_on_fuzz_scenes(built, tmp_path, seed):
    app, export, ref = fuzz_scene(tmp_path, seed)
    rng = np.random.default_rng(seed)
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    rays = H.random_rays(4000, seed=seed, lo=(-5, 0.05, -5), hi=(5, 4, 5))
    check_against_oracle(export, ref, rays, masks, rng, "fuzz %d" % seed)
    app.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_twin_equals_brute_force_on_degenerate_soups(built, seed):
    export, ref, rays = soup_scene(seed)
    rng = np.random.default_rng(100 + seed)
    for _ in range(2):
        masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
        check_against_oracle(export, ref, rays, masks, rng, "soup %d" % seed)
    ref.close()


@pytest.mark.parametrize("seed", [0, 5])
def test_capped_schedules_change_no_hit_and_no_counter(built, tmp_path, seed):
    app, export, ref = fuzz_scene(tmp_path, seed)
    rng = np.random.default_rng(7 + seed)
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    rays = H.random_rays(3000, seed=seed, lo=(-5, 0.05, -5), hi=(5, 4, 5))
    for flags in FLAG_SETS:
        ray_mask = int(rng.integers(1, 256))
        for any_hit in (False, True):
            base = product_trace_ex(export, rays, masks, ray_mask, flags, any_hit=any_hit, cap=0)
            for cap in (1, 2):
                got = product_trace_ex(export, rays, masks, ray_mask, flags, any_hit=any_hit, cap=cap)
                assert H.hits_equal(got[0], base[0]) and got[1] == base[1], (flags, any_hit, cap)
    app.close()


def test_neutral_filter_equals_the_plain_traversal(built, tmp_path):
    app, export, ref = fuzz_scene(tmp_path, 3)
    rays = H.random_rays(6000, seed=3, lo=(-5, 0.05, -5), hi=(5, 4, 5))
    masks = np.full(len(export["instance_gas"]), 0xFF, dtype=np.uint8)
    # the restatement's neutral settings are the unchanged oracle: its brute force and its wide-BVH traversal
    assert H.hits_equal(ref.trace_closest_ex(rays[:2000]), ref.scene.trace_closest(rays[:2000], brute_force=True))
    assert np.array_equal(ref.trace_any_ex(rays[:2000]), ref.scene.trace_any(rays[:2000], brute_force=True))
    for any_hit in (False, True):
        model = orc.wide_trace(export, rays, any_hit=any_hit)
        model_ex = wide_trace_ex(export, rays, any_hit=any_hit)
        assert H.hits_equal(model[0], model_ex[0]) and model[1] == model_ex[1]
    for any_hit in (False, True):
        plain = H.product_trace(export, rays, any_hit=any_hit)
        for cap in (0, 1, 2):
            got = product_trace_ex(export, rays, masks, 0xFF, 0, any_hit=any_hit, cap=cap)
            assert H.hits_equal(got[0], plain[0]) and got[1] == plain[1], (any_hit, cap)
    # every instance masked out: nothing is entered, and the instance-level node visits are what they were
    none = product_trace_ex(export, rays, np.zeros_like(masks), 0xFF, 0)
    assert (none[0]["inst"] == 0xffffffff).all() and none[1][1] == 0 and none[1][2] == 0
    levels = orc.wide_trace(export, rays, levels=True)[1]
    assert none[1][0] == levels[3]
    # a ray mask of 0 sees nothing either
    assert (product_trace_ex(export, rays, masks, 0, 0)[0]["inst"] == 0xffffffff).all()
    app.close()


def facing_cases(seed, n=400):
    """Well-conditioned triangles hit by rays of every direction octant: (verts [n, 3, 3] f4, rays) per case, ray i aims at
    triangle i's centroid."""
    rng = np.random.default_rng(seed)
    centre = rng.uniform(-60, 60, size=(n, 1, 3))
    tris = (centre + rng.uniform(-1, 1, size=(n, 3, 3))).astype(np.float32)
    octant = np.arange(n) % 8
    d = np.abs(rng.normal(size=(n, 3))) + 0.05
    d[:, 0] *= np.where(octant & 4, -1, 1); d[:, 1] *= np.where(octant & 2, -1, 1); d[:, 2] *= np.where(octant & 1, -1, 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return tris, d


def test_det_sign_is_the_geometric_facing(built):
    """The kernels' rule (det > 0 is front-facing) against dot((v1 - v0) x (v2 - v0), d_obj) < 0 in double, for every direction
    octant and for identity, rotated-and-scaled and mirrored instances; triangles at grazing angles (|cos| < 0.05) are left out."""
    transforms = {"identity": [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0],
                  "rotated": [0.0, -2.0, 0.0, 0.3, 1.5, 0.0, 0.0, -0.2, 0.0, 0.0, 0.7, 0.1],
                  "mirrored": [-1.2, 0.1, 0.0, 0.0, 0.0, 0.9, 0.2, 0.4, 0.1, 0.0, 1.1, -0.3]}
    checked = 0
    for k, (name, t) in enumerate(transforms.items()):
        t = np.array(t, dtype=np.float32)
        m = t.reshape(3, 4).astype(np.float64)
        tris, d_world = facing_cases(k)
        verts = tris.reshape(-1, 3)
        idx = np.arange(len(verts), dtype=np.uint32).reshape(-1, 3)
        export, _ = core.host_scene_export([(verts, idx)], [(t, 0)])
        attrs = np.zeros(len(verts), dtype=orc.ATTR_DTYPE)
        attrs["vertex"] = verts
        ref = orc.Scene()
        ref.add_geometry(attrs, idx)
        ref.add_instance(t, 0, 0)
        ref.commit()
        ref = MaskedScene(ref, 1)
        centroid_world = (m[:, :3] @ tris.astype(np.float64).mean(axis=1).T).T + m[:, 3]
        rays = np.zeros(len(tris), dtype=orc.RAY_DTYPE)
        o = centroid_world - 6.0 * d_world
        rays["ox"], rays["oy"], rays["oz"] = o[:, 0], o[:, 1], o[:, 2]
        rays["dx"], rays["dy"], rays["dz"] = d_world[:, 0], d_world[:, 1], d_world[:, 2]
        rays["tmin"], rays["tmax"] = 1e-4, 1e30
        e1 = tris[:, 1].astype(np.float64) - tris[:, 0]
        e2 = tris[:, 2].astype(np.float64) - tris[:, 0]
        nrm = np.cross(e1, e2)
        d_obj = np.linalg.solve(m[:, :3], d_world.T).T
        dot = np.einsum("ij,ij->i", nrm, d_obj)
        cos = dot / (np.linalg.norm(nrm, axis=1) * np.linalg.norm(d_obj, axis=1))
        masks = np.array([0xFF], dtype=np.uint8)
        hit = product_trace_ex(export, rays, masks)[0]["inst"] != 0xffffffff
        kept_back = product_trace_ex(export, rays, masks, flags=core.RAY_CULL_BACK_FACING)[0]
        kept_front = product_trace_ex(export, rays, masks, flags=core.RAY_CULL_FRONT_FACING)[0]
        # the rays aim at one triangle each but may hit others first: judge facing on the triangle the unculled query hits
        plain = product_trace_ex(export, rays, masks)[0]
        own = hit & (plain["prim"] == np.arange(len(rays))) & (np.abs(cos) > 0.05)
        assert own.sum() > 200, name
        front_by_det = kept_back["prim"] == np.arange(len(rays))
        back_by_det = kept_front["prim"] == np.arange(len(rays))
        assert np.array_equal(front_by_det[own], dot[own] < 0), name
        assert np.array_equal(back_by_det[own], dot[own] > 0), name
        # the oracle restates the kernels' det rule and, separately, the geometric rule: both agree with the twin here
        for flags in FLAG_SETS[1:]:
            twin = product_trace_ex(export, rays, masks, flags=flags)[0]
            assert H.hits_equal(twin, ref.trace_closest_ex(rays, 0xFF, flags)), (name, flags)
            assert np.array_equal((twin["inst"] != 0xffffffff)[own], (ref.trace_closest_ex(rays, 0xFF, flags, rule="normal")["inst"] != 0xffffffff)[own]), (name, flags)
        if name == "mirrored":
            assert np.linalg.det(m[:, :3]) < 0
        checked += int(own.sum())
        ref.close()
    assert checked > 800


def test_closed_mesh_culling(built):
    """A closed, outward-wound box seen from outside and from inside: culling back faces keeps exactly the near wall from
    outside and nothing from inside; culling front faces the reverse."""
    v = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float32)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]     # outward normals
    idx = np.array([[a, b, c] for (a, b, c, d) in quads] + [[a, c, d] for (a, b, c, d) in quads], dtype=np.uint32)
    nrm = np.cross(v[idx[:, 1]] - v[idx[:, 0]], v[idx[:, 2]] - v[idx[:, 0]])
    centroid = v[idx].mean(axis=1)
    assert (np.einsum("ij,ij->i", nrm, centroid) > 0).all()
    ident = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)
    export, _ = core.host_scene_export([(v, idx)], [(ident, 0)])
    masks = np.array([0xFF], dtype=np.uint8)
    outside = H.random_rays(1000, seed=1, lo=(-0.9,) * 3, hi=(0.9,) * 3)
    d = np.stack([outside["dx"], outside["dy"], outside["dz"]], axis=1)
    o = np.stack([outside["ox"], outside["oy"], outside["oz"]], axis=1) - 5.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
    outside["ox"], outside["oy"], outside["oz"] = o[:, 0], o[:, 1], o[:, 2]
    inside = H.random_rays(1000, seed=2, lo=(-0.9,) * 3, hi=(0.9,) * 3)
    plain_out = product_trace_ex(export, outside, masks)[0]
    plain_in = product_trace_ex(export, inside, masks)[0]
    assert (plain_out["inst"] == 0).all() and (plain_in["inst"] == 0).all()
    back_out = product_trace_ex(export, outside, masks, flags=core.RAY_CULL_BACK_FACING)[0]
    assert H.hits_equal(back_out, plain_out)                        # the near wall faces the ray
    front_out = product_trace_ex(export, outside, masks, flags=core.RAY_CULL_FRONT_FACING)[0]
    assert (front_out["inst"] == 0).all() and (front_out["t"] > plain_out["t"]).all()     # the far wall, from behind
    assert (product_trace_ex(export, inside, masks, flags=core.RAY_CULL_BACK_FACING)[0]["inst"] == 0xffffffff).all()
    assert H.hits_equal(product_trace_ex(export, inside, masks, flags=core.RAY_CULL_FRONT_FACING)[0], plain_in)
    assert (product_trace_ex(export, outside, masks, flags=3)[0]["inst"] == 0xffffffff).all()


CTYPES = {"rtc_context*": C.c_void_p, "uint64_t": C.c_uint64, "uint32_t": C.c_uint32, "int": C.c_int, "const uint8_t*": C.c_void_p,
          "rtc_trace_counts*": C.POINTER(core.TraceCounts)}


def test_exports_signatures_and_refusals_without_a_device(built):
    L = core.lib()
    nm = subprocess.run(["nm", "-D", "--defined-only", core.LIB_PATH], capture_output=True, text=True, check=True).stdout
    header = open(os.path.join(H.ROOT, "include", "rtc_core.h")).read()
    for name in NEW:
        assert name in core.SYMBOLS and re.search(r"\bT %s\b" % name, nm), name
        proto = re.search(r"int %s\(([^)]*)\);" % name, header)
        assert proto, name
        params = [re.sub(r"\s*\w+$", "", p.strip()).replace(" *", "*") for p in proto.group(1).split(",")]
        assert [CTYPES[p] for p in params] == list(getattr(L, name).argtypes), name
    assert re.search(r"#define RTC_RAY_CULL_BACK_FACING\s+1u", header) and re.search(r"#define RTC_RAY_CULL_FRONT_FACING\s+2u", header)
    assert (core.RAY_CULL_BACK_FACING, core.RAY_CULL_FRONT_FACING) == (1, 2)
    assert L.rtc_version() == 102
    # the filter arguments are checked before anything else: no context is needed to see them refused
    out = core.TraceCounts()
    for call in (lambda m, f: L.rtc_trace_closest_ex(None, 0, 0, 1, 0, m, f), lambda m, f: L.rtc_trace_any_ex(None, 0, 0, 1, 0, m, f),
                 lambda m, f: L.rtc_trace_count_ex(None, 0, 0, 1, 0, m, f, C.byref(out))):
        assert call(0x100, 0) != 0 and b"visibilityMask" in L.rtc_last_error()
        assert call(0xFF, 4) != 0 and b"rayFlags" in L.rtc_last_error()
        assert call(0xFFFFFFFF, 0) != 0 and b"visibilityMask" in L.rtc_last_error()


def test_python_keywords_choose_the_exports():
    """trace_closest / trace_any / trace_count call the _ex exports only when mask or flags is not the default."""
    calls = []

    class FakeLib:
        def __getattr__(self, name):
            return lambda *a: calls.append(name) or 0

    ctx = core.Context.__new__(core.Context)
    ctx.L, ctx.h = FakeLib(), None
    ctx.trace_closest(1, 2, 3, 4)
    ctx.trace_closest(1, 2, 3, 4, mask=1)
    ctx.trace_any(1, 2, 3, 4)
    ctx.trace_any(1, 2, 3, 4, flags=core.RAY_CULL_BACK_FACING)
    ctx.trace_count(1, 2, 3)
    ctx.trace_count(1, 2, 3, mask=0xFE, flags=0)
    assert calls == ["rtc_trace_closest", "rtc_trace_closest_ex", "rtc_trace_any", "rtc_trace_any_ex", "rtc_trace_count", "rtc_trace_count_ex"]
