"""CPU tests of the builders, refits and rebuilds on non-finite, tiny and large inputs, through their host twins
(csrc/accel_host.cpp, which share csrc/bvh_rules.h with the device paths) and the scalar restatement of the traversal
(oracle/wide_bvh.inc).

The reference is the oracle's brute force with the inactive rules of DESIGN.md section 3: a triangle with a vertex coordinate
that is NaN, infinite or beyond B = 2^126, and an instance whose transform has a non-finite entry or whose transformed vertices
reach beyond B, are never hit and bound nothing.  Every other triangle must give exactly the brute-force hits, closest hit and
any hit -- finite coordinates up to B and axis-parallel rays over any extent included -- and every structure must keep the node
format's invariants.

Each case runs in a child process (this file run as a script), so that a builder that crashes fails its case and not the run.
"""
import json
import os
import subprocess
import sys

TESTS = os.path.dirname(os.path.abspath(__file__))
if __name__ == "__main__":
    sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import numpy as np  # noqa: E402
import pytest  # noqa: E402

import helpers as H  # noqa: E402
from oracle import orc  # noqa: E402
from test_cpu_gas_rebuild import IDENT, oracle_of, soup  # noqa: E402
from test_cpu_host_accel import check_structure, tri_boxes  # noqa: E402
from tweeker_raytracer_b200 import core  # noqa: E402

NONFINITE = {"nan": np.nan, "inf": np.inf, "-inf": -np.inf}
B = 2.0 ** 126                                  # bvh_rules.h RTC_COORD_BOUND
MISS = 0xffffffff


# ---- scenes and rays ------------------------------------------------------------------------------------------------------
def rays_at(points, rng, dist=40.0, tmin=0.0, tmax=1e27):
    """One ray per point from `dist` away in a random direction, aimed at the point (vertices and edges that define boxes)."""
    points = np.asarray(points, dtype=np.float64)
    d = rng.normal(size=points.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = np.zeros(len(points), dtype=orc.RAY_DTYPE)
    o = points - dist * d
    r["ox"], r["oy"], r["oz"] = o[:, 0], o[:, 1], o[:, 2]
    r["dx"], r["dy"], r["dz"] = d[:, 0], d[:, 1], d[:, 2]
    r["tmin"], r["tmax"] = tmin, tmax
    return r


def axis_rays(lo, hi, n, seed, tmax=1e27):
    """Axis-parallel rays: one direction component +-1, the other two exactly +0.0 or -0.0, origins outside the box (lo, hi)
    on the side the ray starts from and spread over the box on the other two axes."""
    rng = np.random.default_rng(seed)
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    r = np.zeros(n, dtype=orc.RAY_DTYPE)
    axis = rng.integers(0, 3, n)
    sign = rng.choice([-1.0, 1.0], n)
    o = rng.uniform(lo, hi, size=(n, 3))
    d = np.where(rng.random((n, 3)) < 0.5, 0.0, -0.0)
    for i in range(n):
        a = axis[i]
        d[i, a] = sign[i]
        o[i, a] = lo[a] - 0.25 * (hi[a] - lo[a]) - 1.0 if sign[i] > 0 else hi[a] + 0.25 * (hi[a] - lo[a]) + 1.0
    r["ox"], r["oy"], r["oz"] = o[:, 0], o[:, 1], o[:, 2]
    r["dx"], r["dy"], r["dz"] = d[:, 0], d[:, 1], d[:, 2]
    r["tmin"], r["tmax"] = 0.0, tmax
    return r


def gas_rays(attrs, seed, n=1500):
    v = attrs["vertex"].astype(np.float64)
    fin = np.isfinite(v).all(axis=1)
    lo, hi = v[fin].min(axis=0), v[fin].max(axis=0)
    rng = np.random.default_rng(seed)
    parts = [H.random_rays(n, seed, lo=tuple(lo), hi=tuple(hi), tmin=0.0)]
    pts = v[fin][rng.integers(0, fin.sum(), 300)]
    edges = 0.5 * (pts + v[fin][rng.integers(0, fin.sum(), 300)])
    parts += [rays_at(pts, rng), rays_at(edges, rng)]
    far = H.random_rays(300, seed + 1, lo=tuple(lo - 1e4), hi=tuple(lo - 1e4 + 1.0), tmin=0.0)
    aim = rng.uniform(lo, hi, size=(300, 3)) - np.stack([far["ox"], far["oy"], far["oz"]], axis=1)
    aim /= np.linalg.norm(aim, axis=1, keepdims=True)
    far["dx"], far["dy"], far["dz"] = aim[:, 0], aim[:, 1], aim[:, 2]                  # origins far outside the scene
    parts += [far, axis_rays(lo, hi, 400, seed)]
    return np.concatenate(parts)


def with_vertex(attrs, idx, where, axis, value):
    out = attrs.copy()
    v = out["vertex"]
    if where == "vertex7":
        v[7, axis] = value
    elif where == "first_triangle":
        v[idx[0], axis] = value
    elif where == "last_triangle":
        v[idx[-1], axis] = value
    elif where == "all_three":                                            # every vertex of triangle 5
        v[idx[5], axis] = value
    else:
        raise ValueError(where)
    return out


# ---- checks ---------------------------------------------------------------------------------------------------------------
def check_export(export, geos, insts, rays, leaf_max):
    """Structure of every level, and closest / any hits of the scalar traversal equal to the oracle's brute force."""
    for g, (nodes, tris) in export["gas"].items():
        boxes = tri_boxes(tris)
        bad = ~(np.abs(tris.reshape(-1, 12)[:, [0, 1, 2, 4, 5, 6, 8, 9, 10]].astype(np.float64)) <= B).all(axis=1)
        boxes[bad, 0], boxes[bad, 1] = np.inf, -np.inf                    # inactive: contained by any box
        check_structure(nodes, len(geos[g][1]), boxes, leaf_max)
    check_structure(export["tlas_nodes"], len(insts), None, 1)
    ref = oracle_of(geos, insts)
    want = ref.trace_closest(rays, brute_force=True)
    got, _ = orc.wide_trace(export, rays)
    lost = int(((want["inst"] != MISS) & (got["inst"] == MISS)).sum())
    assert H.hits_equal(got, want), "closest hits differ from brute force: %d of %d hits lost, %d rays differ" % (
        lost, int((want["inst"] != MISS).sum()), int((got["t"].view(np.uint32) != want["t"].view(np.uint32)).sum()))
    occl, _ = orc.wide_trace(export, rays, any_hit=True)
    assert np.array_equal(occl["inst"] != MISS, ref.trace_any(rays, brute_force=True).astype(bool)), "any hit differs from brute force"
    return int((want["inst"] != MISS).sum())


def gas_export(path, attrs, idx, new):
    """The export of one geometry (instanced once, identity) whose vertices are `new`: built from them (sah), or built from
    `attrs` and then rebuilt or refitted to them."""
    geos, insts = [(attrs, idx)], [(IDENT, 0)]
    if path == "sah":
        return core.host_scene_export([(new, idx)], insts)[0]
    if path == "rebuild":
        return core.host_scene_rebuild_export(geos, insts, [("gas_rebuild", 0, new), ([None], [IDENT])])[0]
    if path == "refit":
        return core.host_scene_rebuild_export(geos, insts, [([new], [IDENT])])[0]
    raise ValueError(path)


# ---- cases (run in the child process) -------------------------------------------------------------------------------------
def case_gas_vertex(path, value, wheres, axes):
    """One vertex, a vertex of the first or the last triangle, or all three vertices of one triangle, with the coordinate `value`
    (non-finite, finite up to B or beyond it)."""
    attrs, idx = soup(2000, seed=1)
    rays = gas_rays(attrs, seed=11)
    leaf_max = 1 if path == "rebuild" else 2
    hits = 0
    for where in wheres:
        for axis in axes:
            new = with_vertex(attrs, idx, where, axis, np.float32(value))
            export = gas_export(path, attrs, idx, new)
            try:
                hits += check_export(export, [(new, idx)], [(IDENT, 0)], rays, leaf_max)
            except AssertionError as e:
                raise AssertionError("%s, axis %d: %s" % (where, axis, e))
    assert hits > 0


def case_gas_all_inactive(path):
    """Every triangle inactive: an empty structure that no ray enters, and nothing hit."""
    attrs, idx = soup(50, seed=2)
    new = attrs.copy()
    new["vertex"][::3, 1] = np.inf
    rays = gas_rays(attrs, seed=12, n=300)
    export = gas_export(path, attrs, idx, new)
    check_export(export, [(new, idx)], [(IDENT, 0)], rays, 1 if path == "rebuild" else 2)
    assert (orc.wide_trace(export, rays)[0]["inst"] == MISS).all()


def case_gas_revived(path):
    """Built with inactive triangles, refitted or rebuilt to finite positions: every triangle is found again."""
    attrs, idx = soup(2000, seed=1)
    bad = attrs.copy()
    bad["vertex"][7, 0] = np.nan
    bad["vertex"][3 * 1999, 2] = -np.inf
    geos, insts = [(bad, idx)], [(IDENT, 0)]
    step = ("gas_rebuild", 0, attrs) if path == "rebuild" else [attrs]
    steps = [step, ([None], [IDENT])] if path == "rebuild" else [(step, [IDENT])]
    export = core.host_scene_rebuild_export(geos, insts, steps)[0]
    check_export(export, [(attrs, idx)], insts, gas_rays(attrs, seed=13), 1 if path == "rebuild" else 2)


def case_gas_scale(path, spread, subnormal):
    """A soup in a 10-unit cube with eight small triangles at the corners of a cube of side 2 * spread, so that node extents
    reach `spread` while the hits stay where float triangle arithmetic is exact (and subnormal coordinates): exact hits for
    generic, aimed, far and axis-parallel rays."""
    attrs, idx = soup(500, seed=3)
    rays = gas_rays(attrs, seed=14, n=500)
    if subnormal:
        attrs["vertex"][:30] = np.float32(1e-39) * np.sign(attrs["vertex"][:30])
    corners = np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float64) * spread
    tri = np.array([[0, 0, 0], [0.3, 0, 0], [0, 0.3, 0]])
    far = np.zeros(24, dtype=attrs.dtype)
    far["vertex"] = (corners[:, None, :] + tri[None]).reshape(-1, 3).astype(np.float32)
    attrs = np.concatenate([attrs, far])
    idx = np.arange(len(attrs), dtype=np.uint32).reshape(-1, 3)
    export = gas_export(path, attrs, idx, attrs.copy())
    assert check_export(export, [(attrs, idx)], [(IDENT, 0)], rays, 1 if path == "rebuild" else 2) > 0


def instance_scene(n=50, tris=300):
    attrs, idx = soup(tris, seed=5, spread=2.0, size=0.2)
    rng = np.random.default_rng(6)
    xf = []
    for i in range(n):
        m = IDENT.copy().reshape(3, 4)
        m[:, 3] = rng.uniform(-10, 10, 3)
        xf.append(m.reshape(12))
    return [(attrs, idx)], xf


def changed_transform(kind, entry=None):
    m = IDENT.copy().reshape(3, 4)
    m[:, 3] = (1.0, 2.0, 3.0)
    if kind in NONFINITE:
        m.reshape(12)[entry] = NONFINITE[kind]
    elif kind == "zero_scale":
        m[:, :3] = 0.0
    elif kind == "scale_1e-30":
        m[:, :3] *= np.float32(1e-30)
    elif kind == "scale_1e30":
        m[:, :3] *= np.float32(1e30)
    elif kind == "translate_1e36":                                         # within B: exact, and the others unaffected
        m[0, 3] = np.float32(1e36)
    elif kind == "translate_1e38":                                         # beyond B: inactive
        m[1, 3] = np.float32(1e38)
    elif kind == "mirrored":
        m[0, 0] = -1.0
    elif kind == "rotated_mirrored":
        m[:, :3] = np.array([[0, 1, 0], [1, 0, 0], [0, 0, -2]], dtype=np.float32)
    else:
        raise ValueError(kind)
    return m.reshape(12)


def instance_rays(seed):
    rng = np.random.default_rng(seed)
    r = H.random_rays(2000, seed, lo=(-12, -12, -12), hi=(12, 12, 12), tmin=0.0)
    return np.concatenate([r, rays_at(rng.uniform(-11, 11, size=(400, 3)), rng, dist=60.0), axis_rays((-11, -11, -11), (11, 11, 11), 400, seed)])


def case_instance(path, kind, entries):
    """Instance 17 of 50 given the transform `kind` (for a non-finite kind: in each of the entries `entries`)."""
    geos, xf = instance_scene()
    rays = instance_rays(21)
    for entry in entries:
        new = list(xf)
        new[17] = changed_transform(kind, entry)
        insts = [(t, 0) for t in new]
        if path == "build":
            export = core.host_scene_export(geos, insts)[0]
        elif path == "update":
            export = core.host_scene_rebuild_export(geos, [(t, 0) for t in xf], [([None], new)])[0]
        elif path == "update_rebuild":
            export = core.host_scene_rebuild_export(geos, [(t, 0) for t in xf], [([None], new), "rebuild"])[0]
        else:
            raise ValueError(path)
        try:
            hits = check_export(export, geos, insts, rays, 2)
        except AssertionError as e:
            raise AssertionError("entry %s: %s" % (entry, e))
        assert hits > 100


def case_instance_of_inactive_geometry(path):
    """Instances of a geometry whose triangles are all inactive next to instances of a finite one."""
    attrs, idx = soup(40, seed=7, spread=2.0, size=0.2)
    bad = attrs.copy()
    bad["vertex"][:, 0] = np.nan
    geos = [(attrs, idx), (bad, idx)]
    insts = [(changed_transform("mirrored"), 0), (IDENT, 1), (changed_transform("rotated_mirrored"), 1)]
    rays = instance_rays(22)
    if path == "build":
        export = core.host_scene_export(geos, insts)[0]
    else:
        export = core.host_scene_rebuild_export([(attrs, idx), (attrs, idx)], insts, [("gas_rebuild", 1, bad), ([None, None], [t for t, _ in insts]), "rebuild"])[0]
    check_export(export, geos, insts, rays, 2)


CASES = {f.__name__: f for f in (case_gas_vertex, case_gas_all_inactive, case_gas_revived, case_gas_scale, case_instance,
                                  case_instance_of_inactive_geometry)}


def run_isolated(name, *args):
    """Runs CASES[name](*args) in a child process: a crash (signal) or an assertion fails this case alone."""
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), name, json.dumps(args)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, "%s%r: exit code %d\n%s\n%s" % (name, args, r.returncode, r.stdout[-4000:], r.stderr[-4000:])


# ---- tests ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("value", sorted(NONFINITE))
@pytest.mark.parametrize("path", ["sah", "rebuild", "refit"])
def test_nonfinite_vertex(built, path, value):
    run_isolated("case_gas_vertex", path, value, ["vertex7", "first_triangle", "last_triangle", "all_three"], [0, 1, 2])


# finite magnitudes on both sides of B: 8.5e37 = B is the largest active coordinate, 8.6e37, 1e38 and 3e38 are beyond it
@pytest.mark.parametrize("value", [1e20, 1e30, 1e35, -1e36, 1e37, float(B), float(np.nextafter(np.float32(B), np.float32(np.inf))), 1e38, -3e38])
@pytest.mark.parametrize("path", ["sah", "rebuild", "refit"])
def test_large_finite_vertex(built, path, value):
    run_isolated("case_gas_vertex", path, value, ["vertex7", "all_three"], [0, 1, 2])


@pytest.mark.parametrize("path", ["sah", "rebuild", "refit"])
def test_every_triangle_inactive(built, path):
    run_isolated("case_gas_all_inactive", path)


@pytest.mark.parametrize("path", ["rebuild", "refit"])
def test_inactive_triangles_come_back_when_finite(built, path):
    run_isolated("case_gas_revived", path)


@pytest.mark.parametrize("spread", [1.0, 1e6, 1e11, 1e12, 1e15, 1e20, 1e30, 1e36, 8e37])
@pytest.mark.parametrize("path", ["sah", "rebuild"])
def test_axis_parallel_and_generic_rays_over_scene_extents(built, path, spread):
    run_isolated("case_gas_scale", path, spread, False)


@pytest.mark.parametrize("path", ["sah", "rebuild", "refit"])
def test_subnormal_coordinates(built, path):
    run_isolated("case_gas_scale", path, 1.0, True)


@pytest.mark.parametrize("kind", ["nan", "inf", "-inf"])
@pytest.mark.parametrize("path", ["build", "update", "update_rebuild"])
def test_nonfinite_instance_transform(built, path, kind):
    run_isolated("case_instance", path, kind, [0, 5, 3, 11])          # linear part (two entries) and translation (two entries)


@pytest.mark.parametrize("kind", ["zero_scale", "scale_1e-30", "scale_1e30", "mirrored", "rotated_mirrored", "translate_1e36", "translate_1e38"])
@pytest.mark.parametrize("path", ["build", "update", "update_rebuild"])
def test_singular_scaled_and_mirrored_instances(built, path, kind):
    run_isolated("case_instance", path, kind, [None])


@pytest.mark.parametrize("path", ["build", "rebuild"])
def test_instances_of_a_geometry_without_active_triangles(built, path):
    run_isolated("case_instance_of_inactive_geometry", path)


if __name__ == "__main__":
    CASES[sys.argv[1]](*json.loads(sys.argv[2]))
