"""GPU tests of rtc_gas_create / rtc_gas_build_device: a geometry whose triangle set is read from device memory and rebuilt in
place on the device.  Its nodes and triangle records must equal the host twin (the ("gas_build_device", ...) step of
host_scene_rebuild_export) byte for byte, whatever it held before; scenes that instance it must give the hits and frames of
scenes built from rtc_gas_build over the same buffers once rtc_ias_update has run; out-of-range indices make their triangles
inactive and are counted; refusals leave the GAS as it was; and the build never blocks the host."""
import subprocess
import sys
import time

import numpy as np
import pytest

import helpers as H
from oracle import orc
from test_cpu_gas_build_device import with_bad_indices
from test_cpu_gas_rebuild import oracle_of
from test_cpu_ias_build_device import mesh
from test_cpu_refit import deform, moved
from test_gpu_builder import soup
from test_gpu_gas_rebuild import IDENT, gas_export, same_gas, traded
from test_gpu_ias_build_device import _app_records, _flags, _render, build_device, same_export
from test_gpu_ias_rebuild import check_hits, stream_busy
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

EMPTY = mesh(np.zeros((0, 3), dtype=np.float32), np.zeros((0, 3), dtype=np.uint32))
ZERO = np.zeros((0, 12), dtype=np.float32)


def twin_gas(attrs, idx):
    return core.host_scene_rebuild_export([EMPTY], [(IDENT, 0)], [("gas_build_device", 0, attrs, idx)])[0]["gas"][0]


def build(ctx, g, attrs, idx, keep):
    """gas_build_device from new device buffers (kept alive in `keep`)"""
    d_a, d_i = ctx.to_device(attrs), ctx.to_device(np.ascontiguousarray(idx, dtype=np.uint32))
    keep += [d_a, d_i]
    ctx.gas_build_device(g, d_a, attrs.dtype.itemsize, len(attrs), d_i, len(idx))
    return d_a, d_i


@pytest.mark.parametrize("n", [0, 1, 2, 8, 9, 1000, 100_000, 1_000_000, 10_000_000])
def test_build_equals_the_host_twin(cuda_device, n):
    attrs, idx = soup(n, seed=n, extent=0.5 / max(n, 8) ** (1 / 3))
    twin = twin_gas(attrs, idx)
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(n)
        assert same_gas(gas_export(ctx, g), twin_gas(EMPTY[0], EMPTY[1]))           # created empty
        build(ctx, g, attrs, idx, keep)
        assert same_gas(gas_export(ctx, g), twin)
        assert ctx.gas_rejected_triangles(g) == 0
        ctx.gas_build_device(g, keep[0], attrs.dtype.itemsize, len(attrs), keep[1], n)   # a second build: the same bytes
        assert same_gas(gas_export(ctx, g), twin)
        ctx.gas_rebuild(g)                                                            # a rebuild over its buffers: the same
        assert same_gas(gas_export(ctx, g), twin)


def test_counts_that_grow_and_shrink(cuda_device):
    """one GAS of capacity 100 000 through 100 000 -> 10 -> 0 -> 5000 -> 100 000 -> 1 triangles of different soups"""
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(100_000)
        for k, n in enumerate((100_000, 10, 0, 5000, 100_000, 1)):
            attrs, idx = soup(n, seed=40 + k, extent=0.01)
            build(ctx, g, attrs, idx, keep)
            assert same_gas(gas_export(ctx, g), twin_gas(attrs, idx)), n


def test_scene_hits_and_export(cuda_device):
    """a scene of rtc_ias_build and a created scene instancing the GAS, after gas_build_device + ias_update: the hits of scenes
    built from rtc_gas_build over the same buffers, and the twin's export"""
    a0, i0 = soup(3000, seed=1, extent=0.03)
    a1, i1 = soup(7000, seed=2, extent=0.02)
    other = soup(2000, seed=3, extent=0.04)
    rng = np.random.default_rng(4)
    insts = [(moved([0.5, 0, 0, x, 0, 0.5, 0, y, 0, 0, 0.5, z], seed=k), k % 2) for k, (x, y, z) in enumerate(rng.uniform(-1, 1, size=(10, 3)))]
    xf = [t for t, _ in insts]
    rays = H.random_rays(100000, seed=6, lo=(-1.5,) * 3, hi=(1.5,) * 3, tmin=1e-5)
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(10000)
        build(ctx, g, a0, i0, keep)
        d_o, d_oi = ctx.to_device(other[0]), ctx.to_device(other[1])
        h = ctx.gas_build(d_o, other[0].dtype.itemsize, len(other[0]), d_oi, len(other[1]), core.BUILD_HOST_SAH)
        records = np.zeros(len(insts), dtype=core.INSTANCE_DTYPE)
        records["transform"] = np.asarray(xf, dtype=np.float32)
        records["instanceId"] = np.arange(len(insts))
        records["gas"] = [g if k == 0 else h for _, k in insts]
        records["lightIndex"] = -1
        built = ctx.ias_build(records)
        created = ctx.ias_create(len(insts))
        build_device(ctx, created, records)
        d_a, d_i = build(ctx, g, a1, i1, keep)                                       # another count, new buffers
        for top in (built, created):
            with pytest.raises(core.RtcError, match="rtc_ias_update"):
                ctx.trace_closest_host(top, rays[:10])
            ctx.ias_update(top, ZERO)
        ref_g = ctx.gas_build(d_a, a1.dtype.itemsize, len(a1), d_i, len(i1), core.BUILD_HOST_SAH)
        ref = records.copy()
        ref["gas"][ref["gas"] == g] = ref_g
        fresh = ctx.ias_build(ref)
        geos = [(a0, i0), other]
        twin_b, _ = core.host_scene_rebuild_export(geos, insts, [("gas_build_device", 0, a1, i1), ([None, None], xf)])
        twin_c, _ = core.host_scene_rebuild_export(geos, insts, ["rebuild", ("gas_build_device", 0, a1, i1), ([None, None], xf)])
        for top, twin in ((built, twin_b), (created, twin_c)):
            export = ctx.scene_export(top)
            same_export(export, twin)
            assert same_gas(export["gas"][g], twin["gas"][0])
            got = check_hits(ctx, top, fresh, rays, export)
            assert (got["inst"] != 0xffffffff).mean() > 0.05
            info = ctx.scene_info(top)
            assert info.numTris == len(i1) + len(other[1])
            assert info.numNodes == len(export["gas"][g][0]) + len(export["gas"][h][0]) + info.numTlasNodes


def _mesh_replaced_frames(tmp_path):
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="96 64", samplesSqrt=2), H.scene_path("rtigo3_geometry"))
    try:
        app.render(1)
        app.frame()
        ctx = app.context(0)
        w, h = app.resolution
        sys_data = app.system_data()
        own = sys_data.topObject
        records = _app_records(app, ctx)
        g = int(np.argmax([len(app.geometry(k)[1]) for k in range(app.info.numGeometries)]))
        uses = [i for i in range(app.info.numInstances) if app.instance(i)[1] == g]
        attrs, idx = app.geometry(g)
        # the new mesh: a permuted subset of the triangles (another count, another index buffer) over deformed vertices
        perm = np.random.default_rng(3).permutation(len(idx))[: (2 * len(idx)) // 3]
        new_attrs, new_idx = deform(attrs, 0.2, seed=9), idx[perm]
        keep = []
        gc = ctx.gas_create(len(idx))
        build(ctx, gc, attrs, idx, keep)                                             # the scenes are made over the old mesh
        mine = records.copy()
        mine["gas"][uses] = gc
        cut, albedo = _flags(app, mine)
        built = ctx.ias_build(mine)
        created = ctx.ias_create(len(mine))
        build_device(ctx, created, mine)
        d_a, d_i = build(ctx, gc, new_attrs, new_idx, keep)
        ref_g = ctx.gas_build(d_a, new_attrs.dtype.itemsize, len(new_attrs), d_i, len(new_idx), core.BUILD_DEFAULT)
        ref = records.copy()
        ref["gas"][uses] = ref_g
        ref_top = ctx.ias_build(ref)
        frames = []
        for top in (ref_top, built, created):
            if top != ref_top:
                ctx.ias_update(top, ZERO)
            ctx.set_instance_flags(top, 0, cut)
            ctx.set_albedo_textures(top, albedo)
            frames.append(_render(ctx, sys_data, w, h, app.info.miss, top, 4))
        frames.append(_render(ctx, sys_data, w, h, app.info.miss, own, 4))
        ctx.synchronize()
        sys_data.topObject = own
        return frames
    finally:
        app.close()


def test_frames_of_a_replaced_mesh(cuda_device, tmp_path):
    """one mesh of the geometry scene replaced through a created GAS (another triangle count, new index and vertex buffers) renders
    bit for bit as the scene with that mesh built by rtc_gas_build, for a scene of rtc_ias_build and a created scene; the shading
    interpolates through the new index buffer, which rtc_ias_update takes into every recomputed instance"""
    ref, built, created, original = _mesh_replaced_frames(tmp_path)
    assert built.tobytes() == ref.tobytes()
    assert created.tobytes() == ref.tobytes()
    assert ref.tobytes() != original.tobytes()


def test_rejected_indices_and_non_finite_vertices(cuda_device):
    attrs, idx, bad, (far, ref_idx) = with_bad_indices(20000, seed=8, num_bad=2000)
    # non-finite and huge vertices of some valid triangles: inactive, but not rejected
    rng = np.random.default_rng(2)
    good = np.setdiff1d(np.arange(len(idx)), bad)
    odd = rng.choice(good, size=300, replace=False)
    for k, v in enumerate((np.nan, np.inf, -np.inf, 1e38)):
        attrs["vertex"][idx[odd[k::4], 0]] = v
        far["vertex"][ref_idx[odd[k::4], 0]] = v
    rays = H.random_rays(50000, seed=3, lo=(-2.5,) * 3, hi=(2.5,) * 3, tmax=100.0)
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(len(idx))
        build(ctx, g, attrs, idx, keep)
        assert ctx.gas_rejected_triangles(g) == len(bad)
        twin = twin_gas(attrs, idx)
        assert same_gas(gas_export(ctx, g), twin)
        top = ctx.ias_build(np.array([(IDENT, 0, g, 0, -1)], dtype=core.INSTANCE_DTYPE))
        got = ctx.trace_closest_host(top, rays)
        ref = oracle_of([(far, ref_idx)], [(IDENT, 0)])
        assert H.hits_equal(got[:5000], ref.trace_closest(rays[:5000], brute_force=True))
        assert not np.isin(got["prim"][got["inst"] != 0xffffffff], np.concatenate([bad, odd])).any()
        assert (got["inst"] != 0xffffffff).mean() > 0.05
        short = rays[:5000].copy(); short["tmax"] = 0.5
        assert np.array_equal(ctx.trace_any_host(top, short).astype(bool), ref.trace_any(short).astype(bool))
        # a refit and a rebuild keep the rule: the twin's NaN vertex
        new = deform(attrs, 0.01, seed=4)
        ctx.upload(keep[0], new)
        ctx.gas_refit(g)
        twin_r, _ = core.host_scene_rebuild_export([EMPTY], [(IDENT, 0)], [("gas_build_device", 0, attrs, idx), ([new], [IDENT])])
        assert same_gas(gas_export(ctx, g), twin_r["gas"][0])
        ctx.gas_rebuild(g)
        assert same_gas(gas_export(ctx, g), twin_gas(new, idx))
        assert ctx.gas_rejected_triangles(g) == len(bad)


def test_refusals(cuda_device):
    attrs, idx = soup(100, seed=5)
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(100)
        d_a, d_i = build(ctx, g, attrs, idx, keep)
        before = gas_export(ctx, g)
        built = ctx.gas_build(d_a, 48, len(attrs), d_i, 100, core.BUILD_HOST_SAH)
        doomed = ctx.gas_create(10)
        ctx.gas_destroy(doomed)
        cases = [((999, d_a, 48, 300, d_i, 100), "bad gas handle"), ((doomed, d_a, 48, 300, d_i, 10), "bad gas handle"),
                 ((built, d_a, 48, 300, d_i, 100), "rtc_gas_create"), ((g, d_a, 48, 300, d_i, 101), "capacity"),
                 ((g, d_a, 8, 300, d_i, 100), "stride"), ((g, d_a, 50, 300, d_i, 100), "stride"),
                 ((g, d_a + 2, 48, 300, d_i, 100), "attributes is not 4-byte aligned"),
                 ((g, d_a, 48, 300, d_i + 1, 100), "indices is not 4-byte aligned"),
                 ((g, 0, 48, 300, d_i, 100), "null"), ((g, d_a, 48, 300, 0, 100), "null")]
        for args, msg in cases:
            with pytest.raises(core.RtcError, match=msg):
                ctx.gas_build_device(*args)
            assert same_gas(gas_export(ctx, g), before), msg
        with pytest.raises(core.RtcError, match="bad gas handle"):
            ctx.gas_rejected_triangles(doomed)
        assert ctx.gas_rejected_triangles(built) == 0
        ctx.gas_build_device(g, 0, 12, 0, 0, 0)                                       # no triangle: nothing to read
        assert same_gas(gas_export(ctx, g), twin_gas(EMPTY[0], EMPTY[1]))
        one = ctx.gas_create(0)                                                       # capacity 0 is 1
        build(ctx, one, attrs[:3], idx[:1], keep)
        with pytest.raises(core.RtcError, match="capacity"):
            ctx.gas_build_device(one, d_a, 48, 300, d_i, 2)


def test_seeded_programs(cuda_device):
    """gas_build_device (varying counts, new or in-place buffers, a few bad indices), gas_refit, gas_rebuild, ias_update,
    ias_rebuild and ias_build_device in seeded orders on a scene of rtc_ias_build and a created scene: after every step both exports
    equal the twin's replay"""
    cap = 6000
    other = soup(2500, seed=12, extent=0.04)
    geos = [EMPTY, other]
    rng = np.random.default_rng(21)
    insts = [(moved([0.4, 0, 0, x, 0, 0.4, 0, y, 0, 0, 0.4, z], seed=k), k % 2) for k, (x, y, z) in enumerate(rng.uniform(-1, 1, size=(9, 3)))]
    rays = H.random_rays(30000, seed=2, lo=(-1.5,) * 3, hi=(1.5,) * 3, tmin=1e-5)
    for seed in range(3):
        prog = np.random.default_rng(seed)
        with core.Context(0) as ctx:
            keep = []
            g = ctx.gas_create(cap)
            d_o, d_oi = ctx.to_device(other[0]), ctx.to_device(other[1])
            h = ctx.gas_build(d_o, other[0].dtype.itemsize, len(other[0]), d_oi, len(other[1]), core.BUILD_HOST_SAH)
            cur_xf = [t for t, _ in insts]

            def records():
                r = np.zeros(len(insts), dtype=core.INSTANCE_DTYPE)
                r["transform"] = np.asarray(cur_xf, dtype=np.float32)
                r["instanceId"] = np.arange(len(insts))
                r["gas"] = [g if k == 0 else h for _, k in insts]
                r["lightIndex"] = -1
                return r

            built = ctx.ias_build(records())
            created = ctx.ias_create(len(insts))
            build_device(ctx, created, records())
            steps_b, steps_c = [], ["rebuild"]
            big_a, big_i = ctx.malloc(3 * cap * 48), ctx.malloc(3 * cap * 4)       # the in-place buffers
            keep += [big_a, big_i]
            cur, cur_buf = None, None
            for k in range(10):
                ops = ["gas_build_device", "gas_refit", "gas_rebuild", "ias_update", "ias_rebuild", "ias_build_device"]
                op = "gas_build_device" if cur is None else ops[prog.integers(len(ops))]
                both = []
                if op == "gas_build_device":
                    n = int(prog.choice([0, 1, 9, 500, cap, int(prog.integers(1, cap))]))
                    attrs, idx = soup(n, seed=1000 * seed + k, extent=0.05)
                    if n > 20:
                        idx[prog.choice(n, size=5, replace=False), 1] = 3 * n + 7
                    if n and prog.integers(2):
                        ctx.upload(big_a, attrs)
                        ctx.upload(big_i, idx)
                        cur_buf = big_a
                        ctx.gas_build_device(g, big_a, 48, len(attrs), big_i, n)
                    else:
                        cur_buf, _ = build(ctx, g, attrs, idx, keep)
                    cur = (attrs, idx)
                    both, refit = [("gas_build_device", 0, attrs, idx)], [None, None]
                elif op in ("gas_refit", "gas_rebuild"):
                    attrs, idx = cur
                    new = traded(attrs, seed=k) if op == "gas_rebuild" else deform(attrs, 0.02, seed=k)
                    if len(attrs):
                        ctx.upload(cur_buf, new)
                    (ctx.gas_rebuild if op == "gas_rebuild" else ctx.gas_refit)(g)
                    cur = (new, idx)
                    if op == "gas_rebuild":
                        both, refit = [("gas_rebuild", 0, new)], [None, None]
                    else:
                        both, refit = [], [new, None]
                if op in ("gas_build_device", "gas_refit", "gas_rebuild"):
                    for top in (built, created):
                        ctx.ias_update(top, ZERO)
                    steps_b += both + [(refit, list(cur_xf))]
                    steps_c += both + [(refit, list(cur_xf))]
                elif op == "ias_update":
                    cur_xf = [moved(t, seed=1000 * seed + 10 * k + i) for i, t in enumerate(cur_xf)]
                    for top in (built, created):
                        ctx.ias_update(top, np.asarray(cur_xf, dtype=np.float32))
                    steps_b.append(([None, None], list(cur_xf)))
                    steps_c.append(([None, None], list(cur_xf)))
                elif op == "ias_rebuild":
                    for top in (built, created):
                        ctx.ias_rebuild(top)
                    steps_b.append("rebuild")
                    steps_c.append("rebuild")
                elif op == "ias_build_device":
                    build_device(ctx, created, records())
                    steps_c += [([None, None], list(cur_xf)), "rebuild"]
                for top, steps in ((built, steps_b), (created, steps_c)):
                    twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
                    export = ctx.scene_export(top)
                    same_export(export, twin)
                    assert same_gas(export["gas"][g], twin["gas"][0]), (seed, k, op)
                    assert same_gas(export["gas"][h], twin["gas"][1]), (seed, k, op)
            for top, steps in ((built, steps_b), (created, steps_c)):
                twin, _ = core.host_scene_rebuild_export(geos, insts, steps)
                hits, _ = orc.wide_trace(twin, rays)
                assert H.hits_equal(ctx.trace_closest_host(top, rays), hits)


def test_build_does_not_block_the_host(cuda_device, tmp_path):
    attrs, idx = soup(200_000, seed=3, extent=0.01)
    app = host.App(H.write_system(tmp_path, "rtigo3_geometry", resolution="1920 1080", samplesSqrt=1), H.scene_path("rtigo3_geometry"))
    try:
        app.render(1)
        app.frame()
        ctx = app.context(0)
        ctx.set_trace_schedule("group")
        sys_data = app.system_data()
        keep = []
        g = ctx.gas_create(len(idx))
        build(ctx, g, attrs, idx, keep)                                              # warm: the pool holds the build's scratch
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, 4)
        ctx.synchronize()
        per_iteration = (time.perf_counter() - t0) / 4
        iterations = int(min(2000, max(8, 0.5 / per_iteration)))
        ctx.launch(sys_data, 1920, 1080, core.RAYGEN_FULL_FRAME, app.info.miss, 0, iterations)
        ctx.gas_build_device(g, keep[0], 48, len(attrs), keep[1], len(idx) // 2)
        pending = stream_busy(ctx.stream)
        ctx.synchronize()
        assert pending, "rtc_gas_build_device returned after the launch before it had finished: it synchronised the host"
        assert same_gas(gas_export(ctx, g), twin_gas(attrs, idx[: len(idx) // 2]))
        ctx.gas_destroy(g)
    finally:
        app.close()


_TORCH_TRIANGLES = """
import sys
import numpy as np
import torch
sys.path.insert(0, "tests")
from test_gpu_builder import soup
from test_gpu_gas_build_device import twin_gas
from test_gpu_gas_rebuild import gas_export, same_gas
from tweeker_raytracer_b200 import core

attrs, idx = soup(50000, seed=31, extent=0.01)
twin = twin_gas(attrs, idx)
with core.Context(0) as ctx:
    g = ctx.gas_create(50000)
    ctx.synchronize()
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    with torch.cuda.stream(stream):
        a = torch.from_numpy(attrs.view(np.float32).reshape(len(attrs), 12).copy()).to("cuda")
        verts = torch.zeros_like(a)
        verts.copy_(a * 2.0 - a)                                            # a kernel of torch's writes the vertices
        tris = torch.from_numpy(idx.astype(np.int32)).to("cuda") + 0        # and the indices
        ctx.gas_build_device(g, verts.data_ptr(), 48, len(attrs), tris.data_ptr(), len(idx))   # no host synchronisation
    ctx.synchronize()
    assert same_gas(gas_export(ctx, g), twin)
print("torch triangles ok")
"""


def test_triangles_written_by_torch_on_the_context_stream(cuda_device):
    """vertices and indices a torch kernel writes on torch.cuda.ExternalStream(rtc_context_stream) are consumed in stream order.
    In a fresh interpreter: torch must be imported before the host library brings in its own NCCL."""
    out = subprocess.run([sys.executable, "-c", _TORCH_TRIANGLES], cwd=H.ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "torch triangles ok" in out.stdout, out.stdout + out.stderr


def test_destroy_makes_scenes_unusable(cuda_device):
    attrs, idx = soup(500, seed=6)
    rays = H.random_rays(1000, seed=1, lo=(0,) * 3, hi=(1,) * 3)
    with core.Context(0) as ctx:
        keep = []
        g = ctx.gas_create(500)
        build(ctx, g, attrs, idx, keep)
        rec = np.array([(IDENT, 0, g, 0, -1)], dtype=core.INSTANCE_DTYPE)
        built = ctx.ias_build(rec)
        created = ctx.ias_create(1)
        build_device(ctx, created, rec)
        assert (ctx.trace_closest_host(built, rays)["inst"] == 0).any()
        ctx.gas_destroy(g)
        for top in (built, created):
            with pytest.raises(core.RtcError, match="a GAS of this scene was destroyed"):
                ctx.trace_closest_host(top, rays)
        with pytest.raises(core.RtcError, match="bad gas handle"):
            ctx.gas_build_device(g, keep[0], 48, len(attrs), keep[1], len(idx))
