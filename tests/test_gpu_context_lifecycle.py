"""GPU tests of one context across resource changes: renders again after a scene is destroyed and rebuilt, after the wavefront
buffers grow for a larger batch, after a GAS is destroyed under a live scene, and along seeded programs of App updates.  The
library caches one thing across launches -- the CUDA graph of the ordered any-hit rounds of scenes with cutout materials -- so
every frame is compared bit for bit with the oracle, and rtc_stats.cutoutGraphBuilds says when that graph was captured again."""
import numpy as np
import pytest

import helpers as H
from test_cpu_refit import moved
from test_gpu_builder import IDENTITY, soup
from tweeker_raytracer_b200 import core, host

pytestmark = pytest.mark.gpu

INSTANCE_CUTOUT = 1          # RTC_INSTANCE_CUTOUT (include/rtc_core.h)


def _app(tmp_path, scene="rtigo3_textures", resolution="48 32", samplesSqrt=4, **kw):
    return host.App(H.write_system(tmp_path, scene, resolution=resolution, samplesSqrt=samplesSqrt, **kw), H.scene_path(scene))


def _instances(app):
    return [app.instance(i) for i in range(app.info.numInstances)]


def _oracle_frame(app, iterations, instances=None):
    w, h = app.resolution
    return H.oracle_scene(app, instances=instances).render(H.oracle_sys(app), app.info.miss, w, h, iter_first=0,
                                                           iter_count=iterations).reshape(h, w, 4)


def _assert_same(got, want):
    same = (got.view(np.uint32) == want.view(np.uint32)).all(axis=2)
    assert same.all(), "%d of %d pixels differ" % ((~same).sum(), same.size)


def _builds(ctx):
    return ctx.stats().cutoutGraphBuilds


def _gas_of_geometry(app, ctx):
    """App geometry index -> GAS handle in the App's context."""
    inst_gas = ctx.scene_export(app.system_data().topObject)["instance_gas"]
    return {app.instance(i)[1]: int(inst_gas[i]) for i in range(app.info.numInstances)}


def _build_scene(app, ctx, gas_of, instances):
    """A scene in the App's own context from [(transform, geometry, material, light)], instance i at position i, with the hit
    records Device::updateHitRecords would select: cutout where the material has a cutout texture, albedo textures on when any
    material has one."""
    inst = np.zeros(len(instances), dtype=core.INSTANCE_DTYPE)
    for k, (t, g, m, l) in enumerate(instances):
        inst[k]["transform"], inst[k]["instanceId"], inst[k]["gas"], inst[k]["materialIndex"], inst[k]["lightIndex"] = t, k, gas_of[g], m, l
    top = ctx.ias_build(inst)
    mats = app.materials()
    ctx.set_instance_flags(top, 0, [INSTANCE_CUTOUT if 0 <= m < len(mats) and mats[m]["textureCutout"] != 0 else 0 for _, _, m, _ in instances])
    ctx.set_albedo_textures(top, bool((mats["textureAlbedo"] != 0).any()))
    return top


class _DirectLaunches:
    """rtc_launch with one fixed SystemData: a copy of the App's with its own output buffer, so that the graph's cache key sees
    the same SystemData at every launch unless the test changes topObject."""

    def __init__(self, app, ctx):
        self.app, self.ctx = app, ctx
        self.w, self.h = app.resolution
        self.sys = app.system_data()
        self.out = ctx.malloc(self.w * self.h * 16)
        ctx.memset(self.out, 0, self.w * self.h * 16)
        self.sys.outputBuffer = self.out

    def launch(self, first, count):
        """Launches iterations first .. first + count - 1 (accumulated from sample `first` on); returns the graph captures."""
        before = _builds(self.ctx)
        self.ctx.launch(self.sys, self.w, self.h, core.RAYGEN_FULL_FRAME, self.app.info.miss, first, count)
        return _builds(self.ctx) - before

    def frame(self):
        return self.ctx.download(self.out, np.float32, self.w * self.h * 4).reshape(self.h, self.w, 4)

    def close(self):
        self.ctx.free(self.out)


def _moved_scene(instances, seed):
    """Every instance that is not a light moved (the light definitions do not follow their instance)."""
    return [(moved(t, seed=seed + k) if l < 0 else t, g, m, l) for k, (t, g, m, l) in enumerate(instances)]


def test_app_renders_reuse_the_cutout_graph(cuda_device, tmp_path):
    """One launch per render(1): the graph is captured at the first launch and reused by the next ones (iterationIndex, which
    the App writes before every launch, is not part of its key)."""
    with _app(tmp_path) as app:
        assert (app.materials()["textureCutout"] != 0).any()
        ctx = app.context(0)
        app.set_coalesce(1)
        ctx.stats_reset()
        deltas = []
        for _ in range(3):
            before = _builds(ctx)
            assert app.render(1) == len(deltas) + 1
            deltas.append(_builds(ctx) - before)
        assert deltas == [1, 0, 0]
        _assert_same(app.frame(), _oracle_frame(app, 3))
        assert app.stats().stackOverflows == 0


def test_wavefront_growth_recaptures_the_graph_once(cuda_device, tmp_path, monkeypatch):
    monkeypatch.delenv("RTC_MAX_PATHS", raising=False)
    with _app(tmp_path, resolution="40 24") as app:          # not rendered yet: the first launch allocates the wavefront
        ctx = app.context(0)
        d = _DirectLaunches(app, ctx)
        try:
            assert d.launch(0, 1) == 1
            assert d.launch(1, 4) == 1                         # capacity pixels -> 4 * pixels: both buffers are new
            _assert_same(d.frame(), _oracle_frame(app, 5))
            assert d.launch(5, 2) == 0
            monkeypatch.setenv("RTC_MAX_PATHS", str(2 * d.w * d.h))
            assert d.launch(7, 4) == 0                         # two batches of two iterations in the same buffers
            _assert_same(d.frame(), _oracle_frame(app, 11))
            assert ctx.stats().stackOverflows == 0
        finally:
            d.close()


def test_replaced_scenes_recapture_the_graph_and_render_their_own_frames(cuda_device, tmp_path):
    """Destroy-then-build, as Device::initScene does: a new scene may get the freed scene's addresses, which the graph's key
    cannot tell apart, so rtc_scene_destroy releases the graph.  Alternates scenes of the same and of a different instance count."""
    with _app(tmp_path) as app:
        ctx = app.context(0)
        own = _instances(app)
        gas_of = _gas_of_geometry(app, ctx)
        d = _DirectLaunches(app, ctx)
        own_top = d.sys.topObject
        lights = [x for x in own if x[3] >= 0]
        others = [x for x in own if x[3] < 0]
        assert lights and len(others) >= 4

        def render(top, instances):
            if d.sys.topObject != top:
                d.sys.topObject = top
            builds = d.launch(0, 2)
            _assert_same(d.frame(), _oracle_frame(app, 2, instances))
            return builds

        scene_b = _moved_scene(own, seed=100)
        top = _build_scene(app, ctx, gas_of, scene_b)
        assert render(top, scene_b) == 1
        rounds = [_moved_scene(own, seed=200),                              # same count
                  lights + others[::2],                                     # fewer instances
                  _moved_scene(lights + others[::2], seed=300),             # same count as the last
                  own + [_moved_scene([x], seed=400 + k)[0] for k, x in enumerate(others[:3])]]   # more: repeated geometries
        repeated = []
        for instances in rounds:
            ctx.scene_destroy(top)
            old, top = top, _build_scene(app, ctx, gas_of, instances)
            repeated.append(old == top)
            if old != top:
                with pytest.raises(core.RtcError, match="unknown topObject"):
                    ctx.scene_info(old)
                d.sys.topObject = old
                with pytest.raises(core.RtcError, match="topObject"):
                    d.launch(0, 1)
            assert render(top, instances) == 1
        print("handle repeated after destroy-then-build:", repeated)
        # two live scenes: every switch changes the key
        assert render(own_top, own) == 1
        assert render(top, rounds[-1]) == 1
        assert render(own_top, own) == 1
        assert ctx.stats().stackOverflows == 0
        ctx.scene_destroy(top)
        d.close()


def test_scene_on_a_destroyed_gas_is_refused(cuda_device, tmp_path):
    with _app(tmp_path, resolution="40 24") as app:
        ctx = app.context(0)
        attrs, idx = soup(2000, seed=17, extent=0.05)
        d_a, d_i = ctx.to_device(attrs), ctx.to_device(idx)
        gas = ctx.gas_build(d_a, 48, len(attrs), d_i, len(idx), core.BUILD_HOST_SAH)
        inst = np.zeros(2, dtype=core.INSTANCE_DTYPE)
        for k, t in enumerate([IDENTITY, [0.5, 0, 0, 1.2, 0, 0.5, 0, 0.1, 0, 0, 0.5, 0.3]]):
            inst[k]["transform"], inst[k]["instanceId"], inst[k]["gas"], inst[k]["materialIndex"], inst[k]["lightIndex"] = t, k, gas, 1, -1
        top = ctx.ias_build(inst)
        ctx.set_instance_flags(top, 0, [INSTANCE_CUTOUT, 0])
        rays = H.random_rays(1000, seed=5, lo=(-0.5, -0.5, -0.5), hi=(1.9, 1.6, 1.3), tmin=1e-5)
        assert (ctx.trace_closest_host(top, rays)["inst"] != 0xffffffff).any()
        ctx.gas_destroy(gas)
        d = _DirectLaunches(app, ctx)
        d.sys.topObject = top
        d_r = ctx.to_device(rays)
        try:
            calls = [lambda: d.launch(0, 1), lambda: ctx.trace_closest_host(top, rays), lambda: ctx.trace_any_host(top, rays),
                     lambda: ctx.trace_count(top, d_r, len(rays)), lambda: ctx.trace_count(top, d_r, len(rays), any_hit=True),
                     lambda: ctx.ias_update(top, np.zeros((0, 12), dtype=np.float32))]
            for call in calls:
                with pytest.raises(core.RtcError, match="destroyed"):
                    call()
        finally:
            ctx.free(d_r)
            d.close()
        ctx.scene_destroy(top)
        ctx.free(d_a)
        ctx.free(d_i)
        app.set_coalesce(1)
        app.render(2)
        _assert_same(app.frame(), _oracle_frame(app, 2))
        assert app.stats().stackOverflows == 0


def test_cutout_toggled_between_reused_launches(cuda_device, tmp_path):
    """The kernels read the material table at run time: a graph reused after the materials changed must see the new ones."""
    with _app(tmp_path) as app:
        app.set_coalesce(1)
        mats = app.materials()
        cut = [i for i in range(len(mats)) if mats[i]["textureCutout"] != 0]
        assert len(cut) >= 2
        app.render(2)
        first = app.frame()
        _assert_same(first, _oracle_frame(app, 2))
        for i in range(len(mats)):
            app.update_material_textures(i, False, False)           # the plain path
        app.render(2)
        plain = app.frame()
        _assert_same(plain, _oracle_frame(app, 2))
        app.update_material_textures(cut[0], bool(mats[cut[0]]["textureAlbedo"] != 0), True)
        app.update_material_textures(cut[1], False, True)
        app.render(2)
        again = app.frame()
        _assert_same(again, _oracle_frame(app, 2))
        assert again.tobytes() != plain.tobytes()
        assert app.stats().stackOverflows == 0


@pytest.mark.parametrize("seed", list(range(8)))
def test_seeded_lifecycle_program(cuda_device, tmp_path, monkeypatch, seed):
    """About twelve random steps -- renders with a random coalescing limit, RTC_MAX_PATHS changes, moved instances, material
    and texture-switch updates, restarts -- with the App's frame compared with the oracle after every render step."""
    rng = np.random.default_rng(7100 + seed)
    scene = ["rtigo3_textures", "rtigo3_geometry"][seed % 2]
    w, h = int(rng.integers(24, 57)), int(rng.integers(16, 37))
    monkeypatch.delenv("RTC_MAX_PATHS", raising=False)
    with _app(tmp_path, scene=scene, resolution="%d %d" % (w, h), samplesSqrt=3) as app:
        spp = app.spp
        movable = [i for i in range(app.info.numInstances) if app.instance(i)[3] < 0]
        nm = app.info.numMaterials
        done, renders = 0, 0
        steps = [int(k) for k in rng.integers(0, 6, size=11)] + [0]
        for kind in steps:
            if kind == 0:
                app.set_coalesce(int(rng.integers(1, 5)))
                k = int(rng.integers(1, 5))
                done = min(spp, done + k)
                assert app.render(k) == done
                _assert_same(app.frame(), _oracle_frame(app, done))
                renders += 1
            elif kind == 1:
                monkeypatch.setenv("RTC_MAX_PATHS", str(int(rng.choice([w * h, 2 * w * h, 3 * w * h + 5, 64 << 20]))))
            elif kind == 2:
                i = int(rng.choice(movable))
                app.update_instance_transform(i, moved(app.instance(i)[0], seed=int(rng.integers(1 << 30))))
                done = 0
            elif kind == 3:
                app.update_material_textures(int(rng.integers(1, nm)), bool(rng.random() < 0.5), bool(rng.random() < 0.6))
                done = 0
            elif kind == 4:
                app.update_material(int(rng.integers(1, nm)), int(rng.integers(0, 5)), rng.uniform(0.1, 0.95, 3), roughness=rng.uniform(0.05, 0.6, 2),
                                    absorption_scale=float(rng.choice([0.0, 1.5])), ior=float(rng.uniform(1.1, 1.9)))
                done = 0
            else:
                app.restart()
                done = 0
        assert renders >= 1
        assert app.stats().stackOverflows == 0
