"""CPU tests of the any-hit callbacks of include/rtc_device.cuh (rtc_device_trace_closest_anyhit / rtc_device_trace_any_anyhit).

The header is compiled by g++ with a recording callback (tests/native/device_anyhit_host.cpp) and held, on the fuzz scenes and the
degenerate soups of tests/test_cpu_trace_masks.py, with a random mask and flag set per ray, to
  * (a) brute force with the same decision (tests/native/oracle_anyhit.c), bit for bit, for every pure predicate;
  * (b) the brute-force candidate list: an any query that ignores everything offers every candidate exactly once;
  * (c) rtc_device_trace_closest / _any, when the callback always accepts;
  * accept-and-end: the result is the candidate the callback ended on, with that candidate's exact fields;
  * self-skip: brute force without the triangle the ray starts on;
  * refusals: no callback call and no scene read.
nvcc compiles the user kernels for sm_100a with -Iinclude alone (default and -fmad=false), two -rdc=true units with callbacks
device-link, and the callback parameter changes no instruction of the library's kernels or of the plain device queries."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import helpers as H
from device_anyhit import (ACCEPT, ALPHA, FRONT, IGNORE, NOT_SELF, brute_any, brute_candidates, brute_closest, host_constants, host_trace,
                           record_keys)
from test_cpu_device_trace import ARCH, CSRC, INCLUDE, KERNELS, NATIVE, NVCC, constants, normalized_sass, per_ray_filters, ptxas_report
from test_cpu_trace_masks import fuzz_scene, soup_scene

ANYHIT_KERNELS = os.path.join(NATIVE, "device_anyhit_kernels.cu")
ALPHA_TRANSPARENT = 96                 # of 256 triangles transparent; a quarter of the rest checkered


def scenes():
    return [("fuzz", s) for s in range(3)] + [("soup", s) for s in (1, 2, 3)]


def load(kind, seed, tmp_path):
    """(export, MaskedScene, rays, closer) for a fuzz scene or a degenerate soup"""
    if kind == "fuzz":
        app, export, ref = fuzz_scene(tmp_path, seed)
        return export, ref, H.random_rays(2000, seed=seed, lo=(-5, 0.05, -5), hi=(5, 4, 5)), app.close
    export, ref, rays = soup_scene(seed)
    return export, ref, rays[::2].copy(), ref.close


@pytest.fixture(params=scenes(), ids=lambda p: "%s%d" % p)
def scene(request, built, tmp_path):
    kind, seed = request.param
    export, ref, rays, close = load(kind, seed, tmp_path)
    rng = np.random.default_rng(900 + seed + (50 if kind == "soup" else 0))
    masks = rng.integers(0, 256, size=len(export["instance_gas"])).astype(np.uint8)
    ref.set_instance_masks(0, masks)
    ray_masks, ray_flags = per_ray_filters(rng, len(rays))
    yield dict(export=export, ref=ref, rays=rays, masks=masks, ray_masks=ray_masks, ray_flags=ray_flags, rng=rng)
    close()


def self_params(s):
    """per ray, an (instance, primitive) to skip: the plain closest hit of the ray, so the skip changes the answer"""
    got = host_trace(s["export"], s["masks"], s["rays"], s["ray_masks"], s["ray_flags"], mode="plain_closest")["out"]
    return got["inst"], got["prim"]


@pytest.mark.parametrize("pred", [ACCEPT, ALPHA, FRONT, NOT_SELF], ids=["accept", "alpha", "front", "not_self"])
def test_property_a_pure_predicates_equal_brute_force(scene, pred):
    s = scene
    p0, p1 = (self_params(s) if pred == NOT_SELF else (ALPHA_TRANSPARENT if pred == ALPHA else 0, 0))
    args = (s["export"], s["masks"], s["rays"], s["ray_masks"], s["ray_flags"])
    got = host_trace(*args, mode="closest", pred=pred, p0=p0, p1=p1)
    assert (got["status"] == 0).all() and got["duplicates"] == 0
    want = brute_closest(s["ref"], s["rays"], s["ray_masks"], s["ray_flags"], pred, p0, p1)
    assert H.hits_equal(got["out"], want)
    got_any = host_trace(*args, mode="any", pred=pred, p0=p0, p1=p1)
    assert (got_any["status"] == 0).all() and got_any["duplicates"] == 0
    assert np.array_equal(got_any["out"].astype(bool), brute_any(s["ref"], s["rays"], s["ray_masks"], s["ray_flags"], pred, p0, p1).astype(bool))
    assert (want["inst"] != 0xffffffff).mean() > 0.02
    if pred != ACCEPT:
        plain = host_trace(*args, mode="plain_closest")["out"]
        assert not H.hits_equal(plain, want)                  # the predicate changes some answers


def test_property_b_ignoring_any_query_offers_every_candidate_once(scene):
    s = scene
    got = host_trace(s["export"], s["masks"], s["rays"], s["ray_masks"], s["ray_flags"], mode="any", pred=IGNORE)
    assert (got["status"] == 0).all() and (got["out"] == 0).all() and got["duplicates"] == 0
    want, counts = brute_candidates(s["ref"], s["rays"], s["ray_masks"], s["ray_flags"])
    assert counts.max() <= 256 and counts.sum() > len(s["rays"]) // 10
    assert np.array_equal(got["calls"], counts) and np.array_equal(got["digest"][:, 0], counts)
    for i in np.flatnonzero(counts):
        assert record_keys(got["records"][i], got["calls"][i]) == record_keys(want[i], counts[i]), i


def test_property_c_always_accept_equals_the_plain_queries(scene):
    s = scene
    args = (s["export"], s["masks"], s["rays"], s["ray_masks"], s["ray_flags"])
    got, plain = host_trace(*args, mode="closest"), host_trace(*args, mode="plain_closest")
    assert (got["status"] == 0).all() and H.hits_equal(got["out"], plain["out"])
    assert (plain["calls"] == 0).all() and (got["calls"] > 0).any()
    # each accepted call shrinks the interval: the last call of a ray is its hit, with the hit's exact fields
    for i in np.flatnonzero(got["calls"]):
        r, h = got["records"][i][got["calls"][i] - 1], got["out"][i]
        assert (r["t"], r["u"], r["v"], r["inst"], r["prim"]) == (h["t"], h["u"], h["v"], h["inst"], h["prim"])
    got_any, plain_any = host_trace(*args, mode="any"), host_trace(*args, mode="plain_any")
    assert np.array_equal(got_any["out"], plain_any["out"]) and (got_any["calls"] == got_any["out"]).all()


def test_accept_and_end_returns_the_candidate_it_ended_on(scene):
    s = scene
    args = (s["export"], s["masks"], s["rays"], s["ray_masks"], s["ray_flags"])
    got = host_trace(*args, mode="closest", pred=ALPHA, p0=ALPHA_TRANSPARENT, end=True)
    assert (got["status"] == 0).all() and got["duplicates"] == 0
    hits = got["out"]
    found = hits["inst"] != 0xffffffff
    assert found.mean() > 0.02
    best = brute_closest(s["ref"], s["rays"], s["ray_masks"], s["ray_flags"], ALPHA, ALPHA_TRANSPARENT)
    assert np.array_equal(found, best["inst"] != 0xffffffff)         # ends exactly when some candidate is opaque
    for i in np.flatnonzero(found):
        r = got["records"][i][got["calls"][i] - 1]
        assert (r["t"], r["u"], r["v"], r["inst"], r["prim"]) == tuple(hits[i][["t", "u", "v", "inst", "prim"]].tolist())
        assert r["t"] >= best["t"][i]                     # which accepted candidate it ends on depends on the tree
        assert r["inst"] != 0xffffffff and 0 < got["calls"][i]


def test_self_skip_equals_brute_force_without_that_triangle(scene):
    s = scene
    rays, export, masks = s["rays"], s["export"], s["masks"]
    first = host_trace(export, masks, rays, s["ray_masks"], s["ray_flags"], mode="plain_closest")["out"]
    hit = first["inst"] != 0xffffffff
    sec = rays[hit].copy()
    t = first["t"][hit].astype(np.float32)
    for c in "xyz":
        sec["o" + c] = (sec["o" + c] + t * sec["d" + c]).astype(np.float32)
    rng = s["rng"]
    d = rng.normal(size=(len(sec), 3)).astype(np.float32)
    sec["dx"], sec["dy"], sec["dz"] = d[:, 0], d[:, 1], d[:, 2]
    sec["tmin"], sec["tmax"] = 0.0, 1e27
    rm, rf = s["ray_masks"][hit], s["ray_flags"][hit]
    p0, p1 = first["inst"][hit], first["prim"][hit]
    got = host_trace(export, masks, sec, rm, rf, mode="closest", pred=NOT_SELF, p0=p0, p1=p1)
    want = brute_closest(s["ref"], sec, rm, rf, NOT_SELF, p0, p1)
    assert (got["status"] == 0).all() and H.hits_equal(got["out"], want)
    assert not ((want["inst"] == p0) & (want["prim"] == p1)).any()


def test_refusals_call_nothing_and_read_nothing(built):
    export, _, rays = soup_scene(1)
    k = constants()
    rays = rays[:500]
    masks = np.full(len(export["instance_gas"]), 0xFF, dtype=np.uint8)
    ok = host_trace(export, masks, rays, mode="any", pred=IGNORE)
    assert (ok["status"] == k["OK"]).all() and ok["reads"] > 0 and ok["calls"].sum() > 0
    cases = [("mask 0x100", dict(ray_masks=0x100), k["BAD_ARGUMENT"]), ("flag 4", dict(ray_flags=4), k["BAD_ARGUMENT"]),
             ("usable 0", dict(usable=0), k["SCENE_UNUSABLE"]), ("abi", dict(abi=k["ABI"] ^ 1), k["ABI_MISMATCH"])]
    for label, kw, want in cases:
        for mode in ("closest", "any"):
            got = host_trace(export, masks, rays, mode=mode, pred=IGNORE, **kw)
            assert (got["status"] == want).all() and got["reads"] == 0 and (got["calls"] == 0).all(), (label, mode)
            if mode == "any":
                assert (got["out"] == 0).all(), label
            else:
                assert (got["out"]["inst"] == 0xffffffff).all() and (got["out"]["t"] == -1).all(), label
    empty = rays.copy()
    empty["tmax"] = empty["tmin"]
    got = host_trace(export, masks, empty, mode="any", pred=IGNORE)
    assert (got["status"] == k["OK"]).all() and (got["calls"] == 0).all() and got["reads"] == 0
    c = host_constants()
    assert (c["IGNORE"], c["ACCEPT"], c["ACCEPT_AND_END"], c["CANDIDATE_BYTES"]) == (0, 1, 2, 24)


@pytest.mark.parametrize("flags", [[], ["-fmad=false"]], ids=["default", "fmad-false"])
def test_kernels_compile_for_sm100a_with_the_include_directory_alone(tmp_path, flags):
    r = subprocess.run([NVCC, "-O3", "-std=c++17"] + ARCH + flags + ["-I" + INCLUDE, "-Xptxas", "-v", "-c", ANYHIT_KERNELS,
                        "-o", str(tmp_path / "k.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    report = ptxas_report(r.stderr)
    kernels = {k: v for k, v in report.items() if re.search(r"k_(anyhit|lean|alpha_restart|self_skip)", k)}
    assert len(kernels) == 13
    for name, (regs, stack, spills) in sorted(kernels.items()):
        print("%-12s %-100s %3d registers, %3d B stack, %3d B spilled" % (" ".join(flags) or "default", name, regs, stack, spills))
        if "k_anyhitILb0ELb1E" not in name and "k_anyhitILb1ELb1E" not in name:       # all but the 1024-thread builds
            assert spills == 0 and stack == 320, name


def test_two_translation_units_with_callbacks_device_link(tmp_path):
    srcs = {"a.cu": "__global__ void ka(uint64_t top, const rtc_ray* r, rtc_hit* h, uint32_t skip) { rtc_device_trace_closest_anyhit(top, "
                    "r[threadIdx.x], h + threadIdx.x, [&](const rtc_candidate& c) { return c.prim != skip; }); }",
            "b.cu": "__global__ void kb(uint64_t top, const rtc_ray* r, uint32_t* o, uint32_t* n) { uint32_t k = 0; rtc_device_trace_any_anyhit("
                    "top, r[threadIdx.x], o + threadIdx.x, [&](const rtc_candidate& c) { ++k; return c.frontFacing ? RTC_ANYHIT_ACCEPT_AND_END "
                    ": RTC_ANYHIT_IGNORE; }, 1u, RTC_RAY_CULL_BACK_FACING); n[threadIdx.x] = k; }"}
    objs = []
    for name, body in srcs.items():
        src = tmp_path / name
        src.write_text('#include "rtc_device.cuh"\n' + body + "\n")
        obj = str(tmp_path / (name + ".o"))
        subprocess.run([NVCC, "-std=c++17"] + ARCH + ["-rdc=true", "-I" + INCLUDE, "-c", str(src), "-o", obj], check=True)
        objs.append(obj)
    r = subprocess.run([NVCC] + ARCH + ["-dlink"] + objs + ["-o", str(tmp_path / "link.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def strip_callback(root):
    """the tree under `root` (include/ and tweeker_raytracer_b200/csrc/) with the ANYHIT parameter removed from the traversal"""
    trace = root / "tweeker_raytracer_b200" / "csrc" / "trace.cuh"
    text = trace.read_text()
    subs = [(r", class ANYHIT = TraceNoAnyHit>", ">", 1),
            (r"  static constexpr bool HAS_ANYHIT[^\n]*\n  // ignore is[^\n]*\n  static_assert[^\n]*\n", "", 1),
            (r"          if constexpr \(HAS_ANYHIT\)\n          \{\n.*?\n            continue;\n          \}\n", "", 1),
            (r", ANYHIT\* anyHit = nullptr\)", ")", 2),
            (r"leaf_phase\(sc, filt, anyHit\)", "leaf_phase(sc, filt)", 2)]
    for pat, rep, count in subs:
        text, n = re.subn(pat, rep, text, flags=re.S)
        assert n == count, pat
    assert not re.search(r"class ANYHIT|HAS_ANYHIT|ANYHIT\*|, anyHit\)", text)
    trace.write_text(text)
    header = root / "include" / "rtc_device.cuh"
    text = header.read_text()
    for old, new in (("Traversal<ANY, false, 1, false, 0, true, ANYHIT>", "Traversal<ANY, false, 1, false, 0, true>"),
                     ("tr.step(sc, filt, anyHit)", "tr.step(sc, filt)")):
        assert text.count(old) == 1, old
        text = text.replace(old, new)
    header.write_text(text)


def test_callback_parameter_changes_no_kernel(built, tmp_path):
    """kernels_trace.o, kernels_shade.o (as built) and the plain device queries of device_trace_kernels.cu equal builds against a
    traversal without the callback parameter, instruction for instruction"""
    plain = tmp_path / "plain"
    shutil.copytree(INCLUDE, plain / "include")
    shutil.copytree(CSRC, plain / "tweeker_raytracer_b200" / "csrc")
    strip_callback(plain)
    src = plain / "tweeker_raytracer_b200" / "csrc"
    common = [NVCC, "-O3", "-std=c++17"] + ARCH
    lib = common + ["-lineinfo", "-Xcompiler", "-fPIC", "-I" + str(plain / "include"), "-I" + str(src)]
    jobs = {"kernels_trace": subprocess.Popen(lib + ["-c", str(src / "kernels_trace.cu"), "-o", str(tmp_path / "kernels_trace.o")]),
            "kernels_shade": subprocess.Popen(lib + ["-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-c", str(src / "kernels_shade.cu"),
                                                     "-o", str(tmp_path / "kernels_shade.o")])}
    for variant, flags in (("default", []), ("fmad", ["-fmad=false"])):
        for tree, inc in (("new", INCLUDE), ("plain", str(plain / "include"))):
            jobs["dt_%s_%s" % (variant, tree)] = subprocess.Popen(common + flags + ["-I" + inc, "-c", KERNELS, "-o",
                                                                                   str(tmp_path / ("dt_%s_%s.o" % (variant, tree)))])
    for name, job in jobs.items():
        assert job.wait() == 0, name
    for name in ("kernels_trace", "kernels_shade"):
        built_obj = os.path.join(H.ROOT, "tweeker_raytracer_b200", "lib", name + ".o")
        assert normalized_sass(built_obj) == normalized_sass(str(tmp_path / (name + ".o"))), name
    for variant in ("default", "fmad"):
        assert normalized_sass(str(tmp_path / ("dt_%s_new.o" % variant))) == normalized_sass(str(tmp_path / ("dt_%s_plain.o" % variant))), variant
