"""SURVEY §8f rows 3 and 4 on the GPU: the reference-GPU-compatible mode (TPT_MODE_REFGPU) against its CPU restatement, and
the reference's compile-time switches DO_MITSUBA_COMPARE / DO_BIG_SCENE as runtime flags against the reference compiled
with those switches (oracle/Makefile builds the variants from an edited temporary copy of the sources)."""
import numpy as np
import pytest

from conftest import bits_differ, rel_l2
from test_oracle import assert_equals_reference, golden_scene

pytestmark = pytest.mark.gpu


# ---- f.4: Mitsuba-compare switches and the 9-sphere scene ---------------------------------------------------------
@pytest.mark.parametrize("variant,big,mitsuba", [("mitsuba", True, True), ("small", False, False), ("small_mitsuba", False, True)])
def test_exact_mode_equals_reference_variant_build(gpu_ctx, libs, oracle, variant, big, mitsuba):
    """Bitwise: exact mode with the runtime switches == the reference compiled with Config.h:25 / Test.cpp:11 edited."""
    w, h = 320, 180
    sph, mats, cam, em = libs.reference_scene(w, h, big_scene=big, mitsuba_compare=mitsuba)
    assert len(sph) == (46 if big else 9)
    gpu_ctx.set_option("mitsuba_compare", 1 if mitsuba else 0)
    try:
        gpu_ctx.set_scene(sph, mats, cam, em)
        for flags in (0, 2):
            obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 0, 3, flags=flags, mitsuba=mitsuba)
            for lanes in (32, 1, 65):
                gpu_ctx.set_option("exact_lanes", lanes)
                buf = np.zeros((h, w, 4), np.float32)
                total, pf = gpu_ctx.draw(0, 3, w, h, buf, flags=flags, mode=0, per_frame=True)
                assert pf == orays, (variant, flags, lanes)
                assert not bits_differ(buf, obuf, pads).any(), (variant, flags, lanes)
            assert_equals_reference(buf, pf, pads, f"{variant}_{w}x{h}_t0.0_flags{flags}_frames0+3")
        # fast mode honours the switches too (statistically): 256 spp vs the restatement at 256 spp
        obuf, orays, _ = oracle.orc_render(sph, mats, cam, w, h, 0, 64, flags=2, mitsuba=mitsuba)
        o2 = obuf.copy()
        oracle.orc_render(sph, mats, cam, w, h, 64, 64, flags=2, mitsuba=mitsuba, buf=o2)
        floor = rel_l2(2.0 * o2.astype(np.float64) - obuf, obuf)
        fb = np.zeros((h, w, 4), np.float32)
        frays = gpu_ctx.draw(0, 64, w, h, fb, flags=2, mode=1)
        assert rel_l2(fb, obuf) < 1.15 * floor, variant
        assert abs(frays / sum(orays) - 1) < 3e-3
    finally:
        gpu_ctx.set_option("exact_lanes", 0)
        gpu_ctx.set_option("mitsuba_compare", 0)


def test_dropin_shim_variants_through_drawtest(libs, oracle):
    """The Test.h drop-in with tpt_shim_set_variant(): UpdateTest/DrawTest of the 9-sphere Mitsuba-compare build."""
    w, h = 256, 144
    libs.set_variant(False, True)
    try:
        libs.InitializeTest()
        libs.set_mode(libs.MODE_EXACT)
        assert libs.GetObjectCount()[0] == 9
        buf = np.zeros((h, w, 4), np.float32)
        rays = []
        for f in range(3):
            libs.UpdateTest(0.0, f, w, h, 2)
            rays.append(libs.DrawTest(0.0, f, w, h, buf, 2))
        sph, mats, cam, em = libs.GetSceneDesc()
        _, _, pads = oracle.orc_render(sph, mats, cam, w, h, 0, 3, flags=2, mitsuba=True)
        assert_equals_reference(buf, rays, pads, "small_mitsuba_256x144_t0.0_flags2_frames0+3")
        libs.ShutdownTest()
    finally:
        libs.set_variant(True, False)


# ---- f.3: reference-GPU-compatible mode ---------------------------------------------------------------------------
def test_refgpu_strict_equals_cpu_restatement(gpu_ctx, libs, oracle):
    """TPT_MODE_REFGPU (per-pixel seeds, analytic samplers, <= 10 segments, lerp blend, alpha 1 — ComputeShader.hlsl) vs
    oracle/refgpu_restate.cpp: bit-identical pixels and ray counts, reference scene / 9-sphere Mitsuba scene / a
    203-sphere runtime scene (count not a multiple of 4: the SIMD padding must stay invisible) / odd sizes."""
    cases = []
    sph, mats, cam, em = golden_scene()
    cases.append((sph, mats, cam, 320, 180, False))
    s9 = libs.reference_scene(320, 180, big_scene=False, mitsuba_compare=True)
    cases.append((s9[0], s9[1], s9[2], 320, 180, True))
    s203 = libs.stress_scene(160, 90, count=203)
    cases.append((s203[0], s203[1], s203[2], 160, 90, False))
    cam_odd = libs.make_camera((0, 2, 3), (0, 0, 0), (0, 1, 0), 60, 97 / 53, 0.02, 3)
    cases.append((sph, mats, cam_odd, 97, 53, False))
    for (s, m, c, w, h, mitsuba) in cases:
        gpu_ctx.set_option("mitsuba_compare", 1 if mitsuba else 0)
        gpu_ctx.set_scene(s, m, c, None)
        for flags, f0 in ((0, 5), (2, 0), (3, 2)):
            init = np.full((h, w, 4), 0.25, np.float32)
            obuf, orays = oracle.rgo_render(s, m, c, w, h, f0, 3, flags=flags, mitsuba=mitsuba, buf=init.copy())
            # one call for the 3 frames
            buf = init.copy()
            total, pf = gpu_ctx.draw(f0, 3, w, h, buf, flags=flags, mode=libs.MODE_REFGPU, per_frame=True)
            assert total == sum(orays), (len(s), flags)
            assert not bits_differ(buf, obuf).any(), (len(s), flags)
            assert (buf[..., 3] == 1).all()                       # ComputeShader.hlsl:392
            # frame by frame, and a row shard
            seq = init.copy()
            r = sum(gpu_ctx.draw(f0 + f, 1, w, h, seq, flags=flags, mode=libs.MODE_REFGPU) for f in range(3))
            assert r == sum(orays) and not bits_differ(seq, obuf).any()
            if h >= 40:
                band = init[3:3 + 4 * (h // 8):4].copy()
                gpu_ctx.draw(f0, 3, w, h, band, flags=flags, mode=libs.MODE_REFGPU, rows=(3, h // 8, 4, 1))
                assert not bits_differ(band, obuf[3:3 + 4 * (h // 8):4]).any()
    gpu_ctx.set_option("mitsuba_compare", 0)


def test_refgpu_fast_matches_strict_statistically(gpu_ctx, libs):
    """GPU-native arithmetic (what a shader compiler emits) vs the strict variant: same per-pixel streams, so the two
    only part where a rounding flips a decision — far below the Monte-Carlo noise; ray counts within 1e-4."""
    w, h = 640, 360
    sph, mats, cam, em = libs.reference_scene(w, h)
    gpu_ctx.set_scene(sph, mats, cam, em)
    a = np.zeros((h, w, 4), np.float32); b = np.zeros((h, w, 4), np.float32)
    ra = gpu_ctx.draw(0, 16, w, h, a, flags=2, mode=libs.MODE_REFGPU)
    rb = gpu_ctx.draw(0, 16, w, h, b, flags=2, mode=libs.MODE_REFGPU_FAST)
    assert abs(ra / rb - 1) < 2e-4
    assert rel_l2(b, a) < 0.25 * 0.194 / np.sqrt(64)
    assert (b[..., 3] == 1).all()
    # and against the bit-exact CPU-path mode: the same image up to Monte-Carlo noise (the estimators differ only in the
    # depth limit and sampler parametrisation)
    e1 = np.zeros((h, w, 4), np.float32)
    gpu_ctx.draw(0, 256, w, h, e1, flags=2, mode=0)
    e2 = e1.copy()
    gpu_ctx.draw(256, 256, w, h, e2, flags=2, mode=0)
    floor = rel_l2(2.0 * e2.astype(np.float64) - e1, e1)
    g = np.zeros((h, w, 4), np.float32)
    gpu_ctx.draw(0, 256, w, h, g, flags=2, mode=libs.MODE_REFGPU_FAST)
    assert rel_l2(g, e1) < 1.15 * floor


def test_device_powf_cuberoot_equals_glibc(gpu_ctx, oracle):
    x = (np.arange(1 << 24, dtype=np.uint32).astype(np.float32) / np.float32(16777216.0))
    d = gpu_ctx.debug_libm(3, x)
    g = oracle.libm_eval("powf", x, np.float32(1.0) / np.float32(3.0))
    assert (d.view(np.uint32) == g.view(np.uint32)).all()
