"""Parity tests proper: the CUDA exact mode, called through the C-ABI / the Test.h drop-in, against the oracle
and the golden vectors. Bar: bit-identical pixels and identical ray counts (integer work and float work alike —
the exact mode replays the reference's arithmetic op by op)."""
import json
import os

import numpy as np
import pytest

from conftest import bits_differ
from test_oracle import GOLD, PARITY, assert_equals_reference, golden_scene

pytestmark = pytest.mark.gpu


def test_device_libm_equals_glibc(gpu_ctx, oracle):
    """Device sinf/cosf over all 2^24 arguments the path can produce (Maths.cpp:42, Test.cpp:115) and powf(x,5)
    over 2^24 random bit patterns plus the edge cases, against the libm the reference links."""
    k = np.arange(1 << 24, dtype=np.uint32)
    a = (k.astype(np.float32) / np.float32(16777216.0)) * np.float32(2.0) * np.float32(3.1415926)
    for fn, name in ((0, "sinf"), (1, "cosf")):
        d = gpu_ctx.debug_libm(fn, a); g = oracle.libm_eval(name, a)
        assert (d.view(np.uint32) == g.view(np.uint32)).all(), name
    rng = np.random.default_rng(7)
    x = rng.integers(0, 1 << 32, 1 << 24, dtype=np.uint64).astype(np.uint32).view(np.float32)
    edge = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.17549435e-38, 3.4e38, 0.5, 2.0 ** -24,
                     2.0 ** -30, -0.5, 2.5], np.float32)
    x = np.concatenate([x, edge, np.linspace(-1, 3, 100001, dtype=np.float32)])
    d = gpu_ctx.debug_libm(2, x); g = oracle.libm_eval("powf", x, 5.0)
    same = (d.view(np.uint32) == g.view(np.uint32)) | (np.isnan(d) & np.isnan(g))
    assert same.all()


def test_golden_vectors(gpu_ctx):
    g = np.load(os.path.join(GOLD, "ref_192x108_f0-3.npz"))
    sph, mats, cam, em = golden_scene()
    gpu_ctx.set_scene(sph, mats, cam, em)
    for lanes in (32, 8, 9, 1, 2, 64, 65, 70, 0):
        gpu_ctx.set_option("exact_lanes", lanes)
        # frame by frame (numFrames = 1: blend fused into the trace kernel)
        buf = np.zeros((108, 192, 4), np.float32)
        rays = [gpu_ctx.draw(f, 1, 192, 108, buf, flags=2, mode=0) for f in range(4)]
        assert rays == [int(r) for r in g["rays"]]
        assert not bits_differ(buf, g["image"]).any()
        # one call for the 4 frames (scratch + resolve kernel)
        buf = np.zeros((108, 192, 4), np.float32)
        total, per_frame = gpu_ctx.draw(0, 4, 192, 108, buf, flags=2, mode=0, per_frame=True)
        assert per_frame == [int(r) for r in g["rays"]] and total == int(g["rays"].sum())
        assert not bits_differ(buf, g["image"]).any()
    gpu_ctx.set_option("exact_lanes", 0)


def test_dropin_drawtest_full_size_vs_golden_counts_and_reference(libs):
    """The BASELINE configuration (46 spheres, 1280x720, 4 spp) through the drop-in's UpdateTest/DrawTest."""
    counts = json.load(open(os.path.join(GOLD, "ref_counts.json")))["1280x720_flags0_frames0-5"]
    w, h = 1280, 720
    libs.reset_scene()
    libs.InitializeTest()
    libs.set_mode(libs.MODE_EXACT)
    buf = np.zeros((h, w, 4), np.float32)
    rays = []
    for f in range(3):
        libs.UpdateTest(0.0, f, w, h, 0)
        rays.append(libs.DrawTest(0.0, f, w, h, buf, 0))
    assert rays == counts[:3]                                    # 16 809 105 / 16 822 947 / 16 818 090
    assert (buf[..., 3] == 0).all()                              # alpha untouched (Maths.h:38)
    assert_equals_reference(buf, rays, [], "stock_1280x720_t0.0_flags0_frames0+3")
    libs.ShutdownTest()


def test_progressive_prev_semantics(gpu_ctx, oracle):
    """`prev` is an input: non-zero, NaN and Inf pixels, alpha preserved (Test.cpp:293-295)."""
    sph, mats, cam, em = golden_scene()
    gpu_ctx.set_scene(sph, mats, cam, em)
    w, h = 192, 108
    rng = np.random.default_rng(3)
    init = rng.random((h, w, 4), dtype=np.float32)
    init[5, 7, 0] = np.nan; init[6, 8, 1] = np.inf; init[:, :, 3] = 0.75
    for flags in (0, 2):
        a = init.copy(); b = init.copy()
        obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 3, 2, flags=flags, buf=a)
        rays = gpu_ctx.draw(3, 1, w, h, b, flags=flags, mode=0) + gpu_ctx.draw(4, 1, w, h, b, flags=flags, mode=0)
        assert rays == sum(orays)
        assert not bits_differ(b, obuf, pads).any()
        assert (b[..., 3] == np.float32(0.75)).all()
        c = init.copy()
        gpu_ctx.draw(3, 2, w, h, c, flags=flags, mode=0)
        assert not bits_differ(c, obuf, pads).any()


def test_row_sharding_is_exact(gpu_ctx):
    """Rows are independent units (Test.cpp:278-280): any band / interleave of rows reproduces the same pixels."""
    sph, mats, cam, em = golden_scene()
    gpu_ctx.set_scene(sph, mats, cam, em)
    w, h = 192, 108
    full = np.zeros((h, w, 4), np.float32)
    total = gpu_ctx.draw(0, 2, w, h, full, flags=2, mode=0)
    # two contiguous bands into the full image
    img = np.zeros((h, w, 4), np.float32)
    r = gpu_ctx.draw(0, 2, w, h, img, flags=2, mode=0, rows=(0, 50, 1, 0)) + \
        gpu_ctx.draw(0, 2, w, h, img, flags=2, mode=0, rows=(50, 58, 1, 0))
    assert r == total and not bits_differ(img, full).any()
    # 4-way interleave, packed bands (what the multi-GPU path does per rank)
    img = np.zeros((h, w, 4), np.float32)
    r = 0
    for rank in range(4):
        band = np.zeros((h // 4, w, 4), np.float32)
        r += gpu_ctx.draw(0, 2, w, h, band, flags=2, mode=0, rows=(rank, h // 4, 4, 1))
        img[rank::4] = band
    assert r == total and not bits_differ(img, full).any()


def test_animated_scene(libs, gpu_ctx, oracle):
    sph, mats, cam, em = libs.reference_scene(320, 180, time=2.5, flags=3)
    gpu_ctx.set_scene(sph, mats, cam, em)
    obuf, orays, pads = oracle.orc_render(sph, mats, cam, 320, 180, 10, 3, flags=3)
    buf = np.zeros((180, 320, 4), np.float32)
    total, pf = gpu_ctx.draw(10, 3, 320, 180, buf, flags=3, mode=0, per_frame=True)
    assert pf == orays and not bits_differ(buf, obuf, pads).any()


def test_runtime_scenes_against_restatement(libs, gpu_ctx, oracle):
    """Scenes the reference cannot run (static array, Test.cpp:13-64): counts that are / are not multiples of 4,
    a single sphere, no lights, many lights, the 4096-sphere stress scene (BASELINE configs[4]) at a small size."""
    cases = []
    cam = libs.make_camera((0, 1, 4), (0, 0, 0), (0, 1, 0), 45, 2.0, 0.05, 4)
    for n in (1, 2, 5, 7):
        sph = np.zeros(n, libs.SPHERE_DTYPE); mats = np.zeros(n, libs.MATERIAL_DTYPE)
        for i in range(n):
            sph[i] = ((i - n / 2, 0, 0), 0.45, 0)
            mats[i] = (i % 3, (0.7, 0.6, 0.5), (4, 4, 4) if i == 1 else (0, 0, 0), 0.1, 1.5)
        cases.append((sph, mats, cam, 64, 32))
    s203 = libs.stress_scene(160, 90, count=203)
    cases.append((s203[0], s203[1], s203[2], 160, 90))
    s4096 = libs.stress_scene(96, 54, count=4096)
    cases.append((s4096[0], s4096[1], s4096[2], 96, 54))
    for (sph, mats, cam, w, h) in cases:
        gpu_ctx.set_scene(sph, mats, cam, None)
        obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 0, 2, flags=2)
        for lanes in (32, 1, 64, 65, 70):
            gpu_ctx.set_option("exact_lanes", lanes)
            buf = np.zeros((h, w, 4), np.float32)
            total, pf = gpu_ctx.draw(0, 2, w, h, buf, flags=2, mode=0, per_frame=True)
            assert pf == orays, (len(sph), lanes)
            assert not bits_differ(buf, obuf, pads).any(), (len(sph), lanes)
    gpu_ctx.set_option("exact_lanes", 0)


def test_padded_sphere_hit_frame(gpu_ctx):
    """Frame 28 at 1280x720 holds a ray that hits a padded impossible sphere (reference UB): ray counts must still
    equal the reference's, and every pixel except that one must be bit-identical."""
    sph, mats, cam, em = golden_scene()
    gpu_ctx.set_scene(sph, mats, cam, em)
    buf = np.zeros((720, 1280, 4), np.float32)
    rays = gpu_ctx.draw(28, 1, 1280, 720, buf, flags=0, mode=0)
    assert rays == 16813074
    assert_equals_reference(buf, [rays], [(180, 436, 28)], "stock_1280x720_t0.0_flags0_frames28+1")


def test_4k_frame_ray_count(gpu_ctx, libs):
    """3840x2160 frame 0 = 151 330 258 rays (golden, SURVEY §9.9)."""
    counts = json.load(open(os.path.join(GOLD, "ref_counts.json")))
    sph, mats, cam, em = libs.reference_scene(3840, 2160)
    gpu_ctx.set_scene(sph, mats, cam, em)
    import torch
    buf = torch.zeros((2160, 3840, 4), dtype=torch.float32, device="cuda")
    rays = gpu_ctx.draw(0, 1, 3840, 2160, buf, flags=0, mode=0)
    assert [rays] == counts["3840x2160_flags0_frame0"]


def test_headless_shell_same_output_as_reference_build(libs):
    """One shell source (toypathtracer_b200/csrc/headless_main.cpp, the shape of Cpp/Emscripten/main.cpp:46-61) built
    twice — against the unmodified reference sources (oracle/_ref/ref_headless, its output recorded in
    tests/golden/ref_parity.json) and against the drop-in (toypathtracer_b200/tpt_headless) — must print the same ray
    counts and the same backbuffer checksum."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ours = os.path.join(root, "toypathtracer_b200", "tpt_headless")
    ref = PARITY["headless"]
    env = dict(os.environ, TPT_MODE="exact")
    a = subprocess.run([ours] + ref["args"], capture_output=True, text=True, env=env, timeout=300)
    assert a.returncode == 0, a.stderr
    keep = lambda out: [l for l in out.splitlines() if l.startswith("frame") or l.startswith("checksum")]
    assert keep(a.stdout) == ref["lines"] and len(ref["lines"]) == 5


def test_odd_sizes_and_single_row(gpu_ctx, oracle):
    """Ragged shapes: odd width/height, one row, one column — exact mode vs the CPU restatement, all lane configs."""
    sph, mats, cam0, em = golden_scene()
    import toypathtracer_b200 as tpt
    for (w, h) in [(97, 53), (33, 1), (1, 19), (130, 7)]:
        cam = tpt.make_camera((0, 2, 3), (0, 0, 0), (0, 1, 0), 60, w / h, 0.02, 3)
        gpu_ctx.set_scene(sph, mats, cam, em)
        obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 2, 2, flags=2)
        for lanes in (32, 8, 1, 64, 65, 70):
            gpu_ctx.set_option("exact_lanes", lanes)
            buf = np.zeros((h, w, 4), np.float32)
            total, pf = gpu_ctx.draw(2, 2, w, h, buf, flags=2, mode=0, per_frame=True)
            assert pf == orays, (w, h, lanes)
            assert not bits_differ(buf, obuf, pads).any(), (w, h, lanes)
    gpu_ctx.set_option("exact_lanes", 0)


def test_error_behaviour(libs):
    """Every C-ABI call returns a status; bad arguments are refused with a message instead of rendering garbage."""
    ctx = libs.Context(0)
    buf = np.zeros((8, 8, 4), np.float32)
    with pytest.raises(libs.TptError, match="no scene"):
        ctx.draw(0, 1, 8, 8, buf)
    sph, mats, cam, em = golden_scene()
    ctx.set_scene(sph, mats, cam, em)
    with pytest.raises(libs.TptError, match="rows outside"):
        ctx.draw(0, 1, 8, 8, buf, rows=(4, 8, 1, 0))
    with pytest.raises(libs.TptError, match="unknown mode"):
        ctx.draw(0, 1, 8, 8, buf, mode=7)
    with pytest.raises(libs.TptError, match="bad arguments"):
        ctx.draw(0, 0, 8, 8, buf)
    with pytest.raises(libs.TptError):
        ctx.set_spp(0)
    with pytest.raises(libs.TptError):
        ctx.set_option("no_such_option", 1)
    with pytest.raises(libs.TptError):
        ctx.set_scene(sph[:0], mats[:0], cam, None)
    assert ctx.draw(0, 1, 8, 8, buf) > 0           # still usable after the refusals
    ctx.close()


def test_frame_batches_limited_by_scratch(gpu_ctx, oracle):
    """numFrames larger than what the per-frame scratch may hold: the exact mode renders in several batches and the
    progressive lerp still runs in reference order."""
    sph, mats, cam, em = golden_scene()
    gpu_ctx.set_scene(sph, mats, cam, em)
    w, h = 192, 108
    obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 0, 7, flags=2)
    gpu_ctx.set_option("max_scratch_mb", 16)          # 192*108*16 B = 0.33 MB per frame -> plenty; then squeeze:
    buf = np.zeros((h, w, 4), np.float32)
    total, pf = gpu_ctx.draw(0, 7, w, h, buf, flags=2, mode=0, per_frame=True)
    assert pf == orays and not bits_differ(buf, obuf, pads).any()
    big_w, big_h = 1024, 1024                          # 16 MB per frame -> exactly one frame per batch at 16 MB
    cam2 = __import__("toypathtracer_b200").make_camera((0, 2, 3), (0, 0, 0), (0, 1, 0), 60, 1.0, 0.02, 3)
    gpu_ctx.set_scene(sph, mats, cam2, em)
    o2, r2, p2 = oracle.orc_render(sph, mats, cam2, big_w, big_h, 0, 3, flags=2)
    b2 = np.zeros((big_h, big_w, 4), np.float32)
    t2, pf2 = gpu_ctx.draw(0, 3, big_w, big_h, b2, flags=2, mode=0, per_frame=True)
    gpu_ctx.set_option("max_scratch_mb", 8192)
    assert pf2 == r2 and not bits_differ(b2, o2, p2).any()


def test_adaptive_frame_lookahead(libs, oracle):
    """"exact_lookahead" = -1 (the drop-in's default): the window doubles (1, 2, 4, 8, 16) while the caller keeps asking for
    the next frame and falls back to 1 after any break in the sequence; pixels and per-call ray counts stay those of
    frame-by-frame draws."""
    ctx = libs.Context(0)
    sph, mats, cam, em = golden_scene()
    w, h = 192, 108
    ctx.set_scene(sph, mats, cam, em)
    n = 40
    ref = np.zeros((h, w, 4), np.float32)
    ref_rays = [ctx.draw(f, 1, w, h, ref, flags=2, mode=0) for f in range(n)]
    ctx.set_option("exact_lookahead", -1)
    buf = np.zeros((h, w, 4), np.float32)
    rays, launches = [], []
    for f in range(n):
        ctx.set_scene(sph, mats, cam, em)
        rays.append(ctx.draw(f, 1, w, h, buf, flags=2, mode=0))
        launches.append(ctx.last_launch_count())
    assert rays == ref_rays and not bits_differ(buf, ref).any()
    # trace launches happen at frames 0, 1, 3, 7, 15, 31 (windows of 1, 2, 4, 8, 16, 16): a miss that opens a window of more
    # than one frame is trace + resolve + fold, a window of one is trace + fold, a hit resolve + fold
    misses = [f for f in range(n) if launches[f] == 3 or f == 0]
    assert misses == [0, 1, 3, 7, 15, 31], (misses, launches)
    # a jump in the frame sequence and a camera change both restart at a window of one; results stay exact
    cam2 = cam.copy(); cam2.view(np.float32)[0] += 0.25
    a = np.zeros((h, w, 4), np.float32); b = np.zeros((h, w, 4), np.float32)
    seq = [(50, cam), (51, cam), (52, cam), (60, cam), (61, cam2), (62, cam2), (63, cam2)]
    ctx.set_option("exact_lookahead", 0)
    ra = []
    for f, c in seq:
        ctx.set_scene(sph, mats, c, em); ra.append(ctx.draw(f, 1, w, h, a, flags=2, mode=0))
    ctx.set_option("exact_lookahead", -1)
    rb = []
    for f, c in seq:
        ctx.set_scene(sph, mats, c, em); rb.append(ctx.draw(f, 1, w, h, b, flags=2, mode=0))
    assert ra == rb and not bits_differ(a, b).any()
    ctx.close()


def test_frame_lookahead_is_bit_identical(libs, oracle):
    """"exact_lookahead": a miss traces L frames in one launch, the following one-frame calls only blend their cached
    frame — same pixels, same per-frame ray counts as frame-by-frame draws; scene/camera/size changes invalidate."""
    ctx = libs.Context(0)
    sph, mats, cam, em = golden_scene()
    w, h = 192, 108
    ctx.set_scene(sph, mats, cam, em)
    ref = np.zeros((h, w, 4), np.float32)
    ref_rays = [ctx.draw(f, 1, w, h, ref, flags=2, mode=0) for f in range(13)]
    ctx.set_option("exact_lookahead", 5)
    buf = np.zeros((h, w, 4), np.float32)
    rays = []
    launches = []
    for f in range(13):
        ctx.set_scene(sph, mats, cam, em)                         # a shell calls UpdateTest every frame: same bytes, cache stays
        rays.append(ctx.draw(f, 1, w, h, buf, flags=2, mode=0))
        launches.append(ctx.last_launch_count())
    assert rays == ref_rays and not bits_differ(buf, ref).any()
    assert launches[0] == 3 and launches[1] == 2 and launches[5] == 3     # miss: trace + resolve + fold; hit: resolve + fold
    # a different scene mid-way: the cached frames of the old scene must not be used
    m2 = mats.copy(); m2.view(np.float32).reshape(-1, 9)[0, 1:4] = (0.2, 0.9, 0.2)
    a = np.zeros((h, w, 4), np.float32); b = np.zeros((h, w, 4), np.float32)
    ctx.set_option("exact_lookahead", 0)
    ctx.set_scene(sph, mats, cam, em); ctx.draw(20, 1, w, h, a, flags=0, mode=0)
    ctx.set_scene(sph, m2, cam, em); ra = ctx.draw(21, 1, w, h, a, flags=0, mode=0)
    ctx.set_option("exact_lookahead", 4)
    ctx.set_scene(sph, mats, cam, em); ctx.draw(20, 1, w, h, b, flags=0, mode=0)
    ctx.set_scene(sph, m2, cam, em); rb = ctx.draw(21, 1, w, h, b, flags=0, mode=0)
    assert ra == rb and not bits_differ(a, b).any()
    # non-progressive flags, a row shard, and an animated draw (never cached) through the same context
    c1 = np.zeros((h // 4, w, 4), np.float32); c2 = np.zeros((h // 4, w, 4), np.float32)
    r1 = [ctx.draw(f, 1, w, h, c1, flags=0, mode=0, rows=(1, h // 4, 4, 1)) for f in (30, 31, 32)]
    ctx.set_option("exact_lookahead", 0)
    r2 = [ctx.draw(f, 1, w, h, c2, flags=0, mode=0, rows=(1, h // 4, 4, 1)) for f in (30, 31, 32)]
    assert r1 == r2 and not bits_differ(c1, c2).any()
    ctx.close()
