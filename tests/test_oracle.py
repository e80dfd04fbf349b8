"""Pins the oracle: the CPU restatement (oracle/restate.cpp) against the committed golden vectors generated from
the unmodified reference (tests/golden/make_golden.py, make_golden_parity.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import bits_differ

GOLD = os.path.join(os.path.dirname(__file__), "golden")
PARITY = json.load(open(os.path.join(GOLD, "ref_parity.json")))


def golden_scene():
    g = np.load(os.path.join(GOLD, "scene46_1280x720.npz"))
    return g["spheres"], g["materials"].view(np.float32), g["camera"], g["emissives"]


def parity_scene(key):
    """The reference's GetSceneDesc export recorded under `key` (variant_WxH_tTIME_flagsFLAGS)."""
    g = np.load(os.path.join(GOLD, "ref_parity_scenes.npz"))
    return g[f"{key}/spheres"], g[f"{key}/materials"].view(np.float32), g[f"{key}/camera"], g[f"{key}/emissives"]


def parity_render(key):
    """The reference's render recorded under `key`: {"rays", "pads", "sha256_pads_zeroed"}."""
    r = PARITY["renders"][key]
    return dict(r, pads=[tuple(p) for p in r["pads"]])


def image_hash(img, pads):
    """sha256 of the float32 RGBA bytes with the padded-sphere pixels (x, y[, frame]) zeroed."""
    img = np.array(img, np.float32, copy=True)
    for p in pads:
        img[p[1], p[0]] = 0
    return hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest()


def assert_equals_reference(buf, rays, pads, key):
    """Ray counts, padded-sphere pixels and every other pixel's bits equal the reference's render `key`."""
    g = parity_render(key)
    assert rays == g["rays"], key
    assert pads == g["pads"], key
    assert image_hash(buf, pads) == g["sha256_pads_zeroed"], key


def scene_for(oracle, w, h):
    """46-sphere scene at aspect w/h: spheres/materials from the golden export, camera from the reference when
    available (it depends on the aspect ratio), else only 16:9 sizes are valid."""
    sph, mats, cam, em = golden_scene()
    if oracle.have_ref():
        sph, mats, cam, em = oracle.ref_scene(w, h)
    else:
        assert w * 9 == h * 16
    return sph, mats, cam, em


def test_golden_image_and_counts(oracle):
    g = np.load(os.path.join(GOLD, "ref_192x108_f0-3.npz"))
    sph, mats, cam, em = golden_scene()
    buf, rays, pads = oracle.orc_render(sph, mats, cam, 192, 108, 0, 4, flags=2)
    assert rays == [int(r) for r in g["rays"]]
    assert not pads
    assert not bits_differ(buf, g["image"]).any()


def test_golden_ray_counts_720p(oracle):
    counts = json.load(open(os.path.join(GOLD, "ref_counts.json")))
    sph, mats, cam, em = golden_scene()
    _, rays, _ = oracle.orc_render(sph, mats, cam, 1280, 720, 0, 2, flags=0)
    assert rays == counts["1280x720_flags0_frames0-5"][:2]          # 16 809 105, 16 822 947 (SURVEY §9.2)


def test_restatement_equals_reference_bitwise(oracle):
    for (w, h, f0, nf, flags) in [(320, 180, 0, 3, 2), (200, 120, 7, 2, 0)]:
        sph, mats, cam, em = parity_scene(f"stock_{w}x{h}_t0.0_flags{flags}")
        obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, f0, nf, flags=flags)
        assert_equals_reference(obuf, orays, pads, f"stock_{w}x{h}_t0.0_flags{flags}_frames{f0}+{nf}")


def test_restatement_equals_reference_animated(oracle):
    """kFlagAnimate: spheres 1 and 8 move with time, lerpFac *= 0.9 (Test.cpp:273-274,304-308)."""
    w, h, t, flags = 160, 90, 1.25, 3
    sph, mats, cam, em = parity_scene(f"stock_{w}x{h}_t{t}_flags{flags}")
    obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 40, 2, flags=flags)
    assert_equals_reference(obuf, orays, pads, f"stock_{w}x{h}_t{t}_flags{flags}_frames40+2")


def test_padded_sphere_hit_control_flow(oracle):
    """Frame 28 of the 1280x720 sequence contains a path ray that 'hits' a padded impossible sphere (reference UB,
    see oracle/restate.cpp Trace()). The restatement must follow the reference's control flow: equal ray counts,
    and only that pixel may differ."""
    sph, mats, cam, em = parity_scene("stock_1280x720_t0.0_flags0")
    gs, gm, gc, ge = golden_scene()
    assert sph.tobytes() == gs.tobytes() and mats.tobytes() == gm.tobytes() and cam.tobytes() == gc.tobytes()
    obuf, orays, pads = oracle.orc_render(sph, mats, cam, 1280, 720, 28, 1, flags=0)
    assert orays == [16813074]
    assert pads == [(180, 436, 28)]
    assert_equals_reference(obuf, orays, pads, "stock_1280x720_t0.0_flags0_frames28+1")


def test_scalar_vs_simd_tie_rule_agree_on_reference_scene(oracle):
    sph, mats, cam, em = golden_scene()
    a, ra, _ = oracle.orc_render(sph, mats, cam, 192, 108, 0, 1, simd_tie=1)
    b, rb, _ = oracle.orc_render(sph, mats, cam, 192, 108, 0, 1, simd_tie=0)
    assert ra == rb and not bits_differ(a, b).any()


def test_runtime_scene_edge_cases(oracle):
    """Sizes and scenes the reference itself cannot run: 1 sphere, counts not a multiple of 4, no lights."""
    import toypathtracer_b200 as tpt
    cam = tpt.make_camera((0, 1, 4), (0, 0, 0), (0, 1, 0), 45, 2.0, 0.05, 4)
    for n in (1, 2, 5, 7):
        sph = np.zeros(n, tpt.SPHERE_DTYPE); mats = np.zeros(n, tpt.MATERIAL_DTYPE)
        for i in range(n):
            sph[i] = ((i - n / 2, 0, 0), 0.45, 0)
            mats[i] = (i % 3, (0.7, 0.6, 0.5), (4, 4, 4) if i == 1 else (0, 0, 0), 0.1, 1.5)
        buf, rays, pads = oracle.orc_render(sph, mats, cam, 64, 32, 0, 2, flags=2)
        assert np.isfinite(buf).all() and rays[0] >= 64 * 32 * 4


@pytest.mark.parametrize("variant,big,mitsuba", [("mitsuba", True, True), ("small", False, False), ("small_mitsuba", False, True)])
def test_reference_compile_time_variants(oracle, variant, big, mitsuba):
    """DO_MITSUBA_COMPARE (Config.h:25) and DO_BIG_SCENE 0 (Test.cpp:10-11): the reference compiled from an edited
    temporary copy (oracle/Makefile) vs the restatement's runtime switch and the drop-in shim's scene export."""
    import toypathtracer_b200 as tpt
    w, h = 200, 120
    for flags in (0, 2):
        sph, mats, cam, em = parity_scene(f"{variant}_{w}x{h}_t0.0_flags{flags}")
        assert len(sph) == (46 if big else 9)
        s2, m2, c2, e2 = tpt.reference_scene(w, h, big_scene=big, mitsuba_compare=mitsuba)      # the shim's UpdateTest/GetSceneDesc
        assert s2.tobytes() == sph.tobytes() and m2.tobytes() == mats.tobytes() and c2.tobytes() == cam.tobytes()
        assert list(e2) == list(em)
        obuf, orays, pads = oracle.orc_render(sph, mats, cam, w, h, 0, 3, flags=flags, mitsuba=mitsuba)
        assert_equals_reference(obuf, orays, pads, f"{variant}_{w}x{h}_t0.0_flags{flags}_frames0+3")


def test_refgpu_oracle_is_the_same_estimator_statistically(oracle):
    """oracle/refgpu_restate.cpp (the reference's GPU shader restated; parity unpinned, see its header) against the CPU
    path's restatement: same scene, same estimator up to the depth limit (10 vs 11 segments) and the samplers'
    parametrisation -> the images agree within Monte-Carlo noise, rays per sample within a fraction of a percent."""
    sph, mats, cam, em = golden_scene()
    w, h, nf = 160, 90, 64
    a, ra, _ = oracle.orc_render(sph, mats, cam, w, h, 0, nf, flags=2)
    c = a.copy()
    oracle.orc_render(sph, mats, cam, w, h, nf, nf, flags=2, buf=c)          # progressive mean over 2*nf frames
    a2 = 2.0 * c[..., :3].astype(np.float64) - a[..., :3]                      # = mean of frames [nf, 2nf): independent of a
    b, rb = oracle.rgo_render(sph, mats, cam, w, h, 0, nf, flags=2)
    assert (b[..., 3] == 1).all()
    rl2 = lambda x, y: float(np.sqrt(((x.astype(np.float64) - y) ** 2).sum() / (y.astype(np.float64) ** 2).sum()))
    floor = rl2(a2, a[..., :3])                                                 # CPU path vs itself, other frames
    assert rl2(b[..., :3], a[..., :3]) < 1.15 * floor
    assert 0.985 < sum(rb) / sum(ra) <= 1.0005            # the 11th segment is the only systematic difference in ray count
    ma, mb = a[..., :3].reshape(-1, 3).mean(0), b[..., :3].reshape(-1, 3).mean(0)
    assert (np.abs(ma - mb) < 0.01 * ma).all(), (ma, mb)
