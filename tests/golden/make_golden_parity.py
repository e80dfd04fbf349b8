"""Records what the UNMODIFIED reference produces for every test that compares the restatement, the exact mode or
the drop-in shell with it, so that those tests run without the reference. Needs oracle/_ref/libtoyref*.so and
oracle/_ref/ref_headless, which oracle/Makefile builds where the reference sources are present:

    python tests/golden/make_golden_parity.py

Outputs (small, committed):
  ref_parity_scenes.npz  raw GetSceneDesc exports (spheres, materials, camera, emissive ids) per scene key
  ref_parity.json        per render: per-frame ray counts, the padded-sphere pixels (x, y, frame) reported by the
                         restatement (their colour is undefined behaviour in the reference, DESIGN.md §1.1) and the
                         sha256 of the reference's float image with those pixels zeroed; the headless shell's output
Every render is also checked against the restatement here, as the tests did against the live reference.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle  # noqa: E402

here = os.path.dirname(os.path.abspath(__file__))
VARIANTS = {"": (True, False), "mitsuba": (True, True), "small": (False, False), "small_mitsuba": (False, True)}


def scene_key(variant, w, h, time=0.0, flags=0):
    return f"{variant or 'stock'}_{w}x{h}_t{time}_flags{flags}"


def render_key(variant, w, h, f0, n, flags, time=0.0):
    return f"{variant or 'stock'}_{w}x{h}_t{time}_flags{flags}_frames{f0}+{n}"


def image_hash(img, pads):
    img = np.array(img, np.float32, copy=True)
    for p in pads:
        img[p[1], p[0]] = 0
    return hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest()


def main():
    scenes, renders = {}, {}

    def scene(variant, w, h, time=0.0, flags=0):
        animated = flags & 1
        s = (pyoracle.isolated("ref_scene", w, h, time=time, flags=flags, variant=variant) if animated
             else pyoracle.ref_scene(w, h, time=time, flags=flags, variant=variant))
        k = scene_key(variant, w, h, time, flags)
        for name, a in zip(("spheres", "materials", "camera", "emissives"), s):
            scenes[f"{k}/{name}"] = a
        return s

    def render(variant, w, h, f0, n, flags, time=0.0):
        sph, mats, cam, em = scene(variant, w, h, time, flags)
        if flags & 1:
            rbuf, rrays = pyoracle.isolated("ref_render", w, h, f0, n, flags=flags, time=time, variant=variant)
        else:
            rbuf, rrays = pyoracle.ref_render(w, h, f0, n, flags=flags, time=time, variant=variant)
        obuf, orays, pads = pyoracle.orc_render(sph, mats, cam, w, h, f0, n, flags=flags, mitsuba=VARIANTS[variant][1])
        assert orays == rrays, (variant, w, h, f0, n, flags)
        assert not np.isnan(rbuf).any()
        assert image_hash(obuf, pads) == image_hash(rbuf, pads), (variant, w, h, f0, n, flags)
        renders[render_key(variant, w, h, f0, n, flags, time)] = {
            "rays": rrays, "pads": [list(p) for p in pads], "sha256_pads_zeroed": image_hash(rbuf, pads)}

    # the shim's scene export against the reference's: sizes, aspect ratios, animation
    for (w, h, flags, t) in [(3840, 2160, 0, 0.0), (640, 480, 1, 1.25), (256, 144, 3, 7.5)]:
        scene("", w, h, t, flags)
    # restatement (CPU) and exact mode (GPU) against the reference
    render("", 320, 180, 0, 3, 2)
    render("", 200, 120, 7, 2, 0)
    render("", 160, 90, 40, 2, 3, time=1.25)
    render("", 1280, 720, 28, 1, 0)                    # holds a padded-sphere hit
    render("", 1280, 720, 0, 3, 0)                     # the drop-in's DrawTest at the benchmark size
    render("", 1280, 720, 4, 1, 0)                     # bench.py's last timed step at --warmup 3 --steps 2
    for v in ("mitsuba", "small", "small_mitsuba"):
        for (w, h) in ((200, 120), (320, 180)):
            for flags in (0, 2):
                render(v, w, h, 0, 3, flags)
    render("small_mitsuba", 256, 144, 0, 3, 2)

    headless_args = ["384", "216", "4", "2"]
    out = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "ref_headless")] + headless_args, capture_output=True,
                         text=True, check=True).stdout
    lines = [l for l in out.splitlines() if l.startswith("frame") or l.startswith("checksum")]
    assert len(lines) == 5

    np.savez_compressed(os.path.join(here, "ref_parity_scenes.npz"),
                        **{k: (v.view(np.uint32) if k.endswith("/materials") else v) for k, v in scenes.items()})
    json.dump({"renders": renders, "headless": {"args": headless_args, "lines": lines}},
              open(os.path.join(here, "ref_parity.json"), "w"), indent=1)
    print(len(scenes) // 4, "scenes,", len(renders), "renders")


if __name__ == "__main__":
    main()
