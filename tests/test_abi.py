"""The C-ABI library loads on a CPU-only machine and exports every symbol include/tpt_b200.h declares; the
drop-in shim exports the six functions of the reference's Test.h with their C++-mangled names; host-side logic
of the shim (scene, camera, emissive list) equals the reference's GetSceneDesc export; nothing renders on CPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from test_oracle import golden_scene, parity_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(libs):
    hdr = open(os.path.join(ROOT, "include", "tpt_b200.h")).read()
    names = sorted(set(re.findall(r"\b(tpt_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 12
    L = ctypes.CDLL(libs.LIB_PATH)
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/tpt_b200.h but not exported"


def test_shim_exports_reference_api(libs):
    S = ctypes.CDLL(libs.SHIM_PATH)
    hdr = open(os.path.join(ROOT, "include", "tpt_test_shim.h")).read()
    for n in sorted(set(re.findall(r"\b(tpt_shim_[a-z0-9_]+)\s*\(", hdr))):
        assert hasattr(S, n), f"{n} declared in include/tpt_test_shim.h but not exported by the shim"
    for sym in ("_Z14InitializeTestv", "_Z12ShutdownTestv", "_Z10UpdateTestfiiij", "_Z8DrawTestfiiiPfRij",
                "_Z14GetObjectCountRiS_S_S_", "_Z12GetSceneDescPvS_S_S_Pi"):
        assert hasattr(S, sym), sym


def test_shim_scene_equals_reference_export(libs):
    assert libs.GetObjectCount() == (46, 20, 36, 88)          # TestWin.cpp:132-134
    sph, mats, cam, em = libs.reference_scene(1280, 720)
    gs, gm, gc, ge = golden_scene()
    assert sph.tobytes() == gs.tobytes()
    assert mats.tobytes() == gm.tobytes()
    assert cam.tobytes() == gc.tobytes()
    assert list(em) == list(ge) == [8, 45]


def test_shim_camera_and_animation_equal_reference(libs):
    for (w, h, flags, t) in [(3840, 2160, 0, 0.0), (640, 480, 1, 1.25), (256, 144, 3, 7.5)]:
        rs, rm, rc, re_ = parity_scene(f"stock_{w}x{h}_t{t}_flags{flags}")
        sph, mats, cam, em = libs.reference_scene(w, h, time=t, flags=flags)
        assert sph.tobytes() == rs.tobytes() and mats.tobytes() == rm.tobytes() and cam.tobytes() == rc.tobytes()
        assert list(em) == list(re_)


def test_no_cpu_fallback(libs):
    if libs.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(libs.TptError):
        libs.Context(0)


def test_scene_blob_padding_rules(libs):
    """pack rules mirrored from SpheresSoA (Maths.h:370-388): covered through the host sim + stress scene sizes."""
    sph, mats, cam, em = libs.stress_scene(320, 180, count=4096)
    assert len(sph) == 4096 and len(em) == 6 and sph.dtype.itemsize == 20 and mats.dtype.itemsize == 36
    assert np.isfinite(sph["center"]).all()


def test_header_is_plain_c_and_links(libs, tmp_path):
    """include/tpt_b200.h must be consumable from C (the cgo / JNI / N-API style binding INTEGRATION.md shows): compile a
    C translation unit that takes the address of every declared function and link it against libtpt_b200.so."""
    import subprocess
    hdr = open(os.path.join(ROOT, "include", "tpt_b200.h")).read()
    names = sorted(set(re.findall(r"\b(tpt_[a-z0-9_]+)\s*\(", hdr)))
    src = tmp_path / "use.c"
    src.write_text('#include "tpt_b200.h"\n#include <stdio.h>\ntypedef void (*fn_t)(void);\nint main(void) {\n  fn_t f[] = {' +
                   ", ".join(f"(fn_t){n}" for n in names) +
                   '};\n  printf("%d %d\\n", (int)(sizeof f / sizeof f[0]), tpt_device_count());\n  return f[0] == 0;\n}\n')
    exe = tmp_path / "use"
    libdir = os.path.dirname(libs.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-ltpt_b200", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert int(out[0]) == len(names) and int(out[1]) >= 0


def test_host_code_is_sanitizer_clean(tmp_path, oracle):
    """ASan + UBSan build of the host-side product sources that run on every draw (scene packing, integrator source on
    the host, glibc restatement) and of the oracle restatement: one small render each, no reports."""
    import subprocess
    src = tmp_path / "san.cpp"
    src.write_text('''
#include "tests/host_sim/exact_sim.cpp"
#include <cstdio>
int main() {
    tpt::Sphere20 s[5]; tpt::Material36 m[5];
    for (int i = 0; i < 5; ++i) { s[i] = {{float(i) - 2.f, 0.f, -1.f}, 0.45f, 0.f}; m[i] = {i % 3, {0.7f, 0.6f, 0.5f}, {i == 1 ? 4.f : 0.f, 0.f, 0.f}, 0.1f, 1.5f}; }
    tpt::Camera88 c = {{0, 1, 4}, {-2, -1, 1}, {4, 0, 0}, {0, 2, -0.5f}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}, 0.02f};
    std::vector<float> buf(48 * 27 * 4, 0.f); long long rays[2];
    sim_render_exact(s, m, 5, &c, 48, 27, 0, 2, 2, 4, buf.data(), rays, 2);
    sim_render_exact_flat(s, m, 5, &c, 48, 27, 0, 2, 2, 4, buf.data(), rays, 2);
    std::printf("%lld %lld\\n", rays[0], rays[1]);
    return 0;
}
''')
    exe = tmp_path / "san"
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-mfma", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", ROOT, str(src), "-o", str(exe), "-lpthread", "-lm"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert len(r.stdout.split()) == 2
