"""The C++ shim (reflaxman_b200/shim) mirrors the reference's Render/Scene/Camera class surface on top of the C ABI.

CPU: it compiles — against oracle/ref_harness.cpp (the driver written for the UNMODIFIED reference) and, where the
reference tree is present, against the reference's own Pulse.cpp, unchanged.
GPU: the shim-built harness reproduces the golden vectors the reference-built harness produced."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S
from reflaxman_b200.build import REFERENCE_SRC as REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "reflaxman_b200", "shim")


def test_reference_harness_source_builds_against_shim(rfx_lib):
    from reflaxman_b200 import build
    exe = build.build_shim_harness(force=True)
    assert os.access(exe, os.X_OK)


def test_reference_pulse_compiles_unchanged_against_shim():
    """Pulse.cpp is the only client of Render upstream (reference Pulse.cpp:38-457)."""
    if not os.path.isdir(REF):
        pytest.skip("RFX_REFERENCE_SRC does not name the reference's src/common")
    with tempfile.TemporaryDirectory() as td:
        for f in ("Pulse.h", "Pulse.cpp", "BasePlatformInterface.h", "BasePlatformInterface.cpp", "defaults.h"):
            os.symlink(os.path.join(REF, f), os.path.join(td, f))       # the reference's own files, untouched
        for f in os.listdir(SHIM):
            shutil.copy(os.path.join(SHIM, f), td)                      # our headers take the place of Render.h, Scene.h, ...
        for src in ("Pulse.cpp", "BasePlatformInterface.cpp"):
            subprocess.run(["g++", "-std=c++14", "-O2", "-Wno-multichar", "-I" + os.path.join(ROOT, "include"), "-c",
                            os.path.join(td, src), "-o", os.path.join(td, src + ".o")], check=True)


def test_reference_pulse_links_against_shim_and_library(rfx_lib):
    """f-2: the unchanged Pulse.cpp + BasePlatformInterface.cpp link with the shim, the CUDA library and a headless platform stub."""
    from reflaxman_b200 import build
    exe = build.build_shim_pulse(force=os.path.isdir(REF))
    if exe is None:
        pytest.skip("no reference tree (RFX_REFERENCE_SRC) and no prebuilt build/shim_pulse_headless")
    assert os.access(exe, os.X_OK)


def _run_pulse(exe, td):
    os.makedirs(td, exist_ok=True)
    res = subprocess.run([exe, td + "/", "160", "120", "260", "2", "2"], check=True, capture_output=True, text=True, env=dict(os.environ, RFX_SEED="12345"))
    inter = np.fromfile(os.path.join(td, "interactive.bin"), dtype=np.uint32).reshape(120, 160)
    hud = open(os.path.join(td, "hud.txt")).read()
    bmp = open(os.path.join(td, "scrnshoot_0000000100000002.bmp"), "rb").read()
    return inter, hud, bmp, res.stdout


@pytest.mark.gpu
def test_pulse_runs_headless_on_the_gpu_path(rfx_lib, oracle, tmp_path):
    """SURVEY §8 f-2, for real: the reference's UI controller (Pulse.cpp, unchanged) running on the GPU path behind a headless
    BasePlatformInterface — a scripted interactive session (keys W / LEFT / SPACE / D / A: camera kinematics, motion frames in
    block-preview mode at depth 4, static frames accumulating additively at depth 15, renderNext in adaptive chunks that grow
    and shrink with a virtual clock, a per-pixel repaint after every frame) and then the F2 screenshot flow at 1024x768 with
    2x2 SSAA saved as a BMP — against the same program built with the reference's own Render: same HUD text (resolution,
    blended-frame count), the last repaint and the saved BMP within the parity bar."""
    import hashlib
    from reflaxman_b200 import build
    exe = build.build_shim_pulse()
    if exe is None:
        pytest.skip("build/shim_pulse_headless was not built (needs the reference tree, RFX_REFERENCE_SRC, at build time)")
    inter, hud, bmp, info = _run_pulse(exe, str(tmp_path / "gpu"))
    g = np.load(os.path.join(cases.GOLDEN_DIR, "pulse_headless.npz"))
    assert hud == str(g["hud"]), (hud, str(g["hud"]))
    st = cases.assert_parity(inter, g["interactive"], "Pulse interactive repaint")
    assert len(bmp) == int(g["bmp_bytes"]) == 54 + 1024 * 768 * 4 and bmp[:54] is not None
    same = hashlib.sha256(bmp).hexdigest() == str(g["bmp_sha256"])
    print("Pulse headless:", info.strip(), "interactive", st, "screenshot BMP identical to the reference's:", same)
    ref_exe = os.path.join(oracle.REF_DIR, "ref_pulse_headless")
    if os.access(ref_exe, os.X_OK):
        rinter, rhud, rbmp, _ = _run_pulse(ref_exe, str(tmp_path / "ref"))
        assert rhud == hud and np.array_equal(rinter, g["interactive"])
        assert rbmp[:54] == bmp[:54]                       # identical BMP headers (Texture.cpp:139-173)
        a = np.frombuffer(bmp[54:], dtype="<u4").reshape(768, 1024)
        b = np.frombuffer(rbmp[54:], dtype="<u4").reshape(768, 1024)
        print("screenshot:", cases.assert_parity(a, b, "Pulse screenshot BMP"))
    else:
        assert same, "no reference binary on this box and the BMP differs from the reference's hash"


def run_shim_harness(args, seed, W, H, scene=None, cams=None):
    from reflaxman_b200 import build
    exe = build.build_shim_harness()
    with tempfile.TemporaryDirectory() as td:
        cmd = [exe, "--size", str(W), str(H), *args, "--out", os.path.join(td, "o.bin")]
        if scene is not None:
            tex_paths = []
            for i, t in enumerate(scene["textures"]):
                p = os.path.join(td, "tex%d.tga" % i)
                if t is not None:
                    S.write_tga(p, t, 32)
                tex_paths.append(p)
            sky = os.path.join(td, "sky.tga")
            if scene.get("skybox") is not None:
                S.write_tga(sky, scene["skybox"], 24)      # 24-bpp on purpose: exercises the other loader branch
            with open(os.path.join(td, "scene.txt"), "w") as f:
                f.write(S.scene_to_text(scene, tex_paths, sky))
            cmd += ["--scene", os.path.join(td, "scene.txt")]
        if cams is not None:
            with open(os.path.join(td, "cams.txt"), "w") as f:
                f.write(S.cameras_to_text(cams))
            cmd += ["--cams", os.path.join(td, "cams.txt")]
        subprocess.run(cmd, check=True, env=dict(os.environ, RFX_SEED=str(seed)), stdout=subprocess.DEVNULL)
        raw = np.fromfile(os.path.join(td, "o.bin"), dtype=np.uint8)
    per = W * H * 16
    return [(raw[i * per:i * per + W * H * 12].view(np.float32).reshape(H, W, 3), raw[i * per + W * H * 12:(i + 1) * per].view(np.uint32).reshape(H, W))
            for i in range(len(raw) // per)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["default_160x120_d20", "default_96x64_ss3", "default_96x64_block4", "default_96x64_additive3",
                                  "default_64x48_2frames", "textured_160x120_d20", "synth36_128x72_d8"])
def test_shim_harness_reproduces_reference_harness(rfx_lib, name):
    g = cases.load_golden(name)
    args = ["--refl", str(g["refl"]), "--samples", str(g["samples"]), "--frames", str(g["frames"])]
    if g["additive"]:
        args += ["--additive", str(g["additive"])]
    scene = None if name.startswith("default") else g["scene"]
    frames = run_shim_harness(args, g["seed"], g["W"], g["H"], scene=scene)
    assert len(frames) == g["frames"]
    for i, (rgbf, argb) in enumerate(frames):
        cases.assert_parity(argb, g["argb%d" % i], "%s frame %d via shim" % (name, i))
        assert np.max(np.abs(rgbf - g["rgbf%d" % i])) < 2e-5


@pytest.mark.gpu
def test_shim_scene_trace_matches_render(rfx_lib):
    """--rows mode of the harness goes through Scene::trace (rfx_trace_rays), one ray per call."""
    frames = run_shim_harness(["--refl", "6", "--rows", "3", "1"], 99, 24, 18)
    rgbf, argb = frames[0]
    assert np.all(argb[0::3] == 0) and np.any(argb[1::3] != 0)


def test_shim_texture_file_formats(tmp_path):
    """f-4: 32-bpp bottom-up BMP and type-2 TGA exactly as the reference writes them (Texture.cpp:110-173, image_headers.h)."""
    import struct
    exe = str(tmp_path / "texture_io")
    subprocess.run(["g++", "-std=c++14", "-O1", "-I" + SHIM, "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "texture_io.cpp"), "-o", exe], check=True)
    subprocess.run([exe, str(tmp_path)], check=True)
    px = np.array([(0x01020300 * (i + 1) + i) & 0xFFFFFFFF for i in range(15)], dtype="<u4")
    bmp = (tmp_path / "a.bmp").read_bytes()
    bfType, bfSize, _, _, bfOff = struct.unpack_from("<HIHHI", bmp, 0)
    biSize, w, h, planes, bpp, comp = struct.unpack_from("<IiiHHI", bmp, 14)
    assert (bfType, bfSize, bfOff, biSize, w, h, planes, bpp, comp) == (0x4D42, 54 + 60, 54, 40, 5, 3, 1, 32, 0)
    assert bmp[54:] == px.tobytes()
    tga = (tmp_path / "a.tga").read_bytes()
    assert struct.unpack_from("<bbbhhbhhhhbb", tga, 0) == (0, 0, 2, 0, 0, 0, 0, 0, 5, 3, 32, 0)
    assert tga[18:] == px.tobytes()
