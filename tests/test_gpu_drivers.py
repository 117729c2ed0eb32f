"""Drop-in check on the GPU box: the reference's own benchmark drivers, compiled unchanged
against mpr_b200/inc and linked with libmprb.so (`make -C oracle drivers`, which keeps what it built
in oracle/_ref/drivers where the reference sources are absent), run and produce their tables / images."""
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
DRV = ROOT / "oracle" / "_ref" / "drivers"


def run(name, cwd, *args, timeout=300):
    exe = DRV / name
    if not exe.exists():
        pytest.skip(f"{exe} not built (needs the reference sources at build time)")
    return subprocess.run([str(exe), *args], cwd=cwd, capture_output=True, text=True, timeout=timeout)


def test_render_2d_table_driver(tmp_path):
    r = run("render_2d_table", tmp_path)            # default shape: two spheres (render_2d_table.cpp:40-46)
    assert r.returncode == 0, r.stderr
    rows = [l.split() for l in r.stdout.strip().splitlines()]
    assert [int(x[0]) for x in rows] == [256, 512, 1024, 2048, 3072, 4096]     # "size mean_ms stdev_ms"
    assert all(float(x[1]) > 0 for x in rows)
    png = (tmp_path / "out_gpu_256.png").read_bytes()
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and len(png) > 256 * 256


def test_render_3d_table_driver(tmp_path):
    r = run("render_3d_table", tmp_path)
    assert r.returncode == 0, r.stderr
    rows = [l.split() for l in r.stdout.strip().splitlines()]
    assert [int(x[0]) for x in rows][:3] == [256, 512, 1024]
    assert (tmp_path / "out_gpu_depth_256.png").exists() or any(tmp_path.glob("*.png"))


def test_print_tape_table_driver(tmp_path):
    r = run("print_tape_table", tmp_path)
    assert r.returncode == 0, r.stderr
    # LaTeX rows "op & out & lhs & rhs" for max(sqrt(x^2+y^2) - 1, 0.5 - sqrt(x^2+y^2))
    assert "SQRT" in r.stdout and "MAX" in r.stdout and "SUB" in r.stdout


def test_render_effects_driver(tmp_path):
    # render_effects.cpp: a cut, rotated sphere at 512^3 through mpr::Effects::drawSSAO / drawShaded
    r = run("render_effects", tmp_path)
    assert r.returncode == 0, r.stderr
    for name in ("out_gpu_ssao.png", "out_gpu_shaded.png"):
        png = (tmp_path / name).read_bytes()
        assert png[:8] == b"\x89PNG\r\n\x1a\n" and len(png) > 1000


def _png_ok(path, min_bytes=1000):
    png = path.read_bytes()
    return png[:8] == b"\x89PNG\r\n\x1a\n" and len(png) > min_bytes


def test_render_2d_and_3d_drivers(tmp_path):
    # render_2d.cpp / render_3d.cpp: one frame of the default two-sphere shape + libfive CPU comparison image
    r = run("render_2d", tmp_path)                   # 2048^2 by default
    assert r.returncode == 0, r.stderr
    assert _png_ok(tmp_path / "out_gpu_depth.png") and _png_ok(tmp_path / "out_cpu.png")
    (tmp_path / "out_cpu.png").unlink()
    r = run("render_3d", tmp_path)                   # 512^3 by default
    assert r.returncode == 0, r.stderr
    for name in ("out_gpu_depth.png", "out_gpu_norm.png", "out_cpu.png"):
        assert _png_ok(tmp_path / name), name


def test_heatmap_drivers(tmp_path):
    r = run("render_2d_heatmap", tmp_path)
    assert r.returncode == 0, r.stderr
    assert _png_ok(tmp_path / "out_depth_2d.png") and _png_ok(tmp_path / "out_heatmap_2d.png")
    r = run("render_3d_heatmap", tmp_path)
    assert r.returncode == 0, r.stderr
    assert _png_ok(tmp_path / "out_depth_3d.png") and _png_ok(tmp_path / "out_heatmap_3d.png")


def test_brute_driver(tmp_path):
    # brute.cu: compiled kernel vs interpreter without subdivision vs the full algorithm, 256..2048 / 4096
    r = run("brute", tmp_path, timeout=600)
    assert r.returncode == 0, r.stderr
    out = r.stdout
    assert "compiled kernel" in out and "brute-force with interpreter" in out and "fancy algorithm" in out
    a = (tmp_path / "out_brute_256.png").read_bytes()
    b = (tmp_path / "out_alg_256.png").read_bytes()
    k = (tmp_path / "out_kernel_256.png").read_bytes()
    assert a == b                      # same picture with and without subdivision
    assert len(k) == len(a)


def test_dump_tape_driver(tmp_path):
    r = run("dump_tape", tmp_path)
    assert r.returncode == 0, r.stderr
    assert "const float" in r.stdout or "float" in r.stdout
