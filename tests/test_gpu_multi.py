"""One context over several GPUs of one process (mprb_ctx_opts::n_gpus / MPRB_GPUS; api.cu: render_all):
every device renders the screen columns (x + y) % N == its index and stores its blocks into the primary's
frame over NVLink peer mappings.  The frame on the primary must equal the single-GPU frame bit for bit,
and the reference's unchanged table driver must run on several GPUs by environment alone.
Skipped on boxes with one GPU (run with `gpurun --gpus 2`)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_tape
from mpr_b200 import capi

pytestmark = pytest.mark.gpu


def n_devices():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


need2 = pytest.mark.skipif(n_devices() < 2, reason="needs at least two GPUs")


@need2
@pytest.mark.parametrize("model,dim,size", [("prospero", 2, 1024), ("hello_world", 2, 256), ("bear", 3, 256),
                                            ("architecture", 3, 512), ("bear", 3, 1024)])
def test_multi_gpu_context_equals_single_gpu_frame(model, dim, size):
    cells = load_tape(model)
    one = capi.Context(size, num_subtapes=6400000)
    tape = capi.Tape(cells)
    (one.render2D if dim == 2 else one.render3D)(tape)
    want_img = np.array(one.image(), copy=True)
    want_nrm = np.array(one.normals(), copy=True) if dim == 3 else None
    for n in sorted({2, min(n_devices(), 8)}):
        ctx = capi.Context(size, num_subtapes=6400000, n_gpus=n)
        for _ in range(3):                       # repeated frames: no stale blocks, no ordering luck
            (ctx.render2D if dim == 2 else ctx.render3D)(tape)
            assert np.array_equal(ctx.image(), want_img), (n, "image")
            if dim == 3:
                assert np.array_equal(ctx.normals(), want_nrm), (n, "normals")
        st = ctx.stats()
        assert st.f_tiles == one.stats().f_tiles or dim == 3     # 3D culling depends on arrival order
        ctx.close()
    # host-buffer entry point on two devices
    ctx = capi.Context(size, num_subtapes=6400000, n_gpus=2)
    img = np.zeros((size, size), dtype=np.int32)
    if dim == 2:
        ctx.render2D_host(cells, img)
    else:
        nrm = np.zeros((size, size), dtype=np.uint32)
        ctx.render3D_host(cells, img, nrm)
        assert np.array_equal(nrm, want_nrm)
    assert np.array_equal(img, want_img)
    ctx.close()
    one.close()


@need2
def test_reference_table_driver_runs_on_two_gpus(tmp_path):
    exe = ROOT / "oracle" / "_ref" / "drivers" / "render_3d_table"
    if not exe.exists():
        pytest.skip("drivers not built")
    env = dict(os.environ, MPRB_GPUS="2")
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr
    rows = [l.split() for l in r.stdout.strip().splitlines()]
    assert [int(x[0]) for x in rows][:3] == [256, 512, 1024]
    one = subprocess.run([str(exe)], cwd=tmp_path / "..", capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, MPRB_GPUS="1"))
    assert one.returncode == 0


def test_tape_is_usable_from_a_context_on_another_device():
    """A Tape made while device 0 is current must render on a context of device 1 (per-device copies)."""
    if n_devices() < 2:
        pytest.skip("needs at least two GPUs")
    cells = load_tape("hello_world")
    tape = capi.Tape(cells)                       # created with device 0 current
    a = capi.Context(256, device=0)
    b = capi.Context(256, device=1)
    a.render2D(tape)
    b.render2D(tape)
    assert np.array_equal(a.image(), b.image())
    a.close()
    b.close()
