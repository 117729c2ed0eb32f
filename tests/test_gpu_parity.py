"""GPU parity tests (B200 box): libmprb through its C ABI against
  (1) fixtures minted from the unmodified reference build (tests/golden/ref),
  (2) what the reference build computed for post-effects, brute-force frames and work meters
      (tests/golden/ref_variants, minted by tools/mint_ref_variants.py),
  (3) the CPU restatement,
and size-independent properties at the BASELINE sizes.  Integer / byte results: bit exact."""
import ctypes as C
import json

import numpy as np
import pytest

import oracle
import parity
from conftest import ROOT, golden_cases, load_tape
from mpr_b200 import capi, sharding

pytestmark = pytest.mark.gpu
SUBTAPES = 6400000
CASES = golden_cases()
SMALL = [c for c in CASES if c[5] is not None]
VARIANTS = ROOT / "tests" / "golden" / "ref_variants"


def ref_variant(key):
    return json.loads((VARIANTS / "records.json").read_text())[key]


def render(model, dim, size, **kw):
    ctx = capi.Context(size, num_subtapes=kw.pop("num_subtapes", SUBTAPES), **kw)
    tape = capi.Tape(load_tape(model))
    (ctx.render2D if dim == 2 else ctx.render3D)(tape)
    return ctx, tape


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_matches_reference_fixture(case):
    name, model, dim, size, summary, npz = case
    ctx, tape = render(model, dim, size)
    fp = parity.fingerprint(ctx, dim)
    got = parity.summarize(fp)
    bad = parity.compare_summary(summary, got)
    assert not bad, bad
    if npz is not None:
        ref = dict(np.load(npz))
        ref["dim"], ref["size"] = dim, size
        assert not parity.compare(ref, fp)
    st = ctx.stats()
    assert st.overflow == 0 and st.n_launches > 0
    ctx.close()


@pytest.mark.parametrize("model,dim,size", [("prospero", 2, 512), ("involute_gear_2d", 2, 1024),
                                            ("architecture", 3, 512), ("bear", 3, 512),
                                            ("involute_gear_3d", 3, 512)])
def test_matches_live_reference_build(model, dim, size):
    """Every field of the fingerprint equals the reference build's frame (its digests, recorded in
    tests/golden/ref by tools/gpu_check.py)."""
    want = json.loads((ROOT / "tests" / "golden" / "ref" / f"{model}_{dim}d_{size}.json").read_text())
    ctx, tape = render(model, dim, size)
    got = parity.summarize(parity.fingerprint(ctx, dim))
    assert set(got) == set(want)
    assert not parity.compare_summary(want, got)
    ctx.close()


@pytest.mark.parametrize("model,dim,size", [("hello_world", 2, 128), ("prospero", 2, 256), ("hello_world", 3, 128),
                                            ("architecture", 3, 128)])
def test_matches_cpu_restatement(model, dim, size):
    o = oracle.CpuOracle(size, SUBTAPES)
    (o.render2D if dim == 2 else o.render3D)(load_tape(model))
    ctx, tape = render(model, dim, size)
    assert not parity.compare(parity.fingerprint(o, dim), parity.fingerprint(ctx, dim))
    o.close()
    ctx.close()


def test_view_matrix_and_z_plane_are_honoured():
    # a rotated / translated / perspective view must go through the same interval transform
    m3 = np.array([[0.8, -0.3, 0.1], [0.3, 0.8, -0.2], [0.05, 0.02, 1.0]], dtype=np.float32)
    cells = load_tape("hello_world")
    o = oracle.CpuOracle(256)
    o.render2D(cells, mat=m3, z=0.25)
    ctx = capi.Context(256)
    tape = capi.Tape(cells)
    ctx.render2D(tape, mat=m3, z=0.25)
    assert not parity.compare(parity.fingerprint(o, 2), parity.fingerprint(ctx, 2))
    m4 = np.eye(4, dtype=np.float32)
    m4[0, 1], m4[1, 0], m4[3, 2], m4[2, 3] = 0.2, -0.2, 0.4, 0.1
    o3 = oracle.CpuOracle(128)
    o3.render3D(cells, mat=m4)
    ctx3 = capi.Context(128)
    ctx3.render3D(tape, mat=m4)
    assert not parity.compare(parity.fingerprint(o3, 3), parity.fingerprint(ctx3, 3))


def test_frames_are_idempotent_and_contexts_reusable():
    ctx, tape = render("architecture", 3, 256)
    a = parity.fingerprint(ctx, 3)
    ctx.render3D(tape)
    assert not parity.compare(a, parity.fingerprint(ctx, 3))
    # a different model, then back again, in the same context
    other = capi.Tape(load_tape("bear"))
    ctx.render3D(other)
    ctx.render3D(tape)
    assert not parity.compare(a, parity.fingerprint(ctx, 3))
    # 2D after 3D in the same context
    ctx.render2D(capi.Tape(load_tape("prospero")))
    ref2, _ = render("prospero", 2, 256)
    assert np.array_equal(ctx.image(), ref2.image())


def test_host_buffer_entry_points_equal_device_ones():
    cells = load_tape("bear")
    ctx, tape = render("bear", 3, 256)
    depth = np.zeros((256, 256), dtype=np.int32)
    norm = np.zeros((256, 256), dtype=np.uint32)
    ctx2 = capi.Context(256, num_subtapes=SUBTAPES)
    ctx2.render3D_host(cells, depth, norm)
    assert np.array_equal(depth, ctx.image()) and np.array_equal(norm, ctx.normals())
    img = np.zeros((512, 512), dtype=np.int32)
    c2 = capi.Context(512)
    c2.render2D_host(load_tape("prospero"), img)
    ref, _ = render("prospero", 2, 512)
    assert np.array_equal(img, ref.image())
    assert set(np.unique(img)) <= {0, 1}


@pytest.mark.parametrize("model,dim,size,world", [("prospero", 2, 1024, 4), ("bear", 3, 256, 2), ("architecture", 3, 512, 8)])
def test_row_bands_tile_the_full_frame(model, dim, size, world):
    """Sharding property: rendering tile-row bands separately and stacking them equals one full frame."""
    full, tape = render(model, dim, size)
    img = np.zeros((size, size), dtype=np.int32)
    nrm = np.zeros((size, size), dtype=np.uint32)
    for r in range(world):
        b, e = sharding.band_rows(size, world, r)
        part = capi.Context(size, num_subtapes=SUBTAPES, row_begin=b, row_end=e)
        (part.render2D if dim == 2 else part.render3D)(tape)
        sl = sharding.band_slice(size, world, r)
        img[sl] = part.image()[sl]
        if dim == 3:
            nrm[sl] = part.normals()[sl]
        outside = np.ones(size, dtype=bool)
        outside[sl] = False
        assert not part.image()[outside].any()          # a band context never writes other bands
        part.close()
    assert np.array_equal(img, full.image())
    if dim == 3:
        assert np.array_equal(nrm, full.normals())


@pytest.mark.parametrize("model,dim,size,world", [("prospero", 2, 1024, 4), ("bear", 3, 512, 8)])
def test_interleaved_rows_tile_the_full_frame(model, dim, size, world):
    """Same property for the cyclic assignment bench.py uses (rank r owns tile rows r, r+world, ...)."""
    full, tape = render(model, dim, size)
    img = np.zeros((size, size), dtype=np.int32)
    nrm = np.zeros((size, size), dtype=np.uint32)
    owner = (np.arange(size) // 64) % world
    for r in range(world):
        part = capi.Context(size, num_subtapes=SUBTAPES, **sharding.cyclic_rows(size, world, r))
        (part.render2D if dim == 2 else part.render3D)(tape)
        assert not part.image()[owner != r].any()
        img[owner == r] = part.image()[owner == r]
        if dim == 3:
            nrm[owner == r] = part.normals()[owner == r]
        part.close()
    assert np.array_equal(img, full.image())
    if dim == 3:
        assert np.array_equal(nrm, full.normals())


@pytest.mark.parametrize("model,dim,size,world", [("prospero", 2, 1024, 4), ("bear", 3, 512, 8), ("hello_world", 3, 256, 2)])
def test_diagonal_tiles_tile_the_full_frame(model, dim, size, world):
    """Tile-cyclic assignment (rank r owns the 64x64-px screen columns with (x + y) % world == r):
    the parts are disjoint and their union is the single-context frame, image and normals."""
    full, tape = render(model, dim, size)
    img = np.zeros((size, size), dtype=np.int32)
    nrm = np.zeros((size, size), dtype=np.uint32)
    owner = np.kron(sharding.diagonal_owner(size, world), np.ones((64, 64), dtype=np.int64))
    for r in range(world):
        part = capi.Context(size, num_subtapes=SUBTAPES, **sharding.diagonal_tiles(size, world, r))
        (part.render2D if dim == 2 else part.render3D)(tape)
        assert not part.image()[owner != r].any()
        img[owner == r] = part.image()[owner == r]
        if dim == 3:
            assert not part.normals()[owner != r].any()
            nrm[owner == r] = part.normals()[owner == r]
        part.close()
    assert np.array_equal(img, full.image())
    if dim == 3:
        assert np.array_equal(nrm, full.normals())


@pytest.mark.parametrize("model,dim,size,world,col_step", [("prospero", 2, 1024, 4, 1), ("bear", 3, 512, 8, 1),
                                                          ("hello_world", 3, 256, 2, 0)])
def test_exchange_kernels_reassemble_the_frame(model, dim, size, world, col_step):
    """mprb_exchange_pack / _unpack: every rank's packed blocks, laid end to end as an all-gather
    would leave them, scatter back into the single-context frame (all ranks emulated on one GPU)."""
    import torch
    full, tape = render(model, dim, size)
    parts = []
    for r in range(world):
        opts = sharding.diagonal_tiles(size, world, r) if col_step else sharding.cyclic_rows(size, world, r)
        parts.append(capi.Context(size, num_subtapes=SUBTAPES, **opts))
        (parts[-1].render2D if dim == 2 else parts[-1].render3D)(tape)
    nbytes = parts[0].exchange_bytes(dim)
    assert nbytes == (size // 64) ** 2 // world * 4096 * (6 if dim == 3 else 1)
    gathered = torch.empty(world * nbytes, dtype=torch.uint8, device="cuda")
    for r, p in enumerate(parts):
        p.exchange_pack(dim, gathered.data_ptr() + r * nbytes)
    torch.cuda.synchronize()
    for p in parts:
        p.exchange_unpack(dim, gathered.data_ptr())
    torch.cuda.synchronize()
    for p in parts:
        assert np.array_equal(p.image(), full.image())
        if dim == 3:
            assert np.array_equal(p.normals(), full.normals())
        p.close()
    assert full.exchange_bytes(dim) == 0             # an unsharded context has nothing to exchange
    full.close()


@pytest.mark.parametrize("model,dim,size,world", [("prospero", 2, 1024, 4), ("bear", 3, 512, 8), ("hello_world", 3, 256, 1)])
def test_publish_fills_one_host_frame_from_every_shard(model, dim, size, world):
    """mprb_ctx_publish: each sharded context stores the blocks it owns straight into ONE full-size frame in
    page-locked host memory (no device-side gather); together they make the single-context frame."""
    import torch
    full, tape = render(model, dim, size)
    img = torch.zeros((size, size), dtype=torch.int32).pin_memory()
    nrm = torch.zeros((size, size), dtype=torch.int32).pin_memory() if dim == 3 else None
    for r in range(world):
        opts = sharding.diagonal_tiles(size, world, r) if world > 1 else {}
        part = capi.Context(size, num_subtapes=SUBTAPES, **opts)
        (part.render2D if dim == 2 else part.render3D)(tape)
        part.publish(dim, img.data_ptr(), nrm.data_ptr() if dim == 3 else 0)
        part.close()
    assert np.array_equal(img.numpy(), full.image())
    if dim == 3:
        assert np.array_equal(nrm.numpy().view(np.uint32), full.normals())
    pageable = np.zeros((size, size), dtype=np.int32)
    with pytest.raises(capi.MprbError):
        full.publish(dim, pageable.ctypes.data)
    full.close()


def test_arena_exhaustion_degrades_like_the_reference():
    """With a tiny arena, tiles keep their parent tape (reference context.cu:336-347); the image
    is still correct because every tape that was kept is valid for its tile."""
    full, tape = render("prospero", 2, 512)
    small = capi.Context(512, num_subtapes=200)
    small.render2D(tape)
    assert np.array_equal(small.image(), full.image())
    assert small.stats().tape_index >= 200 * 64 - 64 * 64


def test_full_size_headline_configs():
    """BASELINE configs at full size: golden hash + structural properties."""
    ctx, tape = render("prospero", 2, 4096)
    img = ctx.image()
    assert set(np.unique(img)) <= {0, 1}
    st = ctx.stats()
    assert st.n_active[0] > 0 and st.n_active[1] > 0
    # every filled level-0 tile shows up as a fully set 64x64 block of the final image
    f0 = ctx.filled(0)
    ys, xs = np.nonzero(f0)
    for y, x in list(zip(ys, xs))[:50]:
        assert img[y * 64:(y + 1) * 64, x * 64:(x + 1) * 64].all()
    ctx.close()
    ctx, tape = render("bear", 3, 1024)
    h = ctx.image()
    n = ctx.normals()
    assert h.max() < 1024 and ((h != 0) == (n != 0)).all()     # a normal exactly where there is depth
    assert ((n >> 24) == 0xFF)[n != 0].all()
    ctx.close()


@pytest.mark.parametrize("model,size", [("architecture", 256), ("bear", 256), ("involute_gear_3d", 512)])
def test_effects_match_cpu_restatement(model, size):
    """mpr::Effects::drawSSAO / drawShaded (reference src/effects.cu:253-297) on a real 3D frame.
    The effect kernels are built without FMA contraction, like the restatement, so the two can
    only differ in libdevice powf vs t*t (an ulp inside a sum that is then truncated to 8 bits):
    tolerance = at most 1 grey level, on at most 0.1 % of the pixels."""
    ctx, tape = render(model, 3, size)
    depth, normals = ctx.image().copy(), ctx.normals().copy()
    assert (depth != 0).sum() > size * size // 20
    fx = capi.Effects()
    for shaded in (False, True):
        (fx.drawShaded if shaded else fx.drawSSAO)(ctx)
        got = fx.image().copy()
        want, _ = oracle.effects(depth, normals, fx.kernel, fx.rvecs, shaded=shaded)
        if shaded:
            assert ((got >> 24) & 0xff)[depth != 0].min() == 0xff and (got[depth == 0] == 0).all()
            got, want = got & 0xff, want & 0xff
        diff = np.abs(got.astype(np.int64) - want.astype(np.int64))
        assert diff.max() <= 1, (model, shaded, int(diff.max()))
        assert (diff != 0).mean() <= 1e-3, (model, shaded, float((diff != 0).mean()))
    fx.close()
    ctx.close()


@pytest.mark.parametrize("group", [2, 4])
@pytest.mark.parametrize("name", ["bear_3d_256", "hello_world_3d_128", "hello_world_2d_256"])
def test_float_pass_work_items_of_several_tiles_give_the_reference_frame(name, group):
    """The float pass can walk one tape for 2 or 4 tiles at a time (tiles of a work item share their
    tape; MPRB_FLOAT_GROUP, read once per process): same frame as the reference build, fewer items than
    tiles, and the arena holds shared tapes once."""
    import json
    import os
    import subprocess
    import sys
    model, dim, size = name.rsplit("_", 2)
    want = json.loads((ROOT / "tests" / "golden" / "ref" / f"{name}.json").read_text())
    # MPRB_SUB_WAVES=0: tiles of small levels evaluated by k_eval_sub get a tape each (nothing to share)
    env = dict(os.environ, MPRB_FLOAT_GROUP=str(group), MPRB_SUB_WAVES="0")
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "frame_digest.py"), model, dim[0], size],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["image"] == want["image"]["sha"]
    if dim[0] == "3":
        assert got["normals"] == want["normals"]["sha"]
    assert 0 < got["f_items"] < got["f_tiles"]
    assert 0 < got["p_written"] < got["p_kept"]


@pytest.mark.parametrize("waves", [0, 4, 100000])
@pytest.mark.parametrize("name", ["prospero_2d_256", "prospero_2d_512", "prospero_2d_1024", "bear_3d_256", "bear_3d_512",
                                  "hello_world_2d_256", "hello_world_3d_128", "architecture_3d_256",
                                  "involute_gear_2d_2d_512", "involute_gear_3d_3d_256"])
def test_small_levels_evaluated_clause_parallel_give_the_reference_frame(name, waves, monkeypatch):
    """Levels with few tiles are evaluated one warp per tile on the dependency-level plan k_eval_root
    writes with each shortened tape (k_eval_sub) instead of one lane per tile walking the tape clause
    by clause.  MPRB_SUB_WAVES (read when a context is made) = how many waves of tiles still count as
    few: 0 switches the kernel off, a huge value sends every planned tile through it.  Images, tile
    records and every tile's shortened tape are the reference build's either way."""
    case = [c for c in CASES if c[0] == name][0]
    _, model, dim, size, summary, npz = case
    monkeypatch.setenv("MPRB_SUB_WAVES", str(waves))
    ctx, tape = render(model, dim, size)
    fp = parity.fingerprint(ctx, dim)
    bad = parity.compare_summary(summary, parity.summarize(fp))
    assert not bad, bad
    if npz is not None:
        ref = dict(np.load(npz))
        ref["dim"], ref["size"] = dim, size
        assert not parity.compare(ref, fp)
    st = ctx.stats()
    if waves == 0:
        assert st.i_sub_tiles == 0
    elif waves == 100000 and model != "hello_world":
        assert 0 < st.i_sub_tiles <= st.i_tiles[1]
    ctx.close()


@pytest.mark.parametrize("model,size", [("bear", 256), ("architecture", 512), ("bear", 1024)])
def test_effects_match_reference_build(model, size):
    """mpr::Effects::drawSSAO / drawShaded against the reference's own src/effects.cu, compiled unmodified
    (with the Eigen stand-in of oracle/shim for its small-vector algebra), on the same frame and the same
    sample sets: bit for bit, both result buffers (their digests and the sample sets the reference drew
    are recorded in tests/golden/ref_variants)."""
    want = ref_variant(f"effects/{model}_{size}")
    samples = np.load(VARIANTS / f"effects_{model}_{size}.npz")
    ctx, tape = render(model, 3, size)
    assert parity.digest(ctx.image()) == want["image"] and parity.digest(ctx.normals()) == want["normals"]
    fx = capi.Effects(samples["kernel"], samples["rvecs"])
    for shaded in (False, True):
        effect = "shaded" if shaded else "ssao"
        (fx.drawShaded if shaded else fx.drawSSAO)(ctx)
        got = {"image": parity.digest(fx.image()), "tmp": parity.digest(fx.tmp())}
        assert got == want[effect], (model, size, effect)
    fx.close()
    ctx.close()


@pytest.mark.parametrize("model,size", [("hello_world", 256), ("prospero", 512)])
def test_brute_force_frame(model, size):
    """Context::render2D_brute (context.cu:1461-1508): same image as the subdivided frame, as the
    CPU restatement and the reference build produce it."""
    cells = load_tape(model)
    ctx, tape = render(model, 2, size)
    fancy = ctx.image().copy()
    ctx.render2D_brute(tape)
    got = ctx.image().copy()
    assert np.array_equal(got, fancy)
    assert ctx.tiles(3)["position"].tolist() == list(range((size // 8) ** 2))
    o = oracle.CpuOracle(size, SUBTAPES)
    o.render2D_brute(cells)
    assert np.array_equal(got, o.image())
    o.close()
    assert parity.digest(got) == ref_variant(f"brute/{model}_{size}")["image"]
    ctx.render2D(tape)                       # the context is still good for ordinary frames
    assert np.array_equal(ctx.image(), fancy)
    ctx.close()


@pytest.mark.parametrize("model,size", [("hello_world", 256), ("prospero", 1024), ("involute_gear_2d", 512)])
def test_work_meter_2d_is_exact(model, size):
    """render2D_heatmap (context.cu:1984-2146).  2D frames have no occlusion races, so the meter
    is deterministic: integer-exact against the restatement, and equal to the reference build's
    float atomics up to their summation order."""
    cells = load_tape(model)
    ctx, tape = render(model, 2, size)
    image = ctx.image().copy()
    heat = ctx.render2D_heatmap(tape)
    assert np.array_equal(ctx.image(), image)
    o = oracle.CpuOracle(size, SUBTAPES)
    want, units = o.render2D_heatmap(cells)
    assert np.array_equal(heat, want)
    o.close()
    ref = np.load(VARIANTS / f"heatmap2d_{model}_{size}.npz")["heat"]
    np.testing.assert_allclose(heat, ref, rtol=2e-5, atol=0)
    ctx.close()


@pytest.mark.parametrize("model,size", [("hello_world", 128), ("architecture", 256)])
def test_work_meter_3d(model, size):
    """render3D_heatmap (context.cu:2148-2340).  In 3D the reference's own meter depends on the
    order in which tiles land in the depth image (in-kernel occlusion tests decide which tiles
    push and which voxel columns run), and the more tiles are in flight the fewer are culled: a
    serial CPU run meters ~25 % less than either GPU implementation at 128^3.  So only the frame
    itself is exact; the metered work must cover at least the root walk everywhere and stay within
    a factor of 1.6 of the other implementations in aggregate."""
    cells = load_tape(model)
    ctx, tape = render(model, 3, size)
    depth, normals = ctx.image().copy(), ctx.normals().copy()
    heat = ctx.render3D_heatmap(tape)
    assert np.array_equal(ctx.image(), depth) and np.array_equal(ctx.normals(), normals)
    n = len(cells) - 2
    tps = size // 64
    assert heat.min() >= np.float32(tps / 4096.0) * np.float32(0.999)      # tps level-0 tiles above every pixel
    o = oracle.CpuOracle(size, SUBTAPES)
    want, _ = o.render3D_heatmap(cells)
    assert 1 / 1.6 < float(heat.sum()) / float(want.sum()) < 1.6
    o.close()
    assert 1 / 1.6 < float(heat.sum()) / ref_variant(f"heatmap3d/{model}_{size}")["sum"] < 1.6
    ctx.close()
