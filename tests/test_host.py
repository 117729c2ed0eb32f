"""Host-side logic: the C-ABI library loads and exports what include/mprb.h declares, the
.frep reader + tape packer reproduce the committed tapes, argument validation."""
import ctypes as C
import hashlib
import json
import re

import numpy as np
import pytest

from conftest import GOLDEN, MODELS, ROOT, load_tape
from mpr_b200 import capi

FREP_FILES = GOLDEN / "frep"          # the reference's benchmark models (benchmark/files/*.frep), as shipped


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "mprb.h").read_text()
    declared = set(re.findall(r"\b(mprb_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    L = capi.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in mprb.h but not exported"
    assert declared == set(capi.EXPORTS)
    assert b"sm_100a" in L.mprb_version()


def test_tape_fixture_index_matches_files():
    index = json.loads((GOLDEN / "tapes" / "index.json").read_text())
    for m in MODELS:
        cells = load_tape(m)
        assert cells.size == index[m]["cells"]
        assert hashlib.sha256(cells.tobytes()).hexdigest() == index[m]["sha256"]
        ops = (cells & 0xFF).astype(int)
        assert ops[0] == 0 and ops[-1] == 0                      # header / end cell
        assert ((ops[1:-1] >= 2) & (ops[1:-1] <= 26)).all()       # only clause opcodes, no COPY_*/JUMP
        assert int(((ops >= 17) & (ops <= 20)).sum()) == index[m]["choice_clauses"]


# Clause / slot / choice counts measured in the survey of the reference (SURVEY.md section 8)
SURVEY = {"prospero": (6056, 85, 2354), "involute_gear_2d": (1660, 67, 374), "involute_gear_3d": (1735, 84, 374),
          "architecture": (1296, 93, 488), "bear": (544, 23, 27), "hello_world": (328, 27, 97)}


@pytest.mark.parametrize("model", MODELS)
def test_frep_reader_and_packer_reproduce_committed_tapes(model):
    data = (FREP_FILES / f"{model}.frep").read_bytes()
    cells = capi.tape_from_frep(data, simplify=True)
    assert np.array_equal(cells, load_tape(model))
    clauses, slots, choices = SURVEY[model]
    assert cells.size - 2 == clauses
    used = {int(b) for sh in (8, 16, 24) for b in ((cells >> sh) & 0xFF)}
    assert max(used) + 1 == slots
    ops = (cells & 0xFF).astype(int)
    assert int(((ops >= 17) & (ops <= 20)).sum()) == choices
    # the fixtures are stored already simplified: re-simplifying on load is a no-op
    assert np.array_equal(capi.tape_from_frep(data, simplify=False), cells)


def test_frep_reader_rejects_garbage():
    with pytest.raises(capi.MprbError):
        capi.tape_from_frep(b"\x00\x01\x02", simplify=True)


def _frep(nodes):
    """Builds a minimal archive: 'T' "" "" nodes 0xFF 0xFF (libfive deserializer.cpp:38-143)."""
    import struct
    out = b'T""""'
    for n in nodes:
        if n[0] == "const":
            out += bytes([1]) + struct.pack("<f", n[1])
        elif len(n) == 1:
            out += bytes([n[0]])
        elif len(n) == 2:
            out += bytes([n[0]]) + struct.pack("<I", n[1])
        else:   # binary: rhs is stored first
            out += bytes([n[0]]) + struct.pack("<II", n[2], n[1])
    return out + b"\xff\xff"


def test_archive_bytes_from_libfives_own_tests_are_read_as_written_there():
    """Known answers held by the reference: libfive/libfive/test/archive.cpp:47-105 pins the archive
    byte format with literal strings.  Those exact bytes (packed opcode numbering, as mpr builds
    libfive: CMakeLists.txt:6-8, opcode.hpp:63-101 - VAR_X 2, VAR_Y 3, OP_MIN 22, OP_MAX 23) go through
    the .frep reader + tape packer here and must come out as the one-clause tape of min(x, y)."""
    X, Y, MIN, MAX = 2, 3, 22, 23
    named = b'T"hi"""' + bytes([X, Y, MIN, 1, 0, 0, 0, 0, 0, 0, 0, 0xFF, 0xFF])                  # "With a name"
    escaped = b'T"hi""\\"\\\\"' + bytes([X, Y, MIN, 1, 0, 0, 0, 0, 0, 0, 0, 0xFF, 0xFF])       # "String escaping"
    two = (b'T""""' + bytes([X, Y, MIN, 1, 0, 0, 0, 0, 0, 0, 0, 0xFF, 0xFF]) +                # "Multiple independent trees"
           b'T""""' + bytes([MAX, 1, 0, 0, 0, 0, 0, 0, 0, 0xFF, 0xFF]))
    for blob in (named, escaped, two):
        cells = capi.tape_from_frep(blob)             # the drivers take the archive's first shape
        assert len(cells) == 3
        hdr, clause, end = (int(c) for c in cells)
        sx, sy = (hdr >> 8) & 0xFF, (hdr >> 16) & 0xFF
        assert hdr & 0xFF == 0 and sx and sy and sx != sy and (hdr >> 24) == 0
        assert clause & 0xFF == 18                                        # GPU_OP_MIN_LHS_RHS
        assert ((clause >> 16) & 0xFF, (clause >> 24) & 0xFF) == (sx, sy)  # lhs = x, rhs = y (rhs is stored first)
        assert end & 0xFF == 0 and (end >> 8) & 0xFF == (clause >> 8) & 0xFF


def test_packer_known_answer_circle():
    # max(sqrt(x^2 + y^2) - 1, 0.5 - sqrt(x^2 + y^2)): the default shape of the reference's
    # print_tape_table driver (benchmark/print_tape_table.cpp:29)
    X, Y, CONST, SQUARE, SQRT, ADD, MAX, SUB = 2, 3, 1, 7, 8, 20, 23, 24
    nodes = [(X,), (Y,), (SQUARE, 0), (SQUARE, 1), (ADD, 2, 3), (SQRT, 4), ("const", 1.0), ("const", 0.5),
             (SUB, 5, 6), (SUB, 7, 5), (MAX, 8, 9)]
    cells = capi.tape_from_frep(_frep(nodes))
    ops = [int(c & 0xFF) for c in cells]
    # header, square, square, add, sqrt, sub_lhs_imm, sub_imm_rhs (either order), max_lhs_rhs, end
    assert ops[0] == 0 and ops[-1] == 0 and len(ops) == 9
    assert sorted(ops[1:3]) == [2, 2] and ops[3] == 14 and ops[4] == 3
    assert sorted(ops[5:7]) == [21, 22] and ops[7] == 20
    hdr = int(cells[0])
    assert (hdr >> 8) & 0xFF and (hdr >> 16) & 0xFF and (hdr >> 24) == 0     # x, y bound; z unused
    imms = {int(c & 0xFF): np.frombuffer(np.uint32(int(c) >> 32).tobytes(), dtype="<f4")[0] for c in cells[5:7]}
    assert imms[21] == 1.0 and imms[22] == 0.5
    assert ((int(cells[-1]) >> 8) & 0xFF) == ((int(cells[7]) >> 8) & 0xFF)   # end cell names the result slot
    # operands whose last use is a clause are released first, so outputs reuse slots: <= 3 live + slot 0
    assert max(int((c >> 8) & 0xFF) for c in cells[1:-1]) <= 3


def test_packer_folds_constants_and_dedups():
    X, CONST, ADD, MUL = 2, 1, 20, 21
    # (x + (2 * 3)) * (x + 6): the product of two identical sub-expressions becomes a square
    nodes = [(X,), ("const", 2.0), ("const", 3.0), (MUL, 1, 2), (ADD, 0, 3), ("const", 6.0), (ADD, 0, 5), (MUL, 4, 6)]
    cells = capi.tape_from_frep(_frep(nodes))
    ops = [int(c & 0xFF) for c in cells[1:-1]]
    assert ops == [13, 2]      # ADD_LHS_IMM 6, SQUARE


def test_shared_affine_terms_are_collected():
    # libfive's load-time affine collapse (cache.cpp:463-501): (x + 1) + (x + 2) -> x*2 + 3, and
    # (2*y - x) - (y - 3*x) -> (y + x*2) - 0: terms with equal coefficients are summed first
    X, Y, ADD, MUL, SUB = 2, 3, 20, 21, 24
    nodes = [(X,), ("const", 1.0), ("const", 2.0), (ADD, 0, 1), (ADD, 0, 2), (ADD, 3, 4)]
    cells = capi.tape_from_frep(_frep(nodes))
    imm = lambda c: float(np.frombuffer(np.uint32(int(c) >> 32).tobytes(), dtype="<f4")[0])
    assert [(int(c & 0xFF), imm(c)) for c in cells[1:-1]] == [(15, 2.0), (13, 3.0)]   # MUL_LHS_IMM 2, ADD_LHS_IMM 3
    nodes = [(X,), (Y,), ("const", 2.0), ("const", 3.0), (MUL, 2, 1), (SUB, 4, 0), (MUL, 3, 0), (SUB, 1, 6), (SUB, 5, 7)]
    cells = capi.tape_from_frep(_frep(nodes))
    assert [(int(c & 0xFF), imm(c)) for c in cells[1:-1]] == [(15, 2.0), (14, 0.0)]   # x*2, then y + that
    # without simplification the expression is packed as written
    raw = capi.tape_from_frep(_frep(nodes), simplify=False)
    assert len(raw) - 2 == 5


def test_tape_create_validates_before_touching_the_device():
    L = capi.lib()
    h = C.c_void_p()
    bad = np.array([0, 99, 0], dtype=np.uint64)            # opcode 99 is not a clause
    assert L.mprb_tape_create(bad.ctypes.data, 3, C.byref(h)) == 2
    assert b"opcode" in L.mprb_last_error()
    short = np.array([0], dtype=np.uint64)
    assert L.mprb_tape_create(short.ctypes.data, 1, C.byref(h)) == 2
    no_end = np.array([0, 2 | (1 << 8) | (1 << 16), 5], dtype=np.uint64)
    assert L.mprb_tape_create(no_end.ctypes.data, 3, C.byref(h)) == 2


def test_ctx_create_rejects_bad_sizes():
    L = capi.lib()
    h = C.c_void_p()
    assert L.mprb_ctx_create(100, None, C.byref(h)) == 2
    assert L.mprb_ctx_create(0, None, C.byref(h)) == 2
    assert b"multiple of 64" in L.mprb_last_error()


def test_cpu_heightmap_stand_in_renders_the_driver_default_shape(tmp_path):
    """render_2d.cpp / render_3d.cpp write an out_cpu.png through libfive::Heightmap::render; the
    stand-in the drivers link (mpr_b200/shim/src/heightmap_render.cpp) must get the two-sphere
    default shape right: silhouettes, top height, +z normal on the pole, valid PNG files."""
    import subprocess
    exe = ROOT / "build" / "drivers" / "heightmap_check"
    if not exe.exists():
        pytest.skip("build/drivers/heightmap_check not built (make drivers)")
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    filled3, filled2, wrong, zmax, top = r.stdout.split()
    assert int(wrong) == 0
    assert 380 <= int(filled2) <= 430 and int(filled3) == int(filled2)        # 2 discs of radius 8 voxels: ~402
    assert abs(float(zmax) - 0.234375) < 1e-6                                  # highest voxel centre below z = 0.25
    n = int(top, 16)
    assert n >> 24 == 0xff and (n >> 16) & 0xff >= 0xf8 and abs((n & 0xff) - 0x80) <= 8
    for name, kind in (("depth.png", 0), ("norm.png", 6)):
        png = (tmp_path / name).read_bytes()
        assert png[:8] == b"\x89PNG\r\n\x1a\n"
        w, h, depth, colour = __import__("struct").unpack(">IIBB", png[16:26])
        assert (w, h) == (64, 64) and colour == kind and depth == (16 if kind == 0 else 8)


def test_dump_tape_reproduces_the_kernel_libfive_generated_for_brute_cu():
    """benchmark/brute.cu:44-58 holds the body that the reference's dump_tape (built on the real
    libfive) printed for the default two-sphere shape.  The same driver built on this repository's
    Tree stand-in must print the same statements in the same order - a known answer for operator
    overloads, hash-consing, commutative rebalancing and orderedDfs together."""
    import subprocess
    exe = ROOT / "oracle" / "_ref" / "drivers" / "dump_tape"
    if not exe.exists():
        pytest.skip("oracle/_ref/drivers/dump_tape not built (needs the reference sources at build time)")
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60).stdout
    names = {}
    body = []
    for line in out.splitlines():
        m = re.match(r"\s*const float (v\d+) = (.*);", line)
        if not m:
            continue
        names[m.group(1)] = f"v{len(names)}"
        body.append(re.sub(r"v\d+", lambda k: names[k.group(0)], m.group(2)))
    assert body == [
        "x + 0.500000f", "v0 * v0", "y * y", "z * z", "v2 + v3", "v1 + v4", "sqrt(v5)", "v6 - 0.250000f",
        "x - 0.500000f", "v8 * v8", "v9 + v4", "sqrt(v10)", "v11 - 0.250000f", "min(v7, v12)"]
    assert "if (v13 < 0.0f)" in re.sub(r"v\d+", lambda k: names.get(k.group(0), k.group(0)), out)


def test_generated_ptx_loops_are_current_and_cover_the_opcode_table(tmp_path):
    """csrc/float_loop_ptx.inc and interval_loop_ptx.inc are generated (tools/gen_*_loop.py): the
    committed files must be what the generators emit, every dispatch table must have 256 entries,
    and the opcode classes kernels.cu feeds the annotation pass must be the generators'."""
    import importlib.util
    src = (ROOT / "mpr_b200" / "csrc" / "kernels.cu").read_text()
    for tool, inc in (("gen_float_loop", "float_loop_ptx.inc"), ("gen_interval_loop", "interval_loop_ptx.inc")):
        spec = importlib.util.spec_from_file_location(tool, ROOT / "tools" / f"{tool}.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        path = ROOT / "mpr_b200" / "csrc" / inc
        before = path.read_text()
        mod.main()
        assert path.read_text() == before, f"{inc} is stale: run tools/{tool}.py"
        i = before.index(".branchtargets")
        # 256 entries, or 128 where the store / no-store variants of a handler are one piece of code
        # (bit 7 of the opcode byte is then masked off before the indexed branch)
        n_entries = before[i:before.index(";", i)].count("_%=")
        assert (n_entries, "0x7f;" in before) in ((256, False), (128, True)), inc
        fast = sum(1 << o for o in mod.OPS)
        assert f"0x{fast:08x}u" in src, (tool, hex(fast))
    # every handler the table names is defined exactly once
    for inc in ("float_loop_ptx.inc", "interval_loop_ptx.inc"):
        text = (ROOT / "mpr_b200" / "csrc" / inc).read_text()
        names = set(re.findall(r"(H\d+_\d{2,3}x?)_%=", text[text.index(".branchtargets"):text.index("LOOP_%=:")]))
        for n in names:
            assert len(re.findall(rf'"{n}_%=:', text)) == 1, n


def test_interval_multiply_operand_selection_matches_the_nine_case_table():
    """The MUL_LHS_RHS handler of the PTX interval loop picks its four operands with predicate
    algebra; the table it must equal is iv_mul in csrc/ival.cuh (reference gpu_interval.hpp:85-146)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_interval_loop", ROOT / "tools" / "gen_interval_loop.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    # (class a, class b) -> (lower: a?, b?; upper: a?, b?); class bit0 = lo < 0, bit1 = hi > 0
    table = {(3, 1): ("ah", "bl", "al", "bl"), (3, 2): ("al", "bh", "ah", "bh"),
             (1, 3): ("al", "bh", "al", "bl"), (1, 1): ("ah", "bh", "al", "bl"), (1, 2): ("al", "bh", "ah", "bl"),
             (2, 3): ("ah", "bl", "ah", "bh"), (2, 1): ("ah", "bl", "al", "bh"), (2, 2): ("al", "bl", "ah", "bh")}
    for (ca, cb), want in table.items():
        s = mod.mul_select(bool(ca & 1), bool(ca & 2), bool(cb & 1), bool(cb & 2))
        got = ("ah" if s[0] else "al", "bl" if s[1] else "bh", "al" if s[2] else "ah", "bl" if s[3] else "bh")
        assert got == want, (ca, cb)


# ---- the generated interval handlers, executed on the CPU -------------------------------------

def _interval_handler(op):
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_interval_loop", ROOT / "tools" / "gen_interval_loop.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return " ".join(mod.compute(op))


_IV_OPS = {"SQUARE": 2, "SQRT": 3, "NEG": 4, "SIN": 5, "ABS": 11, "ADD_LI": 13, "ADD_LR": 14, "MUL_LI": 15, "MUL_LR": 16,
           "MIN_LI": 17, "MIN_LR": 18, "MAX_LI": 19, "MAX_LR": 20, "SUB_LI": 21, "SUB_IR": 22, "SUB_LR": 23, "DIV_LI": 24}


@pytest.mark.parametrize("name", sorted(_IV_OPS))
def test_generated_interval_handlers_equal_the_c_restatement(name):
    """Runs the PTX text of each interval handler (tools/gen_interval_loop.py) through a small
    interpreter with exact directed rounding (tests/ptx_emulator.py) and compares bounds and min/max
    verdicts with oracle/mpr_oracle.c, on ordinary intervals and on the awkward ones: zero-width,
    zero-straddling, infinite, inverted and NaN bounds."""
    import oracle
    from ptx_emulator import Machine, b2f, f2b
    L = oracle.oracle_lib()
    L.mpro_interval_op.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    op = _IV_OPS[name]
    text = _interval_handler(op)
    rng = np.random.default_rng(op)
    special = [0.0, -0.0, 1.0, -1.0, 0.5, -2.5, 3.0, 1e-30, -1e-30, 1e30, -1e30, np.inf, -np.inf, np.nan,
               float(np.finfo(np.float32).max), float(np.finfo(np.float32).tiny), 1e-45]
    cases = []
    for _ in range(120):
        a = np.sort(rng.normal(0, 2, 2)).astype(np.float32)
        b = np.sort(rng.normal(0, 2, 2)).astype(np.float32)
        cases.append((a, b))
    for _ in range(120):
        a = np.array(rng.choice(special, 2), dtype=np.float32)
        b = np.array(rng.choice(special, 2), dtype=np.float32)
        cases.append((a, b))
    swap_r = name in ("SUB_IR",)            # the oracle hook takes the interval operand first
    for a, b in cases:
        imm = np.float32(b[0])
        regs = {"ll": f2b(a[0]), "lh": f2b(a[1]), "rl": f2b(b[0]), "rh": f2b(b[1]), "im": f2b(imm),
                "cw": 0, "n": 5, "any": 0, "chbase": 0}
        if swap_r:
            regs.update(rl=f2b(a[0]), rh=f2b(a[1]))
        m = Machine(regs, {"%3": "cw", "%4": "n", "%5": "any", "%7": "chbase"}).run(text)
        got = np.array([b2f(m.r["ol"]), b2f(m.r["oh"])], dtype=np.float32)
        want = np.zeros(2, dtype=np.float32)
        fa = np.ascontiguousarray(a)
        fb = np.ascontiguousarray(b)
        ch = L.mpro_interval_op(op, fa.ctypes.data, fb.ctypes.data, want.ctypes.data)
        same = (got == want) | (np.isnan(got) & np.isnan(want))
        assert same.all(), (name, a, b, got, want)
        if 17 <= op <= 20:
            assert m.r["c"] == ch, (name, a, b, m.r["c"], ch)
            # verdict record: bits (n & 15) * 2 of cw, counter advanced, flag raised iff decided
            assert m.r["cw"] == (ch << 10) and m.r["n"] == 6 and (m.r["any"] != 0) == (ch != 0)
            assert not m.stores


def test_generated_verdict_record_flushes_every_sixteenth_verdict():
    from ptx_emulator import Machine, f2b
    text = _interval_handler(18)            # MIN_LHS_RHS
    base = {"ll": f2b(0.0), "lh": f2b(1.0), "rl": f2b(2.0), "rh": f2b(3.0), "im": 0, "chbase": 1000}
    # 16th verdict of a word (n = 31): the word goes to choices[1] and restarts
    m = Machine(dict(base, cw=0x12345, n=31, any=0), {"%3": "cw", "%4": "n", "%5": "any", "%7": "chbase"}).run(text)
    assert m.r["c"] == 1 and m.stores == [(1000 + 4 * 1, 0x12345 | (1 << 30))] and m.r["cw"] == 0 and m.r["n"] == 32
    # past the 4096-verdict record nothing is stored, the word still restarts (context.cu:257-259)
    m = Machine(dict(base, cw=7, n=4111, any=0), {"%3": "cw", "%4": "n", "%5": "any", "%7": "chbase"}).run(text)
    assert m.stores == [] and m.r["cw"] == 0 and m.r["n"] == 4112 and m.r["any"] == 1


@pytest.mark.parametrize("tool", ["gen_float_loop", "gen_interval_loop"])
def test_forwarding_hints_preserve_the_slot_state_on_random_tapes(tool):
    """Model check of the hint scheme the PTX loops rely on (kernels.cu:annotate_chunk +
    tools/gen_*_loop.py): FL / FR take an operand from the previous result instead of its slot, NS
    skips a store the next clause overwrites.  On random chunks - slot ids colliding on purpose,
    operands equal to the destination, slow cells and jumps in between - running with the hints must
    leave exactly the slot values of plain sequential execution at every point where the loop hands
    control back (those are the only points where anything else reads the slots)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(tool, ROOT / "tools" / f"{tool}.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    fast_ops, uses_l, uses_r = sorted(mod.OPS), mod.USES_L, mod.USES_R
    slow_ops = [o for o in range(2, 30) if o not in mod.OPS] + [0, 1]
    P = (1 << 61) - 1

    def apply(op, l, r, imm):                      # an arbitrary non-commutative stand-in for the arithmetic
        l = l if op in uses_l else 0
        r = r if op in uses_r else 0
        return (op * 1000003 + l * 7919 + r * 104729 + imm * 31 + 17) % P

    def annotate(cells):                            # mirrors annotate_chunk<FAST, LHS, RHS>
        fast = lambda c: c is not None and c["op"] in mod.OPS
        out = []
        for j, c in enumerate(cells):
            prev = cells[j - 1] if j > 0 else None
            nxt = cells[j + 1] if j + 1 < len(cells) else None
            fl = fr = ns = False
            if fast(c):
                if fast(prev):
                    fl = c["op"] in uses_l and c["lhs"] == prev["out"]
                    fr = c["op"] in uses_r and c["rhs"] == prev["out"]
                ns = fast(nxt) and nxt["out"] == c["out"]
            out.append((fl, fr, ns))
        return out

    rng = np.random.default_rng(7)
    for trial in range(300):
        n = 64
        cells = []
        for j in range(n):
            op = int(rng.choice(fast_ops)) if rng.random() < 0.85 else int(rng.choice(slow_ops))
            cells.append(dict(op=op, out=int(rng.integers(1, 6)), lhs=int(rng.integers(0, 6)), rhs=int(rng.integers(0, 6)),
                              imm=int(rng.integers(0, 100))))
        hints = annotate(cells)
        plain = {s: 1000 + s for s in range(6)}
        smem = dict(plain)
        reg = None                                  # (ox, oy) of the PTX loop
        for j, c in enumerate(cells):
            if c["op"] not in mod.OPS:              # the loop exits here: slots must agree
                assert smem == plain, (tool, trial, j)
                reg = None
                if c["op"] >= 2:                    # a slow clause runs in C++ on the slots
                    v = apply(c["op"], plain[c["lhs"]], plain[c["rhs"]], c["imm"])
                    plain[c["out"]] = smem[c["out"]] = v
                continue
            fl, fr, ns = hints[j]
            want = apply(c["op"], plain[c["lhs"]], plain[c["rhs"]], c["imm"])
            plain[c["out"]] = want
            assert not (fl or fr) or reg is not None
            l = reg if fl else smem[c["lhs"]]
            r = reg if fr else smem[c["rhs"]]
            got = apply(c["op"], l, r, c["imm"])
            assert got == want, (tool, trial, j, c, hints[j])
            if not ns:
                smem[c["out"]] = got
            reg = got


def _mini_annotate(cells, mod):
    """annotate_chunk (kernels.cu) on a list of raw 64-bit cells; returns cells with hint bits."""
    fast = lambda c: c is not None and (c & 0xff) in mod.OPS
    out = []
    for j, c in enumerate(cells):
        prev = cells[j - 1] if j > 0 else None
        nxt = cells[j + 1] if j + 1 < len(cells) else None
        flags = 0
        if fast(c):
            op = c & 0xff
            if fast(prev):
                if op in mod.USES_L and ((c >> 16) & 0xff) == ((prev >> 8) & 0xff):
                    flags |= 0x20
                if op in mod.USES_R and ((c >> 24) & 0xff) == ((prev >> 8) & 0xff):
                    flags |= 0x40
            if fast(nxt) and ((nxt >> 8) & 0xff) == ((c >> 8) & 0xff):
                flags |= 0x80
        out.append(c | flags)
    return out


def test_generated_interval_loop_runs_whole_tapes_like_the_c_restatement():
    """The complete generated interval loop - table dispatch, byte-permute addressing, hinted
    handler variants, stores, verdict record - executed on the CPU for one lane over random
    annotated tapes, against clause-by-clause evaluation with oracle/mpr_oracle.c."""
    import importlib.util
    import oracle
    from ptx_emulator import LoopMachine, b2f, f2b, load_asm
    spec = importlib.util.spec_from_file_location("gen_interval_loop", ROOT / "tools" / "gen_interval_loop.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    asm = load_asm(ROOT / "mpr_b200" / "csrc" / "interval_loop_ptx.inc")
    L = oracle.oracle_lib()
    L.mpro_interval_op.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    ops = [o for o in sorted(mod.OPS) if o != 10]          # exp uses ex2.approx: not emulated
    rng = np.random.default_rng(11)
    CH, SB, CHOICES = 0x1000, 0x4000, 0x100000
    for trial in range(40):
        n = int(rng.integers(5, 40))
        cells = []
        for _ in range(n):
            op = int(rng.choice(ops))
            imm = np.float32(rng.choice([0.0, 1.5, -2.0, 0.25, -0.75, 3.0]))
            cells.append(op | int(rng.integers(1, 7)) << 8 | int(rng.integers(0, 7)) << 16 | int(rng.integers(0, 7)) << 24
                         | f2b(imm) << 32)
        cells.append(0 | (int(rng.integers(1, 7)) << 8))            # END cell
        noted = _mini_annotate(cells, mod)
        smem = {}
        for j, c in enumerate(noted):
            smem[CH + 8 * j], smem[CH + 8 * j + 4] = c & 0xffffffff, c >> 32
        slots = {s: np.sort(rng.normal(0, 2, 2)).astype(np.float32) for s in range(7)}
        for s, v in slots.items():
            smem[SB + 256 * s], smem[SB + 256 * s + 4] = f2b(v[0]), f2b(v[1])
        m = LoopMachine(asm, {"cp": CH - 8, "sb": SB, "cw": 0, "n": 3, "any": 0, "ch": CHOICES, "w": 0, "imm": 0},
                        {"%0": "cp", "%1": "w", "%2": "imm", "%3": "cw", "%4": "n", "%5": "any", "%6": "sb", "%7": "ch"},
                        smem).execute()
        assert m.r["cp"] == CH + 8 * n and (m.r["w"] & 0xff) == 0       # stopped on the END cell
        # clause-by-clause reference
        cw, cnt, anyc = 0, 3, 0
        for c in cells[:-1]:
            op, out, lhs, rhs = c & 0xff, (c >> 8) & 0xff, (c >> 16) & 0xff, (c >> 24) & 0xff
            imm = np.array([b2f(c >> 32), 0], dtype=np.float32)
            a = slots[lhs].copy()
            b = slots[rhs].copy()
            if op in (22,):                                 # SUB_IMM_RHS: the hook takes the interval first
                a = b
            second = imm if op in (13, 15, 17, 19, 21, 22, 24, 27) else b
            res = np.zeros(2, dtype=np.float32)
            if op == 27:
                res[:] = imm[0]
                ch = 0
            elif op == 28:
                res, ch = slots[lhs].copy(), 0
            elif op == 29:
                res, ch = slots[rhs].copy(), 0
            else:
                ch = L.mpro_interval_op(op, a.ctypes.data, np.ascontiguousarray(second).ctypes.data, res.ctypes.data)
            if 17 <= op <= 20:
                cw |= ch << ((cnt & 15) * 2)
                if (cnt & 15) == 15:
                    cw = 0
                cnt += 1
                anyc |= ch
            slots[out] = res
        for s, v in slots.items():
            got = np.array([b2f(smem[SB + 256 * s]), b2f(smem[SB + 256 * s + 4])], dtype=np.float32)
            assert ((got == v) | (np.isnan(got) & np.isnan(v))).all(), (trial, s, got, v)
        assert (m.r["cw"], m.r["n"], m.r["any"] != 0) == (cw, cnt, anyc != 0)


@pytest.mark.parametrize("G,inc", [(1, "float_loop_ptx.inc"), (2, "float_loop_ptx_g2.inc"), (4, "float_loop_ptx_g4.inc"),
                                   (2, "float_loop_ptx_g2t.inc"), (4, "float_loop_ptx_g4t.inc")])
def test_generated_float_loop_runs_whole_tapes_like_plain_float32_evaluation(G, inc):
    """Same for the float pass's loops (G tiles per warp, two samples per tile and lane; slot bytes
    pre-multiplied by G as annotate_chunk does), against numpy float32 arithmetic with the
    clause semantics of eval_voxels_f (reference context.cu:887-920).  exp / log are left out: their
    handlers are libdevice's PTX (ex2.approx), which the interpreter does not model."""
    import importlib.util
    from ptx_emulator import LoopMachine, b2f, f2b, fmax, fmin, load_asm
    spec = importlib.util.spec_from_file_location("gen_float_loop", ROOT / "tools" / "gen_float_loop.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    asm = load_asm(ROOT / "mpr_b200" / "csrc" / inc)
    ops = [o for o in sorted(mod.OPS) if o not in (10, 12)]
    rng = np.random.default_rng(5)
    CH, SB, TB = 0x1000, 0x4000, 0x40
    f32 = np.float32
    # ...t.inc: the first G / 2 tiles in shared-memory rows (G / 2 tiles wide), the others in tensor memory,
    # slot s = columns G s .. G s + G - 1 (two per tile)
    TM = inc.endswith("t.inc")
    GS = G // 2 if TM else G          # tiles per shared-memory row = what annotate_chunk multiplies the slot bytes by

    def clause(op, l, r, imm):
        with np.errstate(all="ignore"):
            return {2: lambda: l * l, 3: lambda: np.sqrt(l), 4: lambda: -l, 11: lambda: np.abs(l),
                    13: lambda: l + imm, 14: lambda: l + r, 15: lambda: l * imm, 16: lambda: l * r,
                    17: lambda: fmin(l, imm), 18: lambda: fmin(l, r), 19: lambda: fmax(l, imm), 20: lambda: fmax(l, r),
                    21: lambda: l - imm, 22: lambda: imm - r, 23: lambda: l - r,
                    24: lambda: l / imm, 25: lambda: imm / r, 26: lambda: l / r,
                    27: lambda: imm, 28: lambda: l, 29: lambda: r}[op]()

    for trial in range(40 if G == 1 else 15):
        n = int(rng.integers(5, 40))
        cells = []
        for _ in range(n):
            op = int(rng.choice(ops))
            imm = f32(rng.choice([0.0, 1.5, -2.0, 0.25, -0.75, 3.0]))
            cells.append(op | int(rng.integers(1, 7)) << 8 | int(rng.integers(0, 7)) << 16 | int(rng.integers(0, 7)) << 24
                         | f2b(imm) << 32)
        cells.append(0 | (int(rng.integers(1, 7)) << 8))
        noted = _mini_annotate(cells, mod)
        smem = {}
        for j, c in enumerate(noted):
            w = c & 0xffffffff
            w = (w & 0xff) | (((w >> 8) * GS) << 8)         # slot ids -> row offsets in 256-byte units
            smem[CH + 8 * j], smem[CH + 8 * j + 4] = w, c >> 32
        slots = {s: rng.normal(0, 2, 2 * G).astype(f32) for s in range(7)}
        m = LoopMachine(asm, {"cp": CH - 8, "sb": SB, "tb": TB, "w": 0, "imm": 0},
                        {"%0": "cp", "%1": "w", "%2": "imm", "%3": "sb", "%4": "tb"}, smem)
        for s, v in slots.items():
            for k in range(2 * GS):
                smem[SB + 256 * GS * s + 4 * k] = f2b(v[k])
            if TM:
                for k in range(G):
                    m.tmem[TB + G * s + k] = f2b(v[G + k])
        m.execute()
        assert m.r["cp"] == CH + 8 * n and (m.r["w"] & 0xff) == 0
        for c in cells[:-1]:
            op, out, lhs, rhs = c & 0xff, (c >> 8) & 0xff, (c >> 16) & 0xff, (c >> 24) & 0xff
            imm = b2f(c >> 32)
            slots[out] = np.array([clause(op, slots[lhs][k], slots[rhs][k], imm) for k in range(2 * G)], dtype=f32)
        for s, v in slots.items():
            got = [b2f(smem[SB + 256 * GS * s + 4 * k]) for k in range(2 * GS)]
            if TM:
                got += [b2f(m.tmem[TB + G * s + k]) for k in range(G)]
            got = np.array(got, dtype=f32)
            assert ((got == v) | (np.isnan(got) & np.isnan(v))).all(), (trial, s, got, v)


@pytest.mark.parametrize("model", ["prospero", "architecture", "bear", "involute_gear_2d", "hello_world"])
def test_planned_marking_keeps_the_clauses_the_reference_slot_walk_keeps(model):
    """k_eval_sub marks a dependency-level plan instead of walking the parent's shortened tape backwards
    slot by slot (tests/plan_model.py models both).  On arbitrary verdicts the clauses a child keeps must
    be the same - including those the reference keeps only because a copy left behind by a verdict still
    names its unused operand's slot, and including marks that land on a level the top-down sweep has
    already passed (at least one of these cases needs the second sweep)."""
    import plan_model
    cells = load_tape(model)
    most_sweeps = 0
    for seed, (p_root, p_child) in enumerate([(0.2, 0.1), (0.1, 0.3), (0.5, 0.05), (0.05, 0.05), (0.3, 0.6)]):
        ref, mine, sweeps = plan_model.compare(cells, seed, p_root, p_child)
        assert ref == mine, (model, seed, len(ref), len(mine))
        most_sweeps = max(most_sweeps, sweeps)
    if model == "prospero":
        assert most_sweeps >= 2


@pytest.mark.parametrize("ulps", [-2, -1, 0, 1, 2])
@pytest.mark.parametrize("G,inc", [(1, "float_loop_ptx.inc"), (2, "float_loop_ptx_g2.inc"), (2, "float_loop_ptx_g2t.inc"),
                                   (4, "float_loop_ptx_g4t.inc")])
def test_hand_expanded_sqrt_and_division_by_an_immediate_round_like_ieee(G, inc, ulps):
    """The float loops expand sqrt and x / immediate themselves (tools/gen_float_loop.py, sqrt_fast /
    div_imm_fast: one range vote for all elements of a clause, the reciprocal refined once).  The clause
    semantics are the reference's `sqrtf(lhs)` and `lhs / imm` (context.cu:887-920), i.e. IEEE-754
    correctly rounded results - here for operands inside and outside the fast range (outside, the loop
    falls back to sqrt.rn / div.rn).  MUFU.RSQ / MUFU.RCP are modelled as the correctly rounded value moved by
    `ulps` units in the last place (the reciprocal by one at most, its documented bound): the sqrt sequence
    tolerates that, and so does the division because divisors with an all-ones mantissa - the one class where
    one Newton step does not repair a reciprocal that is a unit off - are sent to div.rn.  G = 1: every handler variant
    carries its own copy; G > 1: one shared body behind stubs, values in shared and (…t.inc) tensor memory."""
    import ptx_emulator
    from ptx_emulator import LoopMachine, b2f, f2b, load_asm
    asm = load_asm(ROOT / "mpr_b200" / "csrc" / inc)
    rng = np.random.default_rng(11 + ulps + 7 * G)
    f32 = np.float32
    CH, SB, TB = 0x1000, 0x4000, 0x40
    TM = inc.endswith("t.inc")
    GS = G // 2 if TM else G
    n = 2 * G                                                     # values per slot and lane

    def rnd(lo, hi, signed):
        m = rng.integers(0, 1 << 23)
        if rng.random() < 0.15:
            m = int(rng.choice([0, 1, (1 << 23) - 1, (1 << 23) - 2, 1 << 22, (1 << 22) + 1, (1 << 22) - 1]))
        bits = (int(rng.integers(lo, hi + 1)) + 127) << 23 | int(m)
        if signed and rng.random() < 0.5:
            bits |= 0x80000000
        return b2f(bits)

    ptx_emulator.RSQ_ULPS = ulps
    ptx_emulator.RCP_ULPS = max(-1, min(1, ulps))                 # MUFU.RCP: one unit in the last place at most
    try:
        for trial in range(400 if G == 1 else 60):
            wide = trial % 4 == 3                                # every fourth case leaves the fast range
            imm = rnd(-80, 80, True) if wide else rnd(-60, 60, True)
            a = [rnd(-110, 110, False) if wide else rnd(-100, 100, False) for _ in range(n)]   # sqrt operands
            d = [rnd(-80, 80, True) if wide else rnd(-60, 60, True) for _ in range(n)]         # dividends
            if trial % 10 == 9:
                d[0] = f32(float(imm) * float(rnd(0, 0, False)))                                # quotient near 1
            # slot 3 = sqrt(slot 1) stored; slot 2 = slot 2 / imm stored; then the same two through the forwarded
            # variants: slot 4 = slot 1 + 0 (result stays in registers), slot 4 = sqrt(slot 4); slot 5 = slot 2 + 0 ...
            cells = [3 | 3 << 8 | 1 << 16, 24 | 2 << 8 | 2 << 16 | f2b(imm) << 32, 0 | 1 << 8]
            smem = {}
            for j, c in enumerate(cells):
                w = c & 0xffffffff
                w = (w & 0xff) | (((w >> 8) * GS) << 8)
                smem[CH + 8 * j], smem[CH + 8 * j + 4] = w, c >> 32
            m = LoopMachine(asm, {"cp": CH - 8, "sb": SB, "tb": TB, "w": 0, "imm": 0},
                            {"%0": "cp", "%1": "w", "%2": "imm", "%3": "sb", "%4": "tb"}, smem)
            for s_, vals in ((1, a), (2, d)):
                for k in range(2 * GS):
                    smem[SB + 256 * GS * s_ + 4 * k] = f2b(vals[k])
                if TM:
                    for k in range(G):
                        m.tmem[TB + G * s_ + k] = f2b(vals[G + k])
            m.execute()

            def got(s_):
                v = [smem[SB + 256 * GS * s_ + 4 * k] for k in range(2 * GS)]
                if TM:
                    v += [m.tmem[TB + G * s_ + k] for k in range(G)]
                return v
            with np.errstate(all="ignore"):
                assert got(3) == [f2b(np.sqrt(f32(x))) for x in a], (trial, a)
                assert got(2) == [f2b(f32(x) / f32(imm)) for x in d], (trial, d, imm)
    finally:
        ptx_emulator.RSQ_ULPS = 0
        ptx_emulator.RCP_ULPS = 0


@pytest.mark.parametrize("model,dim,size", [("involute_gear_3d", 3, 128), ("architecture", 3, 128), ("prospero", 2, 512)])
def test_rows_numbered_by_liveness_walk_a_tape_like_slot_ids_and_need_far_fewer_rows(model, dim, size):
    """DESIGN section 9, item 1 (what the models with renamed slots need next): a backward linear scan - the
    walk a tape push already does with its live-slot set - numbers rows so that a tape needs one per value
    live at once instead of one per distinct slot id.  On the last-level tapes the CPU restatement produces
    for the shipped models: walking by rows gives the value walking by slot ids gives, the rows used equal
    the values live at once (optimal), and they are well under the rows first-sight renaming hands out."""
    import oracle
    import row_model
    cells = load_tape(model)
    o = oracle.CpuOracle(size)
    (o.render3D if dim == 3 else o.render2D)(cells)
    arena = np.ascontiguousarray(o.arena())
    t = o.tiles(2)
    tapes = np.unique(t[t["position"] != -1]["tape"])
    assert len(tapes) > 20
    rng = np.random.default_rng(3)
    by_life, by_sight = [], []
    for tp in rng.choice(tapes, size=min(60, len(tapes)), replace=False):
        flat = oracle.tape_flatten(arena, int(tp))
        _, rows, _, n_rows, most = row_model.allocate(flat)
        assert n_rows == most                                    # never more rows than values live at once
        assert all(0 < ro <= n_rows and rl <= n_rows and rr <= n_rows for ro, rl, rr in rows)
        for _ in range(2):
            xyz = rng.normal(0, 1, 3).astype(np.float32)
            a, b = row_model.run_by_ids(flat, xyz), row_model.run_by_rows(flat, xyz)
            assert a == b or (np.isnan(a) and np.isnan(b)), (model, int(tp), a, b)
        by_life.append(n_rows)
        by_sight.append(row_model.first_sight_rows(flat))
    o.close()
    assert np.mean(by_life) < 0.75 * np.mean(by_sight), (np.mean(by_life), np.mean(by_sight))


def test_generated_float_loop_hands_back_clauses_marked_for_the_spilling_path():
    """With renamed slots TapeStream::rename (tape_stream.cuh) gives a clause that touches a row beyond the
    shared-memory rows the opcode kOpBounce = 31; the float pass relies on the generated G = 1 loop leaving
    at such a cell exactly as it leaves at END / JUMP - pointer on the cell, its two words returned, nothing
    of it executed - and on picking up again behind it (walk_float, kernels.cu)."""
    from ptx_emulator import LoopMachine, b2f, f2b, load_asm
    asm = load_asm(ROOT / "mpr_b200" / "csrc" / "float_loop_ptx.inc")
    text = (ROOT / "mpr_b200" / "csrc" / "tape_stream.cuh").read_text()
    assert "constexpr uint32_t kOpBounce = 31;" in text
    CH, SB = 0x1000, 0x4000
    f32 = np.float32
    cells = [13 | 1 << 8 | 1 << 16 | f2b(f32(2.0)) << 32,           # s1 = s1 + 2
             31 | 2 << 8 | 1 << 16 | 3 << 24 | f2b(f32(7.0)) << 32,  # marked: rows 2, 1, 3 (whatever it was)
             15 | 1 << 8 | 1 << 16 | f2b(f32(3.0)) << 32,           # s1 = s1 * 3
             0 | 1 << 8]
    smem = {}
    for j, c in enumerate(cells):
        smem[CH + 8 * j], smem[CH + 8 * j + 4] = c & 0xffffffff, c >> 32
    for k, v in enumerate((1.5, -4.0)):
        smem[SB + 256 * 1 + 4 * k] = f2b(f32(v))
        smem[SB + 256 * 2 + 4 * k] = f2b(f32(100.0))
    regs = {"cp": CH - 8, "sb": SB, "tb": 0, "w": 0, "imm": 0}
    ops = {"%0": "cp", "%1": "w", "%2": "imm", "%3": "sb", "%4": "tb"}
    m = LoopMachine(asm, regs, ops, smem).execute()
    assert m.r["cp"] == CH + 8 and (m.r["w"] & 0xff) == 31 and m.r["w"] >> 8 == 0x030102 and m.r["imm"] == f2b(f32(7.0))
    assert [b2f(smem[SB + 256 + 4 * k]) for k in range(2)] == [f32(3.5), f32(-2.0)]      # clause 0 ran
    assert [b2f(smem[SB + 512 + 4 * k]) for k in range(2)] == [f32(100.0), f32(100.0)]   # the marked one did not
    m = LoopMachine(asm, {**regs, "cp": m.r["cp"]}, ops, smem).execute()                # the walker re-enters behind it
    assert m.r["cp"] == CH + 24 and (m.r["w"] & 0xff) == 0
    assert [b2f(smem[SB + 256 + 4 * k]) for k in range(2)] == [f32(10.5), f32(-6.0)]
