"""Regenerates tests/golden/tapes/*.u64 from the reference's .frep models.

The packed tapes are what both the reference kernels and this repository's
kernels consume, so they are the common input of every parity test (the parity
contract starts at the packed tape, SURVEY.md section 8c).  They are produced by
this repository's own .frep reader + tape packer (libmprb: mprb_tape_from_frep),
with libfive's load-time simplification rules switched on.

The .frep models under tests/golden/frep are the reference's benchmark/files, unchanged.

No GPU needed:  python tests/golden/make_tapes.py
"""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from mpr_b200 import capi  # noqa: E402

SRC = Path(__file__).resolve().parent / "frep"
OUT = Path(__file__).resolve().parent / "tapes"
MODELS = ["prospero", "involute_gear_2d", "involute_gear_3d", "architecture", "bear", "hello_world"]


def main():
    OUT.mkdir(exist_ok=True)
    index = {}
    for m in MODELS:
        cells = capi.tape_from_frep((SRC / f"{m}.frep").read_bytes(), simplify=True)
        (OUT / f"{m}.u64").write_bytes(cells.astype("<u8").tobytes())
        ops = (cells & 0xFF).astype(int)
        index[m] = {
            "cells": int(cells.size),
            "clauses": int(cells.size - 2),
            "choice_clauses": int(((ops >= 17) & (ops <= 20)).sum()),
            "sha256": hashlib.sha256(cells.astype("<u8").tobytes()).hexdigest(),
        }
        print(m, index[m])
    (OUT / "index.json").write_text(json.dumps(index, indent=1) + "\n")


if __name__ == "__main__":
    main()
