"""Records what the reference build (oracle/_ref, GPU) computes for the analysis variants the GPU tests
compare against: post-effects, brute-force frames and the work meters.  Writes into --out

  records.json                       digests (tools/parity.digest) and sums, keyed "<kind>/<model>_<size>"
  effects_<model>_<size>.npz         the SSAO sample sets the reference's mpr::Effects drew for that frame
  heatmap2d_<model>_<size>.npz       the 2D work meter

which tests/test_gpu_parity.py reads from tests/golden/ref_variants.  Needs a GPU and oracle/_ref/libmpr_ref.so.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import oracle  # noqa: E402
import parity  # noqa: E402

EFFECTS = [("bear", 256), ("architecture", 512), ("bear", 1024)]
BRUTE = [("hello_world", 256), ("prospero", 512)]
HEATMAP2D = [("hello_world", 256), ("prospero", 1024), ("involute_gear_2d", 512)]
HEATMAP3D = [("hello_world", 128), ("architecture", 256)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    out = Path(ap.parse_args().out)
    out.mkdir(parents=True, exist_ok=True)
    rec = {}
    for model, size in EFFECTS:
        ref = oracle.RefGpu(size)
        ref.render3D(parity.load_tape(model))
        rfx = oracle.RefEffects()
        kernel, rvecs = rfx.samples()
        np.savez_compressed(out / f"effects_{model}_{size}.npz", kernel=kernel, rvecs=rvecs)
        r = {"image": parity.digest(ref.image()), "normals": parity.digest(ref.normals())}
        for name, shaded in (("ssao", False), ("shaded", True)):
            image, tmp = rfx.draw(ref, shaded=shaded)
            r[name] = {"image": parity.digest(image), "tmp": parity.digest(tmp)}
        rec[f"effects/{model}_{size}"] = r
        rfx.close()
        ref.close()
    for model, size in BRUTE:
        ref = oracle.RefGpu(size)
        ref.render2D_brute(parity.load_tape(model))
        rec[f"brute/{model}_{size}"] = {"image": parity.digest(ref.image())}
        ref.close()
    for model, size in HEATMAP2D:
        ref = oracle.RefGpu(size)
        heat = ref.render2D_heatmap(parity.load_tape(model))
        np.savez_compressed(out / f"heatmap2d_{model}_{size}.npz", heat=heat)
        ref.close()
    for model, size in HEATMAP3D:
        ref = oracle.RefGpu(size)
        heat = ref.render3D_heatmap(parity.load_tape(model))
        rec[f"heatmap3d/{model}_{size}"] = {"sum": float(heat.sum())}
        ref.close()
    (out / "records.json").write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
