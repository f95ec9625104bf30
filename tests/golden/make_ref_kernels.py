"""Generates tests/golden/ref_kernels.npz and tests/golden/ref_frames.npz: what the REFERENCE'S OWN CUDA kernels compute on the inputs of
tests/test_ref_parity_gpu.py and tests/test_frame_parity_gpu.py.  Needs a GPU and the reference's extensions built into oracle/_ref by
oracle/build_ref.py.

    python tests/golden/make_ref_kernels.py [OUT_DIR]        # default: tests/golden
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]

import build_ref  # noqa: E402
import test_frame_parity_gpu as F  # noqa: E402
import test_ref_parity_gpu as T  # noqa: E402


def main(out_dir):
    dev = torch.device("cuda:0")
    ref = {n: build_ref.load(n) for n in ("_lotd", "_pack_ops", "_occ_grid", "_shencoder")}
    missing = [n for n, m in ref.items() if m is None]
    if missing:
        raise SystemExit(f"oracle/_ref is not built: {missing}")
    rec = {}
    rec.update(T.record(T.lotd_calls(ref["_lotd"], dev)[0], T.LOTD_RULES))
    march = T.march_calls(ref["_occ_grid"], dev)
    rec.update(T.record(march, {k: ("exact",) for k in march}))
    pack = T.pack_calls(ref["_pack_ops"], dev)[0]
    rec.update(T.record(pack, T.pack_rules(pack)))
    rec.update(T.record(T.sh_calls(ref["_shencoder"], dev), T.SH_RULES))
    frames = {}
    with tempfile.TemporaryDirectory() as tmp:
        for case in F.CASES:
            frames.update(F.reference_render(case, os.path.join(tmp, f"{case}.pt")))
    os.makedirs(out_dir, exist_ok=True)
    for name, data in (("ref_kernels.npz", rec), ("ref_frames.npz", frames)):
        path = os.path.join(out_dir, name)
        np.savez_compressed(path, **data)
        print(f"wrote {path}: {len(data)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
