"""Generates tests/golden/ref_binds.json from the reference's own Python tree: every `nr3d_lib.bindings` import and every
`_backend.<name>` call of the files that bind to the CUDA extensions, and what the reference's `LoTD` module built on top of
`install_as_nr3d_lib_bindings()`.  tests/test_reference_binds.py checks the shim against this record, so it runs without the tree.

    python tests/golden/make_ref_binds.py /path/to/nr3d_lib/nr3d_lib

The reference's package __init__ files pull uninstallable dependencies (addict, kornia, imageio ...), so -- as make_golden.py --
the parent packages are registered empty with the right __path__ and the reference FILES are executed verbatim.
"""
import importlib
import json
import os
import re
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

# the files whose import of nr3d_lib.bindings is exercised, and the files each backend's calls are collected from
IMPORTING = ["graphics/pack_ops/pack_ops.py", "graphics/raymarch/occgrid_raymarch.py", "models/grid_encodings/lotd/lotd.py",
             "models/embedders/spherical_harmonics/sphere_harmonics.py", "graphics/raytest.py", "models/spatial/forest.py",
             "models/embedders/sinusoidal_cuda/freq.py", "models/grid_encodings/permuto/permuto.py"]
CALLING = {"_pack_ops": ["graphics/pack_ops/pack_ops.py"], "_occ_grid": ["graphics/raymarch/occgrid_raymarch.py"],
           "_lotd": ["models/grid_encodings/lotd/lotd.py", "models/grid_encodings/lotd/lotd_encoding.py",
                     "models/grid_encodings/lotd/lotd_batched.py", "models/grid_encodings/lotd/lotd_forest.py"],
           "_shencoder": ["models/embedders/spherical_harmonics/sphere_harmonics.py"]}
LOTD_CFG = dict(res=[8, 12, 18, 40, 64], feats=[2] * 5, types=["Dense", "Dense", "Dense", "Hash", "Hash"], hashmap_size=2 ** 12)


def _pkg(name, path):
    m = types.ModuleType(name)
    m.__path__ = [path]
    sys.modules[name] = m
    return m


def scan_imports(ref):
    out = []
    for f in IMPORTING:
        for line in open(os.path.join(ref, f)):
            m = re.match(r"\s*import (nr3d_lib\.bindings\.\w+) as \w+", line)
            if m:
                out.append(dict(file=f, module=m.group(1), names=None))
            m = re.match(r"\s*from (nr3d_lib\.bindings\.\w+) import (.+)", line)
            if m:
                out.append(dict(file=f, module=m.group(1), names=[n.strip() for n in m.group(2).split(",")]))
    return out


def scan_calls(ref):
    calls = {}
    for mod, fs in CALLING.items():
        names = set()
        for f in fs:
            names |= set(re.findall(r"_backend\.(\w+)", open(os.path.join(ref, f)).read()))
        calls[mod] = sorted(names)
    return calls


def lotd_module(ref):
    """the reference's `LoTD` nn.Module constructed over the shim (host side only): the LoDMeta call it makes and the sizes it derives"""
    import neuralsim_b200.bindings as B
    _pkg("nr3d_lib", ref)
    for sub in ("models", "models/grid_encodings", "models/grid_encodings/lotd"):
        _pkg("nr3d_lib." + sub.replace("/", "."), f"{ref}/{sub}")
    B.install_as_nr3d_lib_bindings()
    utils = types.ModuleType("nr3d_lib.utils")
    utils.check_to_torch = lambda x, **kw: torch.as_tensor(x, **{k: v for k, v in kw.items() if k in ("dtype", "device")})
    sys.modules["nr3d_lib.utils"] = utils
    calls = []
    real = B._lotd.LoDMeta

    def recording(*args):
        calls.append(list(args))
        return real(*args)
    B._lotd.LoDMeta = recording
    try:
        lotd = importlib.import_module("nr3d_lib.models.grid_encodings.lotd.lotd")
        c = LOTD_CFG
        m = lotd.LoTD(3, c["res"], c["feats"], c["types"], hashmap_size=c["hashmap_size"], dtype=torch.half, device=torch.device("cpu"))
    finally:
        B._lotd.LoDMeta = real
    assert len(calls) == 1, calls
    return dict(cfg=c, meta_args=calls[0], n_params=int(m.n_params), level_n_feats=[int(v) for v in m.level_n_feats],
                level_offsets=[int(v) for v in list(m.meta.level_offsets)], out_features=int(m.out_features), in_features=int(m.in_features))


def main(ref):
    out = dict(imports=scan_imports(ref), backend_calls=scan_calls(ref), lotd_module=lotd_module(ref))
    path = os.path.join(ROOT, "tests", "golden", "ref_binds.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(f"wrote {path}: {len(out['imports'])} imports, {sum(map(len, out['backend_calls'].values()))} backend names")


if __name__ == "__main__":
    main(sys.argv[1])
