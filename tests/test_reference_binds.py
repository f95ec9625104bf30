"""The drop-in boundary from the reference's side: what an UNMODIFIED nr3d_lib Python tree imports from and calls on
`nr3d_lib.bindings` resolves over `install_as_nr3d_lib_bindings()` (SURVEY.md §8b: "all of these names must resolve").  What the reference's
files import and call, and what its `LoTD` module built over the shim, are recorded in tests/golden/ref_binds.json by
tests/golden/make_ref_binds.py from the reference tree."""
import importlib
import json
import os
import sys
import types

import pytest

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_binds.json")))


@pytest.fixture(scope="module")
def ref_tree():
    saved = {k: v for k, v in sys.modules.items() if k == "nr3d_lib" or k.startswith("nr3d_lib.")}
    for k in saved:
        del sys.modules[k]
    import neuralsim_b200.bindings as B
    root = types.ModuleType("nr3d_lib")
    root.__path__ = []
    sys.modules["nr3d_lib"] = root
    B.install_as_nr3d_lib_bindings()
    yield B
    for k in [k for k in sys.modules if k == "nr3d_lib" or k.startswith("nr3d_lib.")]:
        del sys.modules[k]
    sys.modules.update(saved)


def test_reference_modules_import_over_the_shim(ref_tree):
    B = ref_tree
    built = {"nr3d_lib.bindings._pack_ops": B._pack_ops, "nr3d_lib.bindings._occ_grid": B._occ_grid, "nr3d_lib.bindings._lotd": B._lotd,
             "nr3d_lib.bindings._shencoder": B._shencoder}
    modules = {imp["module"] for imp in GOLDEN["imports"]}
    assert set(built) <= modules and "nr3d_lib.bindings._forest" in modules
    for imp in GOLDEN["imports"]:
        mod = importlib.import_module(imp["module"])                      # `import nr3d_lib.bindings._x as _backend`
        if imp["module"] in built:
            assert mod is built[imp["module"]], imp
        for name in imp["names"] or ():                                   # `from nr3d_lib.bindings._x import a, b` at import time
            assert callable(getattr(mod, name)), imp


def test_every_backend_name_the_reference_calls_exists(ref_tree):
    B = ref_tree
    assert set(GOLDEN["backend_calls"]) == {"_pack_ops", "_occ_grid", "_lotd", "_shencoder"}
    for mod, names in GOLDEN["backend_calls"].items():
        shim = getattr(B, mod)
        assert names and not [n for n in names if not hasattr(shim, n)], mod


def test_placeholders_resolve_and_raise_on_use(ref_tree):
    from nr3d_lib.bindings._forest import ForestMeta, raytrace_cuda_fixed            # the two import-time names (forest.py:26, raytest.py:198)
    import nr3d_lib.bindings._permuto as permuto
    with pytest.raises(RuntimeError, match="_forest.ForestMeta"):
        ForestMeta()
    with pytest.raises(RuntimeError, match="raytrace_cuda_fixed"):
        raytrace_cuda_fixed(None, None)
    with pytest.raises(RuntimeError, match="permutohedral"):
        permuto.permuto_enc_fwd(1, 2, 3)
    with pytest.raises(RuntimeError, match="not built"):
        ref_tree._pack_ops.octree_mark_consecutive_segments(None)


def test_reference_lotd_module_builds_its_meta_through_the_shim(ref_tree):
    """the LoDMeta call the reference's own `LoTD` nn.Module makes (host-side: no GPU needed), replayed on the shim: sizes as the oracle's
    and as the reference module derived them"""
    from oracle import lotd as olotd
    rec = GOLDEN["lotd_module"]
    c = rec["cfg"]
    assert rec["meta_args"] == [3, c["res"], c["feats"], c["types"], c["hashmap_size"], False]
    m = importlib.import_module("nr3d_lib.bindings._lotd").LoDMeta(*rec["meta_args"])
    om = olotd.LoDMeta(3, c["res"], c["feats"], c["types"], hashmap_size=c["hashmap_size"])
    n_lvl = len(c["res"])
    assert m.n_params == om.n_params == rec["n_params"] and m.level_n_feats == c["feats"] == rec["level_n_feats"]
    assert m.level_offsets[:n_lvl + 1] == list(om.level_offsets)[:n_lvl + 1] == rec["level_offsets"][:n_lvl + 1]
    assert sum(m.level_n_feats) == m.n_encoded_dims == rec["out_features"] == 10 and m.n_dims_to_encode == rec["in_features"] == 3
