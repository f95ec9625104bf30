"""GPU: our kernels AND the CPU oracle against the REFERENCE'S OWN CUDA kernels.  What the reference kernels computed on these inputs is
stored in tests/golden/ref_kernels.npz by tests/golden/make_ref_kernels.py, which runs the same calls against the reference's extensions
(compiled by oracle/build_ref.py): a SHA-256 digest of every output compared bit for bit, a fixed seeded sample of every output compared
within a tolerance.  Every input is made on the host from a seed, so both runs see the same bits.
This is what pins the oracle for the parts the reference ships no fixtures for: LoTD, marching, alpha compositing."""
import hashlib
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.npz")
f32 = np.float32


# ---------------------------------------------------------------------------------------------- digests and samples
def _np(t):
    t = t.detach().contiguous().cpu() if isinstance(t, torch.Tensor) else torch.as_tensor(t)
    return t.view(torch.int16).numpy() if t.dtype == torch.float16 else t.numpy()


def digest(t):
    a = np.ascontiguousarray(_np(t))
    return hashlib.sha256(str(a.dtype).encode() + a.tobytes()).hexdigest()


def sample_rows(key, n_rows, k, hi=None):
    """a fixed sample of `k` row indices of output `key` (rows below `hi`), the same in the generator and the test"""
    hi = n_rows if hi is None else min(hi, n_rows)
    seed = int.from_bytes(hashlib.sha256(key.encode()).digest()[:4], "little")
    return np.sort(np.random.default_rng(seed).choice(hi, min(k, hi), replace=False))


def record(out, rules):
    """the reference side: outputs -> what the golden file keeps (see `rules`)"""
    rec = {}
    for key, t in out.items():
        rule = rules[key]
        rec[f"{key}.shape"] = np.asarray(tuple(t.shape), dtype=np.int64)
        if rule[0] == "exact":
            rec[f"{key}.sha"] = np.asarray(digest(t))
        elif rule[0] == "value":
            rec[f"{key}.val"] = _np(t)
        else:
            x = t.detach().contiguous().cpu()
            rec[f"{key}.val"] = x[torch.from_numpy(sample_rows(key, x.shape[0], rule[1], rule[2] if len(rule) > 2 else None))].float().numpy()
    return rec


def ref_sample(g, key, rule):
    shape = tuple(g[f"{key}.shape"])
    idx = sample_rows(key, shape[0], rule[1], rule[2] if len(rule) > 2 else None)
    return torch.from_numpy(idx), torch.from_numpy(g[f"{key}.val"])


def check(g, out, rules):
    """ours against the stored reference side"""
    for key, t in out.items():
        rule = rules[key]
        assert tuple(t.shape) == tuple(g[f"{key}.shape"]), key
        if rule[0] == "exact":
            assert digest(t) == str(g[f"{key}.sha"]), key
        elif rule[0] == "value":
            assert np.array_equal(_np(t), g[f"{key}.val"]), key
        else:
            idx, ref = ref_sample(g, key, rule)
            got = t.detach().contiguous().cpu()[idx].float()
            if rule[0] == "close":
                assert torch.allclose(got, ref, rtol=rule[3], atol=rule[4]), key
            else:                                                    # "relnorm": |ref - ours| / |ours| over the sample
                err = float((ref - got).norm() / got.norm())
                assert err < rule[3], (key, err)


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(GOLDEN))


# ---------------------------------------------------------------------------------------------- LoTD
LOTD_N = 60000
LOTD_RULES = {"n_params": ("value",), "level_offsets": ("value",), "level_sizes": ("value",), "y": ("exact",), "y_first5000": ("exact",),
              "dydx": ("close", 64, 5000, 1e-6, 1e-7), "y_ml7": ("exact",), "y_ml0": ("exact",), "gx": ("close", 1024, None, 1e-4, 1e-4),
              # the reference accumulates grid gradients with fp16 atomics (order dependent, saturating); ours in fp32 -> tolerance
              "gp": ("relnorm", 8192, None, 2e-2), "bb_a": ("relnorm", 256, None, 5e-3), "bb_b": ("relnorm", 8192, None, 5e-2)}


def lotd_calls(B, dev):
    from oracle import lotd as olotd
    cfg = olotd.gen_ngp_cfg()
    m = B.LoDMeta(3, cfg["lod_res"], cfg["lod_n_feats"], cfg["lod_types"], cfg["hashmap_size"], False)
    rng = np.random.default_rng(0)
    p = torch.from_numpy(rng.uniform(-0.1, 0.1, m.n_params).astype(np.float16)).to(dev)
    x = torch.from_numpy(rng.uniform(1e-6, 1 - 1e-6, (LOTD_N, 3)).astype(f32)).to(dev)
    g = torch.from_numpy((rng.normal(size=(LOTD_N, 32)) * 0.05).astype(np.float16)).to(dev)
    gin = torch.from_numpy(rng.normal(size=(LOTD_N, 3)).astype(f32)).to(dev)
    y, d = B.lod_fwd(m, x, p, None, None, None, None, True)
    y, d = y.contiguous(), d.contiguous().reshape(LOTD_N, -1)
    out = dict(n_params=torch.tensor(m.n_params), level_offsets=torch.tensor(list(m.level_offsets)), level_sizes=torch.tensor(list(m.level_sizes)),
               y=y, y_first5000=y[:5000], dydx=d)
    for ml in (7, 0):
        out[f"y_ml{ml}"] = B.lod_fwd(m, x, p, None, None, None, ml, False)[0].contiguous()
    out["gx"], out["gp"] = B.lod_bwd(m, g, x, p, d, None, None, None, None, True, True)
    out["bb_a"], out["bb_b"], _ = B.lod_bwd_bwd_input(m, gin, g, x, p, d, None, None, None, None, True, True, False)
    return out, (x, p)


def test_lotd_against_reference_kernels(cuda, golden):
    from oracle import lotd as olotd
    from neuralsim_b200.bindings import _lotd as ours
    out, (x, p) = lotd_calls(ours, cuda)
    check(golden, out, LOTD_RULES)
    cm = olotd.LoDMeta(3, **olotd.gen_ngp_cfg())                                                   # the CPU oracle, same check
    assert cm.n_params == int(golden["n_params.val"]) and list(cm.level_offsets) == list(golden["level_offsets.val"])
    y_c, d_c = olotd.lod_fwd(cm, x[:5000].cpu().numpy(), p.cpu().numpy(), need_input_grad=True)
    assert digest(torch.from_numpy(y_c)) == str(golden["y_first5000.sha"])                          # features: bit-exact
    idx, d_r = ref_sample(golden, "dydx", LOTD_RULES["dydx"])
    assert np.allclose(d_c.reshape(5000, -1)[idx.numpy()], d_r.numpy(), rtol=1e-6, atol=1e-7)


# ---------------------------------------------------------------------------------------------- marching
MARCH_KEYS = ("packed_info", "t_starts", "t_ends", "ridx", "gidx")


def march_inputs():
    from oracle import render as orender, scene as oscene
    os_, ds_ = [], []
    for k in range(4):
        o, d = oscene.pinhole_rays(60, 80, oscene.orbit_camera(k, 4, radius=2.5 + 0.3 * k, elev_deg=10 + 15 * k))
        os_.append(o); ds_.append(d)
    rt = orender.ray_test(torch.cat(os_), torch.cat(ds_), near=0.01)
    rng = np.random.default_rng(1)
    grids = (oscene.make_occ_grid(64), torch.from_numpy(rng.random((48, 32, 40)) < 0.1))
    return tuple(rt[k].contiguous() for k in ("rays_o", "rays_d", "near", "far")), grids, torch.tensor([-1., -1, -1, 1, 1, 1])


def march_calls(B, dev):
    (o, d, near, far), grids, roi = march_inputs()
    out = {}
    for dt_gamma in (0.0, 0.01):
        for gi, grid in enumerate(grids):
            r = B.ray_marching(o.to(dev), d.to(dev), near.to(dev), far.to(dev), roi.to(dev), grid.to(dev), B.ContractionType.AABB, 0.005, 0.1,
                               dt_gamma, 1024, True)
            for k, t in zip(MARCH_KEYS, r):
                out[f"{dt_gamma}.{gi}.{k}"] = t
    return out


@pytest.mark.parametrize("dt_gamma", [0.0, 0.01])
def test_marching_against_reference_kernels(cuda, golden, dt_gamma):
    from oracle import march as omarch
    from neuralsim_b200.bindings import _occ_grid as ours
    (o, d, near, far), grids, roi = march_inputs()
    for gi, grid in enumerate(grids):
        g = ours.ray_marching(o.to(cuda), d.to(cuda), near.to(cuda), far.to(cuda), roi.to(cuda), grid.to(cuda), ours.ContractionType.AABB, 0.005, 0.1,
                              dt_gamma, 1024, True)
        keys = [f"{dt_gamma}.{gi}.{k}" for k in MARCH_KEYS]
        check(golden, dict(zip(keys, g)), {k: ("exact",) for k in keys})      # counts, t_starts, t_ends, ridx, gidx: bit-exact
        c = omarch.ray_marching(o, d, near, far, roi, grid, 0.005, 0.1, dt_gamma, 1024)            # and the C oracle
        for i in (0, 1, 4):
            assert digest(c[i]) == str(golden[f"{keys[i]}.sha"]), keys[i]
        assert int(g[0][:, 1].sum()) > 1000


# ---------------------------------------------------------------------------------------------- pack_ops
def pack_calls(B, dev):
    from util import random_packs
    rng = np.random.default_rng(2)
    pi = random_packs(rng, 500, 1, 140)
    n = pi[:, 1].numpy()
    S = int(n.sum())
    seg = lambda v, excl=False: np.concatenate([np.cumsum(np.concatenate([[0.], s[:-1]]) if excl else s) for s in np.split(v, np.cumsum(n)[:-1])])
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    f = rng.normal(size=(S, 3)).astype(f32)
    o = (rng.random((500, 3)) + 1).astype(f32)
    a = (rng.random(S) ** 3).astype(f32)
    a[rng.random(S) < 0.3] = 0
    a[rng.random(S) < 0.02] = 0.999
    gw = rng.normal(size=S).astype(f32)
    cdf = seg(a.astype(np.float64), excl=True)
    last = np.repeat(np.maximum(cdf[np.cumsum(n) - 1], 1e-5), n)
    cdf = (cdf / last).astype(f32)
    bins = seg(rng.random(S)).astype(f32)
    u = np.broadcast_to(np.linspace(0, 1, 35)[1:-1].astype(f32), (500, 33))
    pib = random_packs(rng, 500, 1, 40)
    nb = pib[:, 1].numpy()
    vb = np.concatenate([np.cumsum(s) for s in np.split(rng.random(int(nb.sum())), np.cumsum(nb)[:-1])]).astype(f32)
    st, step = rng.normal(size=500).astype(f32), rng.random(500).astype(f32)
    v = rng.normal(size=S).astype(f32)
    pi, pib, f, o, a, gw, cdf, bins, u, vb, st, step, v = (T(x) if isinstance(x, np.ndarray) else x.to(dev)
                                                           for x in (pi, pib, f, o, a, gw, cdf, bins, u, vb, st, step, v))
    out = dict(sum=B.packed_sum(f, pi))
    for ex in (False, True):
        for rev in (False, True):
            out[f"cumsum.{int(ex)}{int(rev)}"] = B.packed_cumsum(f, pi, ex, rev)
    out.update(diff=B.packed_diff(f, pi, None, None), bdiff=B.packed_backward_diff(f, pi, None, None), div=B.packed_div(f, o, pi), add=B.packed_add(f, o, pi))
    w = out["vw"] = B.packed_alpha_to_vw_forward(a, pi, 1e-4, 0.0, False)[0]
    _, info, out["vw.sel"] = B.packed_alpha_to_vw_forward(a, pi, 1e-4, 0.0, True)
    out["vw.info"] = info.long()
    out["vw.grad"] = B.packed_alpha_to_vw_backward(w, gw, a, pi, 1e-4, 0.0)
    out["invert_cdf.s"], out["invert_cdf.i"] = B.packed_invert_cdf(bins, cdf, u, pi)
    out["searchsorted"] = B.packed_searchsorted(cdf, u, pi)
    for b_sorted in (True, False):
        for i, t in enumerate(B.try_merge_two_packs_sorted_aligned(bins, pi, vb, pib, b_sorted)):
            out[f"merge.{int(b_sorted)}.{i}"] = t
    nn = pi[:, 1].contiguous()
    for i, t in enumerate(B.interleave_arange(nn, True)):
        out[f"interleave_arange.{i}"] = t
    for i, t in enumerate(B.interleave_linstep(st, nn, step, True)):
        out[f"interleave_linstep.{i}"] = t
    vs = v.clone()
    idx = B.packed_sort_qsort(vs, pi, True)
    out["qsort.values"], out["qsort.gathered"] = vs, v[idx]                  # quicksort is unstable: compare values
    out["boundaries"] = B.mark_pack_boundaries_cuda(torch.repeat_interleave(torch.arange(500, device=dev), nn))
    return out, (a, pi)


def pack_rules(out):
    rules = {k: ("exact",) for k in out}                                     # the serial recurrences and index algebra: bit-exact
    rules["sum"] = ("close", 500, None, 1e-5, 1e-5)
    rules.update({k: ("close", 256, None, 1e-5, 2e-5) for k in out if k.startswith("cumsum.")})
    rules["vw.grad"] = ("relnorm", 4096, None, 1e-4)
    return rules


def test_pack_ops_against_reference_kernels(cuda, golden):
    from oracle import pack_ops as opk
    from neuralsim_b200.bindings import _pack_ops as ours
    out, (a, pi) = pack_calls(ours, cuda)
    check(golden, out, pack_rules(out))
    assert digest(opk.packed_alpha_to_vw_forward(a.cpu(), pi.cpu(), 1e-4, 0.0, False)[0]) == str(golden["vw.sha"])   # and the CPU oracle


# ---------------------------------------------------------------------------------------------- spherical harmonics
SH_N = 5000
SH_RULES = {f"{k}.{C}": ("close", 64, None) + tol for C in (1, 2, 3, 4)
            for k, tol in (("out", (1e-6, 1e-7)), ("jac", (1e-5, 1e-6)), ("grad", (1e-4, 1e-5)))}


def sh_calls(B, dev):
    rng = np.random.default_rng(3)
    v = torch.nn.functional.normalize(torch.from_numpy(rng.normal(size=(SH_N, 3)).astype(f32)), dim=-1).to(dev)
    out = {}
    for C in (1, 2, 3, 4):
        y, j = torch.empty(SH_N, C * C, device=dev), torch.empty(SH_N, 3 * C * C, device=dev)
        B.sh_encode_forward(v, y, SH_N, 3, C, True, j)
        torch.cuda.synchronize()                                         # the reference launches on the default stream
        g = torch.from_numpy(rng.normal(size=(SH_N, C * C)).astype(f32)).to(dev)
        gi = torch.zeros(SH_N, 3, device=dev)
        B.sh_encode_backward(g, v, SH_N, 3, C, j, gi)
        torch.cuda.synchronize()
        out[f"out.{C}"], out[f"jac.{C}"], out[f"grad.{C}"] = y, j, gi
    return out


def test_shencoder_against_reference_kernel(cuda, golden):
    from neuralsim_b200.bindings import _shencoder as ours
    check(golden, sh_calls(ours, cuda), SH_RULES)
