"""Parity AT THE BENCHMARK'S OWN SIZE (BASELINE.json: "PSNR vs ref"; north_star: rgb / depth / normals within 1e-4 relative L2 on identical rays
and weights): the 800x600 frame of bench.py rendered by our kernels (host-sized fused path AND the static / graph path) against the render of the
REFERENCE'S OWN KERNELS (`_lotd`, `_pack_ops`, `_occ_grid`, `_shencoder` compiled by oracle/build_ref.py, driven op by op).  Also: 4096 random
rays (MODE-1 traversal, the training batch).  The reference renders are stored in tests/golden/ref_frames.npz by tests/golden/make_ref_kernels.py
(`reference_render` below, run where the reference kernels are built) as a fixed sample of pixels: most on the object, some of the background."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_frames.npz")
pytestmark = pytest.mark.gpu
KEYS = ("rgb_volume", "depth_volume", "normals_volume", "mask_volume")
CASES = {"view0_eval": (0, False, False, False), "view3_train": (3, True, False, False), "rays4096_view5_train": (5, True, True, True)}
N_OBJECT, N_BACKGROUND = 768, 64

CHILD = r'''
import sys, torch
sys.path.insert(0, %(root)r)
import bench
assert bench.use_reference_cuda_kernels(), "oracle/_ref is not built"
from neuralsim_b200.renderer import SingleVolumeRenderer
dev = torch.device("cuda:0")
model = bench.build_model(dev, collect_samples=%(collect)r)
model.train(%(train)r)
o, d = bench.pinhole_rays(bench.H, bench.W, bench.orbit(%(view)d, 8))
if %(random)r:
    sel = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(11))[:4096]
    o, d = o[sel].contiguous(), d[sel].contiguous()
r = SingleVolumeRenderer(dict(near=0.01)).train(%(train)r)
with torch.no_grad():
    out = r.render(model, o.to(dev), d.to(dev), rays_h_appear=torch.zeros(o.shape[0], 4, device=dev))["rendered"]
torch.save({k: v.cpu() for k, v in out.items()}, %(path)r)
'''


def reference_render(case, path):
    """the render of `case` by the reference's kernels (a child process: it patches module-level back ends), sampled as stored"""
    view, train, random, collect = CASES[case]
    subprocess.run([sys.executable, "-c", CHILD % dict(root=ROOT, view=view, train=train, random=random, collect=collect, path=path)],
                   check=True, timeout=600)
    ref = torch.load(path)
    rng = np.random.default_rng(7)
    hit = (ref["mask_volume"] > 0).numpy()
    on, off = np.flatnonzero(hit), np.flatnonzero(~hit)
    idx = np.sort(np.concatenate([rng.choice(on, min(N_OBJECT, on.size), replace=False), rng.choice(off, min(N_BACKGROUND, off.size), replace=False)]))
    rec = {f"{case}.idx": idx.astype(np.int64), f"{case}.n_rays": np.asarray(hit.size), f"{case}.n_hit": np.asarray(on.size)}
    rec.update({f"{case}.{k}": ref[k][torch.from_numpy(idx)].numpy() for k in KEYS})
    return rec


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(GOLDEN))


def _report(tag, got, golden, case):
    idx = torch.from_numpy(golden[f"{case}.idx"])
    assert got["mask_volume"].shape[0] == int(golden[f"{case}.n_rays"])
    assert int((got["mask_volume"] > 0).sum()) == pytest.approx(int(golden[f"{case}.n_hit"]), rel=1e-3)
    res = {}
    for k in KEYS:
        x, y = got[k].detach().cpu()[idx].double(), torch.from_numpy(golden[f"{case}.{k}"]).double()
        mse = float((x - y).square().mean())
        res[k] = dict(rel_l2=float((x - y).norm() / y.norm().clamp_min(1e-30)), psnr_db=(None if mse == 0 else -10.0 * float(torch.log10(torch.tensor(mse)))))
    print(tag, json.dumps(res))
    return res


@pytest.mark.parametrize("view,train", [(0, False), (3, True)])
def test_800x600_frame_vs_the_reference_kernels(cuda, golden, view, train):
    import bench
    from neuralsim_b200.renderer import SingleVolumeRenderer
    from neuralsim_b200.graphics.neus_static import StaticFrame
    model = bench.build_model(cuda).train(train)
    o, d = bench.pinhole_rays(bench.H, bench.W, bench.orbit(view, 8))
    o, d, ha = o.to(cuda), d.to(cuda), torch.zeros(bench.H * bench.W, 4, device=cuda)
    with torch.no_grad():
        got = SingleVolumeRenderer(dict(near=0.01)).train(train).render(model, o, d, rays_h_appear=ha)["rendered"]
        res = _report(f"frame view {view} {'train' if train else 'eval'} (host-sized fused path)", got, golden, f"view{view}_{'train' if train else 'eval'}")
        for k in ("rgb_volume", "depth_volume", "normals_volume"):
            assert res[k]["rel_l2"] <= 1e-4, (k, res[k])
        assert res["rgb_volume"]["psnr_db"] is None or res["rgb_volume"]["psnr_db"] >= 80.0
        frame = StaticFrame(model, o.shape[0], near=0.01)          # the graph step renders the same images bit for bit
        frame.step(o, d, ha)
        assert frame.counts()["overflow"] == 0
        for k in KEYS:
            assert torch.equal(frame.rendered[k], got[k]), k


def test_4096_random_rays_vs_the_reference_kernels(cuda, golden):
    import bench
    from neuralsim_b200.renderer import SingleVolumeRenderer
    model = bench.build_model(cuda, collect_samples=True).train()
    o, d = bench.pinhole_rays(bench.H, bench.W, bench.orbit(5, 8))
    sel = torch.randperm(o.shape[0], generator=torch.Generator().manual_seed(11))[:4096]
    o, d = o[sel].contiguous().to(cuda), d[sel].contiguous().to(cuda)
    with torch.no_grad():
        got = SingleVolumeRenderer(dict(near=0.01)).train().render(model, o, d, rays_h_appear=torch.zeros(4096, 4, device=cuda))["rendered"]
    res = _report("4096 random rays, training mode, sample collection on", got, golden, "rays4096_view5_train")
    for k in ("rgb_volume", "depth_volume", "normals_volume"):
        assert res[k]["rel_l2"] <= 1e-4, (k, res[k])
    assert float(model.accel.occ._occ_val_grid_pcl.sum()) > 0          # the in-kernel collection ran
