"""API-surface checks on the GPU: the calls the reference's own code makes against `nksr`
(SURVEY.md Appendix A) resolve and behave -- adaptive hierarchy, voxel status, the training-model
wiring of models/nksr_net.py:57-133 and the headless example."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import clouds

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_adaptive_hierarchy_prunes_flat_regions(cuda):
    """build_adaptive_normal_variation (models/nksr_net.py:175-179): a flat plane has consistent normals,
    so its level-1 voxels become leaves and level 0 disappears there; a sphere of small radius keeps it."""
    import nksr
    rng = np.random.default_rng(0)
    plane = np.stack([rng.uniform(-1, 1, 20000), rng.uniform(-1, 1, 20000), np.zeros(20000)], 1).astype(np.float32)
    pn = np.tile(np.array([[0, 0, 1.0]], np.float32), (20000, 1))
    ball, bn = clouds.sphere(20000, radius=0.12, centre=(3.0, 0.0, 0.0))
    xyz, nrm = np.concatenate([plane, ball]), np.concatenate([pn, bn])
    t = lambda a: torch.from_numpy(a).to(cuda)
    full = nksr.SparseFeatureHierarchy(0.05, 4, cuda).build_point_splatting(t(xyz))
    ada = nksr.SparseFeatureHierarchy(0.05, 4, cuda)
    ada.build_adaptive_normal_variation(t(xyz), t(nrm), tau=0.02, adaptive_depth=2)   # ball voxels vary by ~0.07
    assert ada.num_voxels(0) < 0.5 * full.num_voxels(0)
    for l in (1, 2, 3):
        assert torch.equal(ada.keys[l], full.keys[l])
    c0 = ada.get_voxel_centers(0).cpu().numpy()
    assert (c0[:, 0] > 2.0).mean() > 0.9                  # what is left of level 0 sits on the ball
    # voxel status of the full hierarchy against the adaptive one (models/loss.py:155): 0 absent, 1 leaf, 2 inner
    st0 = ada.evaluate_voxel_status(full.grids[0], 0)
    st1 = ada.evaluate_voxel_status(full.grids[1], 1)
    assert set(st0.unique().tolist()) <= {0, 1} and (st0 == 0).any() and (st0 == 1).any()
    assert set(st1.unique().tolist()) <= {1, 2} and (st1 == 1).any() and (st1 == 2).any()


def test_training_model_wiring(cuda):
    """The piecewise construction of models/nksr_net.py:57-133 against the alias package."""
    import nksr
    from nksr.svh import SparseFeatureHierarchy
    from nksr.fields import KernelField, LayerField
    xyz, nrm = clouds.sphere(20000, noise=0.001)
    t = lambda a: torch.from_numpy(a).to(cuda)
    hp = dict(voxel_size=0.03, tree_depth=4, adaptive_depth=2, kernel_dim=4)
    network = nksr.NKSRNetwork(hp).to(cuda)
    enc_svh = SparseFeatureHierarchy(voxel_size=hp["voxel_size"], depth=hp["tree_depth"], device=cuda)
    enc_svh.build_point_splatting(t(xyz))
    feat = network.encoder(t(xyz), t(nrm), enc_svh, 0)
    feat, dec_svh, udf_svh = network.unet(feat, enc_svh, adaptive_depth=hp["adaptive_depth"], gt_decoder_svh=None)
    assert not all(dec_svh.grids[d] is None for d in range(hp["adaptive_depth"]))
    field = KernelField(svh=dec_svh, interpolator=network.interpolators, features=feat.basis_features,
                        approx_kernel_grad=False)
    field.solver_config["verbose"] = False
    normal_xyz = torch.cat([dec_svh.get_voxel_centers(d) for d in range(hp["adaptive_depth"])])
    normal_value = torch.cat([feat.normal_features[d] for d in range(hp["adaptive_depth"])])
    normal_weight = 1e4 / normal_xyz.size(0) * (hp["voxel_size"] ** 2)
    field.solve_non_fused(pos_xyz=t(xyz), normal_xyz=normal_xyz, normal_value=-normal_value,
                          pos_weight=1e4 / xyz.shape[0], normal_weight=normal_weight, reg_weight=1.0)
    field.set_mask_field(LayerField(dec_svh, hp["adaptive_depth"]))
    mesh = field.extract_dual_mesh(grid_upsample=2)                         # models/nksr_net.py:284
    r = np.linalg.norm(mesh.v.cpu().numpy(), axis=1)
    assert mesh.f.shape[0] > 1000 and abs(np.median(r) - 0.35) < 0.005
    res = field.evaluate_f(t(xyz[:500]), grad=True)                          # models/loss.py:189-198
    pd = -res.gradient / (torch.linalg.norm(res.gradient, dim=-1, keepdim=True) + 1e-6)
    assert float(1.0 - torch.sum(pd * t(nrm[:500]), dim=-1).mean()) < 0.05
    grid = dec_svh.grids[0]
    ijk = grid.active_grid_coords()                                          # models/loss.py:36-46
    assert torch.allclose(grid.grid_to_world(ijk.float()), dec_svh.get_voxel_centers(0))


def test_headless_example_runs(tmp_path):
    obj = str(tmp_path / "recons_simple.obj")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "recons_simple.py"), "-", obj],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    assert os.path.getsize(obj) > 10000


def test_fields_follow_their_tensors_device():
    """ADVICE r1 (medium): every C-ABI call must run on the device that owns its tensors, not on the current one.
    Needs two GPUs (skipped on a one-GPU box): reconstruct + mesh on cuda:1 while cuda:0 is current."""
    import nksr_b200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from tests import clouds
    torch.cuda.set_device(0)
    dev = torch.device("cuda:1")
    xyz, nrm = clouds.sphere(6000, noise=0.001)
    rec = nksr_b200.Reconstructor(dev)
    field = rec.reconstruct(torch.from_numpy(xyz).to(dev), torch.from_numpy(nrm).to(dev), voxel_size=0.05)
    assert field.alpha.device == dev and torch.cuda.current_device() == 0
    mesh = field.extract_dual_mesh(mise_iter=1)
    r = mesh.v.norm(dim=1)
    assert mesh.v.device == dev and mesh.f.shape[0] > 500 and abs(float(r.median()) - 0.35) < 0.01
