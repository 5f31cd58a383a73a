"""Full-size parity: the BASELINE.json configs at their real shapes (range +-102.4 m -> 512x512 pillars / 2048x2048x40 voxels,
256x256 fusion map, 64-line clouds, 704x256 images), CUDA path vs the UNMODIFIED reference modules on CPU (C1, C2: their
heads stored under tests/golden by oracle/make_golden.py) or the oracle port (C3 SECOND: no spconv-free reference; C4: the
reference's LiftSplatShoot constructor hard-codes CUDA).  Tolerances are north_star's: 1e-3 (fp32-equivalent tc32) and
1e-2 (bf16), relative to max(1, max|ref|)."""
import copy
import os

import numpy as np
import pytest
import torch

from workloads import configs as wcfg, synth, procedural

pytestmark = pytest.mark.gpu
HEADS = ("cls_preds", "reg_preds", "dir_preds")


@pytest.fixture(autouse=True)
def _restore_precision():
    from heal_b200 import engine
    old = engine.PRECISION
    yield
    engine.set_precision(old)


def _check(out, ref, tol, tag):
    for k in HEADS:
        g, r = out[k].float().cpu(), ref[k].float().cpu()
        assert g.shape == r.shape, (tag, k, g.shape, r.shape)
        err = (g - r).abs().max().item()
        scale = max(r.abs().max().item(), 1.0)
        print(f"{tag}/{k}: max|ref|={scale:.3f} max_abs_err={err:.3e} (tol {tol * scale:.3e})")
        assert err <= tol * scale, (tag, k, err, scale)


def _scene(n_agents, rings=64, azimuth=1024, seed=321):
    sc = synth.scene(seed, n_agents=n_agents, max_cav=max(5, n_agents), rings=rings, azimuth=azimuth)
    pts = np.concatenate(sc["points"]).astype(np.float32)
    offs = np.concatenate([[0], np.cumsum([p.shape[0] for p in sc["points"]])]).astype(np.int32)
    return sc, torch.from_numpy(pts).cuda(), torch.from_numpy(offs).cuda()


def _check_golden(out, heads, tol, tag):
    """`_check` against a golden file of the reference's heads (oracle/make_golden.py::make_full_size_golden): the tolerance scale
    is max|ref| over the whole head, the error is taken at the stored sample of its elements."""
    from oracle.make_golden import full_size_sample_index
    for k in HEADS:
        h = heads[k]
        g = out[k].float().cpu()
        assert tuple(g.shape) == tuple(h["shape"]), (tag, k, g.shape, h["shape"])
        err = (g.reshape(-1)[torch.from_numpy(full_size_sample_index(g.numel()))] - h["value"]).abs().max().item()
        scale = max(h["max_abs"], 1.0)
        print(f"{tag}/{k}: max|ref|={scale:.3f} max_abs_err={err:.3e} over {h['value'].numel()} samples (tol {tol * scale:.3e})")
        assert err <= tol * scale, (tag, k, err, scale)


@pytest.fixture(scope="module")
def c2_reference(golden_dir):
    """One full-size 5-agent frame through the unmodified reference HeterPyramidCollab on CPU, stored in full_size_c2.pt."""
    g = torch.load(os.path.join(golden_dir, "full_size_c2.pt"), weights_only=False)
    sc, pts, offs = _scene(5)
    return sc, pts, offs, procedural.make_state_dict(g["shapes"]), g["heads"]


BF16_TOL = 2.5e-2      # see tests/test_gpu_models.py: bf16 storage noise through ~60 stored tensors; tc32 is the 1e-3 path


@pytest.mark.parametrize("prec,tol", [("tc32", 1e-3), ("bf16", BF16_TOL)])
def test_c2_full_size_vs_unmodified_reference(c2_reference, prec, tol):
    from heal_b200 import engine
    from heal_b200.models.heter_pyramid_collab import HeterPyramidCollab
    sc, pts, offs, sd, heads = c2_reference
    engine.set_precision(prec)
    m = HeterPyramidCollab(wcfg.c2_args()).eval()
    m.load_state_dict(sd, strict=True)
    m = m.cuda()
    data = {"inputs_m1": {"points": pts, "agent_offsets": offs}, "agent_modality_list": ["m1"] * 5, "record_len": torch.tensor([5]),
            "pairwise_t_matrix": torch.from_numpy(sc["pairwise_t_matrix"]).cuda()}
    with torch.no_grad():
        out = m(data)
    _check_golden(out, heads, tol, f"C2-full/{prec}")


def test_c1_full_size_vs_unmodified_reference(golden_dir):
    """configs[0]: models/point_pillar.py, one 20k-ray cloud, range +-102.4 m (512x512 pillars); the reference's heads are
    stored in full_size_c1.pt."""
    from heal_b200 import engine
    from heal_b200.models.point_pillar import PointPillar
    engine.set_precision("tc32")
    g = torch.load(os.path.join(golden_dir, "full_size_c1.pt"), weights_only=False)
    cloud = synth.lidar_cloud(np.random.default_rng(77), rings=20, azimuth=1000)
    sd = procedural.make_state_dict(g["shapes"])
    m = PointPillar(wcfg.c1_args()).eval()
    m.load_state_dict(sd, strict=True)
    m = m.cuda()
    offs = torch.tensor([0, cloud.shape[0]], dtype=torch.int32).cuda()
    with torch.no_grad():
        out = m({"processed_lidar": {"points": torch.from_numpy(cloud).cuda(), "agent_offsets": offs}})
    _check_golden(out, g["heads"], 1e-3, "C1-full/tc32")


def test_c1_gpu_point_filters_equal_host_filters():
    """The on-GPU input path (filter_on_gpu): an UNFILTERED cloud + the host-drawn shuffle permutation through heal_mask_points ->
    voxeliser -> model gives bit-identical predictions to the reference's host filters (oracle/pcd.py) feeding the same model."""
    from oracle import pcd
    from heal_b200 import engine
    from heal_b200.models.point_pillar import PointPillar
    engine.set_precision("tc32")
    rng = np.random.default_rng(78)
    cloud = synth.lidar_cloud(rng, rings=32, azimuth=1000)
    cloud = np.concatenate([cloud, rng.uniform(-3, 3, size=(500, 4)).astype(np.float32),          # ego-box hits
                            rng.uniform(-130, 130, size=(500, 4)).astype(np.float32)])             # out-of-range points
    perm = rng.permutation(cloud.shape[0]).astype(np.int32)
    host = pcd.filter_cloud(cloud, wcfg.RANGE, perm)
    assert 0 < host.shape[0] < cloud.shape[0]
    m = PointPillar(wcfg.c1_args()).eval()
    m.load_state_dict(procedural.make_state_dict(procedural.shapes_of(m)), strict=True)
    m = m.cuda()
    with torch.no_grad():
        a = m({"processed_lidar": {"points": torch.from_numpy(host).cuda(), "agent_offsets": torch.tensor([0, host.shape[0]], dtype=torch.int32).cuda()}})
        b = m({"processed_lidar": {"points": torch.from_numpy(cloud).cuda(), "agent_offsets": torch.tensor([0, cloud.shape[0]], dtype=torch.int32).cuda(),
                                   "filter_points": True, "remove_ego": True, "shuffle_perm": torch.from_numpy(perm).cuda()}})
    for k in ("cls_preds", "reg_preds", "dir_preds"):
        assert torch.equal(a[k], b[k]), k


def test_c3_full_size_second_attfusion_vs_oracle():
    """configs[2]: SECOND (0.1 m voxels, 2048x2048x40 grid, ~300k voxels) + BaseBEVBackbone + per-agent shrinker + AttFusion, 5 agents."""
    from oracle import nets, sparse_conv as sc_, voxelizer
    from heal_b200 import engine
    from heal_b200.models.heter_model_baseline import HeterModelBaseline
    engine.set_precision("tc32")
    args = wcfg.c3_args()
    m = HeterModelBaseline(copy.deepcopy(args)).eval()
    sd = procedural.make_state_dict(procedural.shapes_of(m))
    m.load_state_dict(sd, strict=True)
    m = m.cuda()
    sc, pts, offs = _scene(5, seed=322)
    per_agent = [voxelizer.points_to_voxel_c(p, wcfg.SECOND_VOXEL, wcfg.RANGE, 5, 70000) for p in sc["points"]]
    col = {k: torch.from_numpy(v) for k, v in voxelizer.collate(per_agent).items()}
    pw = torch.from_numpy(sc["pairwise_t_matrix"])
    enc_args = args["m1"]["encoder_args"]
    dd = {"inputs_m1": col, "agent_modality_list": ["m1"] * 5, "record_len": torch.tensor([5]), "pairwise_t_matrix": pw}
    with torch.no_grad():
        ref = nets.heter_model_baseline(sd, args, dd, encoder_fns={
            "m1": lambda d, mm: sc_.second_encoder(sd, "encoder_m1", enc_args, d["inputs_m1"])})
        out = m({"inputs_m1": {"points": pts, "agent_offsets": offs}, "agent_modality_list": ["m1"] * 5,
                 "record_len": torch.tensor([5]), "pairwise_t_matrix": pw.cuda()})
    _check(out, ref, 1e-3, "C3-full/tc32")


def test_c4_full_size_lss_hetero_bf16_vs_oracle():
    """configs[3]: agents [PointPillars, LSS 4x704x256, LSS], camera grid +-51.2 m zero-padded into the +-102.4 m map, bf16."""
    from oracle import hetero, voxelizer
    from heal_b200 import engine
    from heal_b200.models.heter_pyramid_collab import HeterPyramidCollab
    engine.set_precision("bf16")
    args = wcfg.c4_args()
    m = HeterPyramidCollab(copy.deepcopy(args)).eval()
    sd = procedural.make_state_dict(procedural.shapes_of(m))
    m.load_state_dict(sd, strict=True)
    m = m.cuda()
    sc, _, _ = _scene(3, seed=323)
    cloud = sc["points"][0]
    col = {k: torch.from_numpy(v) for k, v in voxelizer.collate([voxelizer.points_to_voxel_c(cloud, wcfg.PILLAR_VOXEL, wcfg.RANGE, 32, 70000)]).items()}
    rots, trans, intr, post_rots, post_trans = [torch.from_numpy(a) for a in synth.camera_rig(2, 4, 256, 704)]
    imgs = torch.randn(2, 4, 3, 256, 704, generator=torch.Generator().manual_seed(9))
    cam = {"imgs": imgs, "rots": rots, "trans": trans, "intrins": intr, "post_rots": post_rots, "post_trans": post_trans}
    pw = torch.from_numpy(sc["pairwise_t_matrix"])
    aml = ["m1", "m2", "m2"]
    ref = hetero.heter_pyramid_collab_hetero(sd, args, col, cam, pw, aml)
    offs = torch.tensor([0, cloud.shape[0]], dtype=torch.int32).cuda()
    with torch.no_grad():
        out = m({"inputs_m1": {"points": torch.from_numpy(cloud).cuda(), "agent_offsets": offs},
                 "inputs_m2": {k: v.cuda() for k, v in cam.items()}, "agent_modality_list": aml,
                 "record_len": torch.tensor([3]), "pairwise_t_matrix": pw.cuda()})
    _check(out, ref, BF16_TOL, "C4-full/bf16")
