"""Pins the oracle (oracle/nets.py) against vectors produced by the UNMODIFIED reference modules
(oracle/make_golden.py, run in the build container).  CPU only."""
import os

import numpy as np
import torch

from oracle import nets, procedural


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def test_heter_pyramid_collab_small(golden_dir):
    g = _load(golden_dir, "heter_pyramid_collab_small.pt")
    sd = procedural.make_state_dict(g["shapes"])
    with torch.no_grad():
        out = nets.heter_pyramid_collab(sd, g["args"], g["data"])
    for k in ("cls_preds", "reg_preds", "dir_preds"):
        torch.testing.assert_close(out[k], g["out"][k], rtol=1e-4, atol=1e-4)
    for a, b in zip(out["occ_single_list"], g["out"]["occ_single_list"]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4)


def test_encoder_and_backbone_small(golden_dir):
    g = _load(golden_dir, "heter_pyramid_collab_small.pt")
    sd = procedural.make_state_dict(g["shapes"])
    args = g["args"]
    with torch.no_grad():
        enc = nets.point_pillar_encoder(sd, "encoder_m1", args["m1"]["encoder_args"], g["data"]["inputs_m1"])
        bb = nets.resnet_bev_backbone(enc, sd, "backbone_m1", args["m1"]["backbone_args"])
    torch.testing.assert_close(enc[:, :, ::4, ::4], g["encoder_feature_sample"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(bb[:, ::4], g["backbone_feature"], rtol=1e-4, atol=1e-4)


def test_warp_and_att(golden_dir):
    g = _load(golden_dir, "warp_att.pt")
    aff = nets.normalize_pairwise_tfm(g["pairwise_t_matrix"], g["H"], g["W"], 1)
    torch.testing.assert_close(aff, g["affine"], rtol=0, atol=0)
    w = nets.warp_affine_simple(g["x"], aff[0, 0, :3], (24, 40))
    torch.testing.assert_close(w[:, ::8], g["warp_s"], rtol=1e-5, atol=1e-5)
    w = nets.warp_affine_simple(g["x"], aff[0, 0, :3], (24, 40), align_corners=True)
    torch.testing.assert_close(w[:, ::8], g["warp_align_corners_s"], rtol=1e-5, atol=1e-5)
    att = nets.att_fusion(g["x"], torch.tensor([3]), aff)
    torch.testing.assert_close(att, g["att"], rtol=1e-4, atol=1e-5)


def test_base_bev_backbone_small(golden_dir):
    g = _load(golden_dir, "base_bev_backbone_small.pt")
    sd = procedural.make_state_dict(g["shapes"])
    sd = {"bb." + k: v for k, v in sd.items()}
    with torch.no_grad():
        y = nets.base_bev_backbone(g["x"], sd, "bb", g["cfg"])
    torch.testing.assert_close(y[:, ::4], g["y_s"], rtol=1e-4, atol=1e-4)


def test_lss_geometry_and_pool(golden_dir):
    from oracle import lss
    g = _load(golden_dir, "lss_small.pt")
    cfg = g["cfg"]
    fr = lss.create_frustum(cfg["grid_conf"], cfg["data_aug_conf"]["final_dim"], cfg["img_downsample"])
    geom = lss.get_geometry(fr, g["rots"], g["trans"], g["intrins"], g["post_rots"], g["post_trans"])
    torch.testing.assert_close(geom, g["geom"], rtol=0, atol=0)
    dx, bx, nx = lss.gen_dx_bx(cfg["grid_conf"]["xbound"], cfg["grid_conf"]["ybound"], cfg["grid_conf"]["zbound"])
    B, N = g["trans"].shape[:2]
    D, fH, fW, _ = fr.shape
    x = lss.outer_product(g["depth_logits"], g["feat"]).view(B, N, -1, D, fH, fW).permute(0, 1, 3, 4, 5, 2)
    bev = lss.voxel_pooling(geom, x, dx, bx, nx, exact=False)
    torch.testing.assert_close(bev, g["bev"], rtol=1e-5, atol=1e-5)          # faithful cumsum-trick restatement
    bev_exact = lss.voxel_pooling(geom, x, dx, bx, nx, exact=True)
    torch.testing.assert_close(bev_exact, g["bev"], rtol=1e-3, atol=1e-4)    # the trick's own cancellation noise


def test_heter_model_baseline_att_small(golden_dir):
    g = _load(golden_dir, "heter_model_baseline_att_small.pt")
    sd = procedural.make_state_dict(g["shapes"])
    with torch.no_grad():
        out = nets.heter_model_baseline(sd, g["args"], g["data"])
    for k in ("cls_preds", "reg_preds", "dir_preds"):
        torch.testing.assert_close(out[k], g["out"][k], rtol=1e-4, atol=1e-4)


def test_convnext_aligner_oracle_vs_reference_golden(golden_dir):
    """oracle.nets.convnext_aligner == the UNMODIFIED reference AlignNet(convnext) output (feature_alignnet_modules.py:299-360)."""
    import os
    g = torch.load(os.path.join(golden_dir, "convnext_aligner.pt"), weights_only=False)
    sd = {"al." + k: v for k, v in procedural.make_state_dict(g["shapes"]).items()}
    with torch.no_grad():
        y = nets.convnext_aligner(g["x"], sd, "al", g["cfg"]["args"]["num_of_blocks"])
    assert (y - g["y"]).abs().max().item() <= 1e-5


def test_point_filters_match_reference(golden_dir):
    """oracle/pcd.py vs the unmodified reference's pcd_utils (mask_points_by_range / mask_ego_points / shuffle_points), whose
    outputs point_filters.npz stores as row masks (oracle/make_golden.py::make_point_filter_golden)."""
    from oracle import make_golden, pcd
    g = np.load(os.path.join(golden_dir, "point_filters.npz"))
    pts, lim = make_golden.point_filter_cloud(), g["limit"].tolist()
    n = pts.shape[0]
    assert np.array_equal(pcd.mask_points_by_range(pts, lim), pts[np.unpackbits(g["by_range"], count=n).astype(bool)])
    assert np.array_equal(pcd.mask_ego_points(pts), pts[np.unpackbits(g["ego"], count=n).astype(bool)])
    np.random.seed(3)                                             # the reference's shuffle_points draws np.random.permutation
    perm = np.random.permutation(n)
    expect = pts[perm][np.unpackbits(g["shuffle_seed3_ego_range"], count=n).astype(bool)]
    assert np.array_equal(pcd.filter_cloud(pts, lim, perm), expect)
