"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.pt by running the UNMODIFIED reference
modules (imported from /root/reference through oracle/ref_shim.py) on CPU with procedural weights and
seeded inputs.  Run in the build container only:  python -m oracle.make_golden
The fixtures pin oracle/nets.py (tests/test_oracle_golden.py) and are the reference-derived vectors
the CUDA path is checked against on the GPU box (tests/test_gpu_*.py)."""
import copy
import os
import sys

import numpy as np
import torch

from oracle import ref_shim, procedural, voxelizer

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")

SMALL_RANGE = [-12.8, -12.8, -3, 12.8, 12.8, 1]     # 64 x 64 pillars @ 0.4 m
VOXEL = [0.4, 0.4, 4]


def small_model_args():
    return {
        "lidar_range": SMALL_RANGE, "supervise_single": True,
        "m1": {
            "core_method": "point_pillar", "sensor_type": "lidar",
            "encoder_args": {"voxel_size": VOXEL, "lidar_range": SMALL_RANGE,
                             "pillar_vfe": {"use_norm": True, "with_distance": False, "use_absolute_xyz": True,
                                            "num_filters": [64]},
                             "point_pillar_scatter": {"num_features": 64}},
            "backbone_args": {"layer_nums": [3], "layer_strides": [2], "num_filters": [64]},
            "aligner_args": {"core_method": "identity"},
        },
        "fusion_backbone": {"resnext": True, "layer_nums": [3, 5, 8], "layer_strides": [1, 2, 2],
                            "num_filters": [64, 128, 256], "upsample_strides": [1, 2, 4],
                            "num_upsample_filter": [128, 128, 128], "anchor_number": 2},
        "shrink_header": {"kernal_size": [3], "stride": [1], "padding": [1], "dim": [256], "input_dim": 384},
        "in_head": 256, "anchor_number": 2, "dir_args": {"dir_offset": 0.7853, "num_bins": 2, "anchor_yaw": [0, 90]},
    }


def baseline_att_args(core_method="point_pillar", encoder_args=None, inplanes=64, strides=(2, 2, 2)):
    enc = encoder_args or {"voxel_size": VOXEL, "lidar_range": SMALL_RANGE,
                           "pillar_vfe": {"use_norm": True, "with_distance": False, "use_absolute_xyz": True, "num_filters": [64]},
                           "point_pillar_scatter": {"num_features": 64}}
    return {
        "lidar_range": SMALL_RANGE, "ego_modality": "m1",
        "m1": {"core_method": core_method, "sensor_type": "lidar", "encoder_args": enc,
               "backbone_args": {"layer_nums": [3, 5, 8], "layer_strides": list(strides), "num_filters": [64, 128, 256],
                                 "upsample_strides": [1, 2, 4], "num_upsample_filter": [128, 128, 128], "inplanes": inplanes},
               "shrink_header": {"kernal_size": [3], "stride": [1], "padding": [1], "dim": [256], "input_dim": 384}},
        "fusion_method": "att", "att": {"feat_dim": 256},
        "in_head": 256, "anchor_number": 2, "dir_args": {"dir_offset": 0.7853, "num_bins": 2, "anchor_yaw": [0, 90]},
    }


def lss_small_cfg():
    return {"grid_conf": {"xbound": [-12.8, 12.8, 0.4], "ybound": [-12.8, 12.8, 0.4], "zbound": [-10, 10, 20.0],
                          "ddiscr": [2, 30, 16], "mode": "LID"},
            "data_aug_conf": {"final_dim": [64, 128]}, "img_downsample": 8, "img_features": 32,
            "camera_encoder": "Resnet101", "use_depth_gt": False, "depth_supervision": False}


def small_scene(seed=7, n_agents=3, pts_per_agent=1500):
    rng = np.random.default_rng(seed)
    per_agent = []
    for a in range(n_agents):
        p = np.concatenate([rng.uniform(-14, 14, (pts_per_agent, 2)), rng.uniform(-3.5, 1.5, (pts_per_agent, 1)),
                            rng.uniform(0, 1, (pts_per_agent, 1))], 1).astype(np.float32)
        per_agent.append(voxelizer.points_to_voxel_c(p, VOXEL, SMALL_RANGE, 32, 70000))
    col = voxelizer.collate(per_agent)
    from heal_b200 import synth
    poses = [[0, 0, 0, 0, 0, 0]] + [[rng.uniform(-5, 5), rng.uniform(-5, 5), 0, 0, rng.uniform(-180, 180), 0]
                                    for _ in range(n_agents - 1)]
    pw = synth.pairwise_t_matrix(poses, 5)[None]
    return {
        "inputs_m1": {k: torch.from_numpy(v) for k, v in col.items()},
        "agent_modality_list": ["m1"] * n_agents,
        "record_len": torch.tensor([n_agents], dtype=torch.long),
        "pairwise_t_matrix": torch.from_numpy(pw),
    }


def main():
    ref_shim.install()
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    from opencood.models.heter_pyramid_collab import HeterPyramidCollab
    from opencood.models.fuse_modules.fusion_in_one import AttFusion
    from opencood.models.sub_modules.torch_transformation_utils import warp_affine_simple
    from opencood.models.sub_modules.base_bev_backbone import BaseBEVBackbone
    from opencood.models.sub_modules.pillar_vfe import PillarVFE
    from opencood.utils.transformation_utils import normalize_pairwise_tfm

    # ---- 1. full HeterPyramidCollab (C2-shaped, small grid) -------------------------------------
    args = small_model_args()
    model = HeterPyramidCollab(copy.deepcopy(args)).eval()
    shapes = procedural.shapes_of(model)
    sd = procedural.make_state_dict(shapes)
    model.load_state_dict(sd, strict=True)
    data = small_scene()
    with torch.no_grad():
        dd = copy.deepcopy(data)
        out = model(dd)
        # intermediate: encoder + backbone features, for finer-grained parity
        enc = model.encoder_m1(copy.deepcopy(data), "m1")
        bb = model.backbone_m1({"spatial_features": enc})["spatial_features_2d"]
    torch.save({
        "args": args, "shapes": shapes, "data": data,
        "out": {"cls_preds": out["cls_preds"], "reg_preds": out["reg_preds"], "dir_preds": out["dir_preds"],
                "occ_single_list": out["occ_single_list"]},
        "encoder_feature_sample": enc[:, :, ::4, ::4].contiguous(),
        "backbone_feature": bb[:, ::4].contiguous(),
    }, os.path.join(OUT, "heter_pyramid_collab_small.pt"))
    print("heter_pyramid_collab_small:", {k: tuple(v.shape) for k, v in out.items() if torch.is_tensor(v)})

    # ---- 2. warp_affine_simple + normalize_pairwise_tfm + AttFusion ------------------------------
    g = torch.Generator().manual_seed(11)
    x = torch.randn(3, 128, 24, 40, generator=g)
    aff = normalize_pairwise_tfm(data["pairwise_t_matrix"].clone(), 9.6, 16.0, 1)
    with torch.no_grad():
        w = warp_affine_simple(x, aff[0, 0, :3], (24, 40))
        w_ac = warp_affine_simple(x, aff[0, 0, :3], (24, 40), align_corners=True)
        att = AttFusion(128)(x, torch.tensor([3]), aff)
    torch.save({"x": x, "pairwise_t_matrix": data["pairwise_t_matrix"], "H": 9.6, "W": 16.0, "affine": aff,
                "warp_s": w[:, ::8].contiguous(), "warp_align_corners_s": w_ac[:, ::8].contiguous(), "att": att}, os.path.join(OUT, "warp_att.pt"))
    print("warp_att:", tuple(w.shape), tuple(att.shape))

    # ---- 3. BaseBEVBackbone [1,1,1] (AttFuse-config family, small) -------------------------------
    cfg = {"layer_nums": [1, 2, 1], "layer_strides": [2, 2, 2], "num_filters": [64, 128, 256],
           "upsample_strides": [1, 2, 4], "num_upsample_filter": [128, 128, 128]}
    bbm = BaseBEVBackbone(copy.deepcopy(cfg), 64).eval()
    bshapes = procedural.shapes_of(bbm)
    bbm.load_state_dict(procedural.make_state_dict(bshapes), strict=True)
    xin = torch.randn(2, 64, 32, 48, generator=g)
    with torch.no_grad():
        y = bbm({"spatial_features": xin})["spatial_features_2d"]
    torch.save({"cfg": cfg, "shapes": bshapes, "x": xin, "y_s": y[:, ::4].contiguous()}, os.path.join(OUT, "base_bev_backbone_small.pt"))
    print("base_bev_backbone_small:", tuple(y.shape))
    # ---- 4. Lift-Splat-Shoot geometry + voxel pooling (reference methods on a ctor-less instance) ------
    from opencood.models.heter_encoders import LiftSplatShoot
    from opencood.utils.camera_utils import gen_dx_bx
    from heal_b200 import synth
    lcfg = lss_small_cfg()
    obj = LiftSplatShoot.__new__(LiftSplatShoot)
    torch.nn.Module.__init__(obj)
    obj.grid_conf, obj.data_aug_conf, obj.downsample = lcfg["grid_conf"], lcfg["data_aug_conf"], lcfg["img_downsample"]
    obj.dx, obj.bx, obj.nx = gen_dx_bx(lcfg["grid_conf"]["xbound"], lcfg["grid_conf"]["ybound"], lcfg["grid_conf"]["zbound"])
    obj.frustum = obj.create_frustum()
    obj.use_quickcumsum = True
    D, fH, fW, _ = obj.frustum.shape
    Bn, Nc, Cc = 2, 2, 32
    rots, trans, intr, post_rots, post_trans = [torch.from_numpy(a) for a in synth.camera_rig(Bn, Nc, 64, 128)]
    gl = torch.Generator().manual_seed(21)
    post_rots = post_rots.clone()
    post_rots[:, :, 0, 0] = 0.9 + 0.2 * torch.rand(Bn, Nc, generator=gl)
    post_rots[:, :, 1, 1] = post_rots[:, :, 0, 0]
    post_trans = post_trans.clone()
    post_trans[:, :, :2] = torch.randn(Bn, Nc, 2, generator=gl) * 3
    depth_logits = torch.randn(Bn * Nc, D, fH, fW, generator=gl) * 2
    feat = torch.randn(Bn * Nc, Cc, fH, fW, generator=gl)
    with torch.no_grad():
        geom = obj.get_geometry(rots, trans, intr, post_rots, post_trans)
        new_x = torch.softmax(depth_logits, dim=1).unsqueeze(1) * feat.unsqueeze(2)        # lss_submodule.py:228-229
        xx = new_x.view(Bn, Nc, Cc, D, fH, fW).permute(0, 1, 3, 4, 5, 2)                   # heter_encoders.py:156-157
        bev = obj.voxel_pooling(geom, xx)
    torch.save({"cfg": lcfg, "rots": rots, "trans": trans, "intrins": intr, "post_rots": post_rots, "post_trans": post_trans,
                "depth_logits": depth_logits, "feat": feat, "geom": geom, "bev": bev}, os.path.join(OUT, "lss_small.pt"))
    print("lss_small:", tuple(geom.shape), tuple(bev.shape), float(bev.abs().max()))
    # ---- 5. HeterModelBaseline + AttFusion (C3 family; PointPillar encoder so that the reference runs without spconv) ----
    from opencood.models.heter_model_baseline import HeterModelBaseline
    bargs = baseline_att_args()
    bm = HeterModelBaseline(copy.deepcopy(bargs)).eval()
    bshapes2 = procedural.shapes_of(bm)
    bm.load_state_dict(procedural.make_state_dict(bshapes2), strict=True)
    with torch.no_grad():
        bout = bm(copy.deepcopy(data))
    torch.save({"args": bargs, "shapes": bshapes2, "data": data,
                "out": {k: bout[k] for k in ("cls_preds", "reg_preds", "dir_preds")}},
               os.path.join(OUT, "heter_model_baseline_att_small.pt"))
    print("heter_model_baseline_att_small:", {k: tuple(v.shape) for k, v in bout.items() if torch.is_tensor(v)})
    make_convnext_golden()
    make_postprocess_golden()
    make_point_filter_golden()
    make_full_size_golden()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")


def make_convnext_golden():
    """UNMODIFIED reference AlignNet(core_method='convnext') (feature_alignnet.py:12-39 -> feature_alignnet_modules.ConvNeXt)."""
    ref_shim.install()
    from opencood.models.sub_modules.feature_alignnet import AlignNet
    cfg = {"core_method": "convnext", "spatial_align": False, "args": {"num_of_blocks": 3, "dim": 64}}
    m = AlignNet(copy.deepcopy(cfg)).eval()
    shapes = procedural.shapes_of(m)
    m.load_state_dict(procedural.make_state_dict(shapes), strict=True)
    x = torch.randn(2, 64, 24, 40, generator=torch.Generator().manual_seed(31))
    with torch.no_grad():
        y = m(x)
    torch.save({"cfg": cfg, "shapes": shapes, "x": x, "y": y}, os.path.join(OUT, "convnext_aligner.pt"))
    print("convnext_aligner:", tuple(y.shape), float(y.abs().max()), float((y - x).abs().max()))


def postprocess_params(rng=(-25.6, -25.6, -3, 25.6, 25.6, 1), voxel=(0.4, 0.4, 4)):
    """`postprocess:` block of opv2v/MoreModality/HEAL/stage1/m1_pyramid.yaml:67-88 with the anchor grid that
    yaml_utils.load_point_pillar_params (:121-135) derives, on a small range."""
    import math
    rng = list(rng)
    return {"core_method": "VoxelPostprocessor", "gt_range": rng,
            "anchor_args": {"cav_lidar_range": rng, "l": 3.9, "w": 1.6, "h": 1.56, "r": [0, 90], "feature_stride": 2, "num": 2,
                            "vw": voxel[0], "vh": voxel[1], "vd": voxel[2],
                            "W": math.ceil((rng[3] - rng[0]) / voxel[0]), "H": math.ceil((rng[4] - rng[1]) / voxel[1]),
                            "D": math.ceil((rng[5] - rng[2]) / voxel[2])},
            "target_args": {"pos_threshold": 0.6, "neg_threshold": 0.45, "score_threshold": 0.2},
            "order": "hwl", "max_num": 150, "nms_thresh": 0.15,
            "dir_args": {"dir_offset": 0.7853, "num_bins": 2, "anchor_yaw": [0, 90]}}


def postprocess_inputs(params, seed=3, logit_mean=-3.0):
    """seeded head outputs: ~14 % of the anchors above the score threshold (more than the NMS's top-1000 cut on the 64x64 map),
    deltas small enough that neighbouring boxes overlap, a rigid ego transform."""
    g = torch.Generator().manual_seed(seed)
    aa = params["anchor_args"]
    h, w = aa["H"] // aa["feature_stride"], aa["W"] // aa["feature_stride"]
    cls = logit_mean + 1.5 * torch.randn((1, 2, h, w), generator=g)
    reg = 0.3 * torch.randn((1, 14, h, w), generator=g)
    reg[:, 2::7] *= 0.3                                    # z delta: keep most boxes inside [-3, 1]
    dirp = torch.randn((1, 4, h, w), generator=g)
    yaw = 0.3
    T = torch.tensor([[np.cos(yaw), -np.sin(yaw), 0, 1.5], [np.sin(yaw), np.cos(yaw), 0, -0.7], [0, 0, 1, 0.1], [0, 0, 0, 1]],
                     dtype=torch.float32)
    return cls, reg, dirp, T


def make_postprocess_golden():
    """UNMODIFIED reference VoxelPostprocessor.post_process (voxel_postprocessor.py:245-405).  shapely is absent: the reference's
    `from shapely.geometry import Polygon` resolves to oracle.postprocess.QuadPolygon (see that file's header); the cython
    opencood.utils.box_overlaps (training labels only) is stubbed."""
    import types
    from unittest.mock import MagicMock
    from oracle import postprocess as opp
    sg = types.ModuleType("shapely.geometry")
    sg.Polygon = opp.QuadPolygon
    sh = types.ModuleType("shapely")
    sh.geometry = sg
    sys.modules["shapely"], sys.modules["shapely.geometry"] = sh, sg
    sys.modules.setdefault("opencood.utils.box_overlaps", MagicMock())
    for m in [k for k in sys.modules if k.startswith("opencood.utils.common_utils") or k.startswith("opencood.utils.box_utils")]:
        del sys.modules[m]
    ref_shim.install()
    from opencood.data_utils.post_processor.voxel_postprocessor import VoxelPostprocessor
    import opencood.utils.common_utils as cu
    assert cu.Polygon is opp.QuadPolygon
    params = postprocess_params()
    pp = VoxelPostprocessor(copy.deepcopy(params), train=False)
    anchors = torch.from_numpy(pp.generate_anchor_box())
    cases = {}
    for name, seed, mean in (("dense", 3, -3.0), ("sparse", 4, -6.0)):
        cls, reg, dirp, T = postprocess_inputs(params, seed, mean)
        data = {"ego": {"transformation_matrix": T, "anchor_box": anchors}}
        out = {"ego": {"cls_preds": cls.clone(), "reg_preds": reg.clone(), "dir_preds": dirp.clone()}}
        with torch.no_grad():
            boxes, scores = pp.post_process(data, out)
        cases[name] = {"cls": cls, "reg": reg, "dir": dirp, "T": T, "boxes": boxes, "scores": scores}
        print("postprocess", name, "candidates", int((torch.sigmoid(cls) > 0.2).sum()), "-> kept", 0 if boxes is None else boxes.shape[0])
    # late fusion (two cavs, each with its own cav->ego transform; one NMS over both box sets) and iou_preds rescoring
    multi = {}
    T2 = torch.tensor([[np.cos(-0.4), -np.sin(-0.4), 0, -3.0], [np.sin(-0.4), np.cos(-0.4), 0, 2.5], [0, 0, 1, -0.05], [0, 0, 0, 1]],
                      dtype=torch.float32)
    heads = [postprocess_inputs(params, 5, -4.0), postprocess_inputs(params, 6, -4.0)]
    data = {"ego": {"transformation_matrix": heads[0][3], "anchor_box": anchors}, "cav1": {"transformation_matrix": T2, "anchor_box": anchors}}
    out = {k: {"cls_preds": h[0].clone(), "reg_preds": h[1].clone(), "dir_preds": h[2].clone()} for k, h in zip(("ego", "cav1"), heads)}
    with torch.no_grad():
        boxes, scores = pp.post_process(data, out)
    multi["late2"] = {"cavs": [{"cls": h[0], "reg": h[1], "dir": h[2], "T": t} for h, t in zip(heads, (heads[0][3], T2))],
                      "boxes": boxes, "scores": scores}
    print("postprocess late2 -> kept", boxes.shape[0])
    cls, reg, dirp, T = postprocess_inputs(params, 7, -3.5)
    iou = torch.randn(cls.shape, generator=torch.Generator().manual_seed(17))
    with torch.no_grad():
        boxes, scores = pp.post_process({"ego": {"transformation_matrix": T, "anchor_box": anchors}},
                                        {"ego": {"cls_preds": cls.clone(), "reg_preds": reg.clone(), "dir_preds": dirp.clone(), "iou_preds": iou.clone()}})
    multi["iou"] = {"cavs": [{"cls": cls, "reg": reg, "dir": dirp, "iou": iou, "T": T}], "boxes": boxes, "scores": scores}
    print("postprocess iou -> kept", boxes.shape[0])
    torch.save({"params": params, "anchors": anchors, "cases": cases, "multi": multi}, os.path.join(OUT, "postprocess.pt"))


def point_filter_cloud():
    """(20000, 4) cloud with plenty of points in and around the ego box and on the range / ego-box edges."""
    rng = np.random.default_rng(5)
    pts = rng.uniform(-120, 120, size=(20000, 4)).astype(np.float32)
    pts[:, 2] = rng.uniform(-4, 2, size=20000)
    pts[:2000, :2] = rng.uniform(-3, 3, size=(2000, 2))
    pts[2000:2006] = [[-1.95, 0, 0, 1], [2.95, 1.1, 0, 1], [102.4, 0, 0, 1], [0, -102.4, 0, 1], [5, 5, -3, 1], [5, 5, 1, 1]]
    return pts


POINT_FILTER_LIMIT = [-102.4, -102.4, -3, 102.4, 102.4, 1]


def make_point_filter_golden():
    """UNMODIFIED reference pcd_utils mask_points_by_range / mask_ego_points / shuffle_points (pcd_utils.py:41-95) on
    point_filter_cloud().  Their outputs are stored as bit-packed row masks: over the cloud for the two filters, over the cloud
    shuffled with np.random.seed(3) for shuffle -> ego mask -> range mask.  To read the masks off the reference's outputs, the
    cloud gets its row index as a fifth column, which the filters carry along untouched (they read columns 0-2 only)."""
    from unittest.mock import MagicMock
    ref_shim.install()
    sys.modules.setdefault("pypcd", MagicMock(name="pypcd"))
    from opencood.utils import pcd_utils as ref
    pts = point_filter_cloud()
    n, lim = pts.shape[0], POINT_FILTER_LIMIT
    tagged = np.concatenate([pts, np.arange(n, dtype=np.float32)[:, None]], 1)
    np.random.seed(3)
    perm = np.random.permutation(n)

    def mask(out5, out4, order):
        rows = out5[:, 4].astype(np.int64)
        assert np.array_equal(pts[rows], out4)
        m = np.isin(order, rows)
        assert np.array_equal(order[m], rows)                      # the filters keep the order of their input
        return np.packbits(m)
    by_range = mask(ref.mask_points_by_range(tagged, lim), ref.mask_points_by_range(pts, lim), np.arange(n))
    ego = mask(ref.mask_ego_points(tagged), ref.mask_ego_points(pts), np.arange(n))
    np.random.seed(3)
    s5 = ref.shuffle_points(tagged)
    np.random.seed(3)
    s4 = ref.shuffle_points(pts)
    assert np.array_equal(s5[:, 4].astype(np.int64), perm)
    chain = mask(ref.mask_points_by_range(ref.mask_ego_points(s5), lim), ref.mask_points_by_range(ref.mask_ego_points(s4), lim), perm)
    np.savez_compressed(os.path.join(OUT, "point_filters.npz"), limit=np.asarray(lim, np.float64),
                        by_range=by_range, ego=ego, shuffle_seed3_ego_range=chain)


FULL_SIZE_SAMPLES = 8192        # values stored per head: keeps the files small
FULL_SIZE_STRIDE = 104729       # prime: on the 256x256 heads the sample visits every (channel, row) pair and every column


def full_size_sample_index(numel):
    """Flat positions of the stored sample of a head with `numel` elements."""
    return (np.arange(FULL_SIZE_SAMPLES, dtype=np.int64) * FULL_SIZE_STRIDE) % numel


def make_full_size_golden():
    """UNMODIFIED reference PointPillar (configs[0]) and HeterPyramidCollab (configs[1]) at full size on CPU, on the clouds
    tests/test_gpu_fullsize.py feeds the CUDA path.  Stored per head: its shape, max |ref| over the whole head (the tolerance
    scale) and the values at full_size_sample_index()."""
    from oracle import ref_runner
    from workloads import configs as wcfg, synth
    torch.set_num_threads(max(1, min(32, os.cpu_count() or 1)))

    def heads(out):
        rec = {}
        for k in ("cls_preds", "reg_preds", "dir_preds"):
            v = out[k].detach().float()
            idx = torch.from_numpy(full_size_sample_index(v.numel()))
            rec[k] = {"shape": tuple(v.shape), "max_abs": float(v.abs().max()), "value": v.reshape(-1)[idx].clone()}
        return rec
    # C2: tests/test_gpu_fullsize.py::_scene(5) (seed 321, 64 x 1024 rays per agent)
    sc = synth.scene(321, n_agents=5, max_cav=5, rings=64, azimuth=1024)
    model, _ = ref_runner.build_model("heter_pyramid_collab", wcfg.c2_args())
    data, _ = ref_runner.c2_data({"clouds": sc["points"], "pairwise": sc["pairwise_t_matrix"]}, 5)
    torch.save({"shapes": procedural.shapes_of(model), "heads": heads(ref_runner.forward(model, data))},
               os.path.join(OUT, "full_size_c2.pt"))
    # C1: one 20 x 1000-ray cloud
    cloud = synth.lidar_cloud(np.random.default_rng(77), rings=20, azimuth=1000)
    model, _ = ref_runner.build_model("point_pillar", wcfg.c1_args())
    data, _ = ref_runner.c1_data(cloud)
    torch.save({"shapes": procedural.shapes_of(model), "heads": heads(ref_runner.forward(model, data))},
               os.path.join(OUT, "full_size_c1.pt"))


if __name__ == "__main__":
    main()
