"""CPU: the stage-4 tail (SURVEY.md section 8f rank 3) -- pycolmap-free COLMAP sparse-model writer/reader, the cloud and
camera exports of stages/camera_and_pointcloud/minimal_demo_vggt.py.  pycolmap is not installed here, so the builder is
checked against a literal restatement of the reference's per-point loop (np_to_pycolmap.py:201-290), the files against
the format's layout and their own reader, and the small numeric helpers and the image loader against the reference's
outputs (tests/golden/host_helpers.npz, oracle/make_golden.py)."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "stages", "camera_and_pointcloud"))
colmap_io = importlib.import_module("colmap_io")
stage4 = importlib.import_module("minimal_demo_vggt")


def _rand_rot(rng):
    q = rng.normal(size=4)
    return colmap_io.qvec_to_rotmat(q / np.linalg.norm(q))


def test_rotmat_qvec_roundtrip_all_branches():
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(0)
    mats = [_rand_rot(rng) for _ in range(200)]
    mats += [np.diag([1.0, -1, -1]), np.diag([-1.0, 1, -1]), np.diag([-1.0, -1, 1]), np.eye(3)]   # trace <= 0 branches
    for R in mats:
        q = colmap_io.rotmat_to_qvec(R)
        assert abs(np.linalg.norm(q) - 1) < 1e-12
        assert np.allclose(colmap_io.qvec_to_rotmat(q), R, atol=1e-12)
        qs = Rotation.from_matrix(R).as_quat()   # x, y, z, w
        qs = np.array([qs[3], qs[0], qs[1], qs[2]])
        assert min(np.abs(q - qs).max(), np.abs(q + qs).max()) < 1e-9


def _loop_builder(points3d, points_xyf, points_rgb, extrinsics, intrinsics, image_size):
    """np_to_pycolmap.py:201-290 restated with plain containers (PINHOLE, not shared)."""
    pts = {i + 1: dict(xyz=points3d[i], rgb=points_rgb[i], track=[]) for i in range(len(points3d))}
    cams, imgs = {}, {}
    for f in range(len(extrinsics)):
        K = intrinsics[f]
        cams[f + 1] = dict(params=np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]]), width=image_size[0], height=image_size[1])
        p2d = []
        for b in np.nonzero(points_xyf[:, 2].astype(np.int32) == f)[0]:
            pts[b + 1]["track"].append((f + 1, len(p2d)))
            p2d.append((points_xyf[b, :2], b + 1))
        imgs[f + 1] = dict(name=f"image_{f + 1}", camera_id=f + 1, R=extrinsics[f][:3, :3], t=extrinsics[f][:3, 3], p2d=p2d)
    return pts, cams, imgs


def _scene(rng, S=2, H=6, W=7, keep=0.6):
    xyf = stage4.create_pixel_coordinate_grid(S, H, W)
    mask = rng.random((S, H, W)) < keep
    p3 = rng.normal(size=(S, H, W, 3))
    rgb = rng.integers(0, 256, (S, H, W, 3)).astype(np.uint8)
    E = np.stack([np.concatenate([_rand_rot(rng), rng.normal(size=(3, 1))], 1) for _ in range(S)])
    K = np.stack([np.array([[500 + f, 0, W / 2], [0, 510 + f, H / 2], [0, 0, 1.0]]) for f in range(S)])
    return p3[mask], xyf[mask], rgb[mask], E, K, mask


def test_builder_matches_the_reference_loop_and_files_roundtrip(tmp_path):
    rng = np.random.default_rng(1)
    p3, xyf, rgb, E, K, _ = _scene(rng)
    rc = colmap_io.build_reconstruction_wo_track(p3, xyf, rgb, E, K, np.array([518, 518]))
    pts, cams, imgs = _loop_builder(p3, xyf, rgb, E, K, (518, 518))
    assert sorted(rc.cameras) == sorted(cams) and sorted(rc.images) == sorted(imgs)
    for cid in cams:
        assert np.array_equal(rc.cameras[cid]["params"], cams[cid]["params"]) and rc.cameras[cid]["model"] == "PINHOLE"
    for iid, im in imgs.items():
        got = rc.images[iid]
        assert got["name"] == im["name"] and got["camera_id"] == im["camera_id"]
        assert np.allclose(colmap_io.qvec_to_rotmat(got["qvec"]), im["R"], atol=1e-12) and np.array_equal(got["tvec"], im["t"])
        assert len(got["xys"]) == len(im["p2d"])
        for j, (xy, pid) in enumerate(im["p2d"]):
            assert np.array_equal(got["xys"][j], xy) and got["point3D_ids"][j] == pid
    for pid, p in pts.items():
        assert np.array_equal(rc.points_xyz[pid - 1], p["xyz"]) and np.array_equal(rc.points_rgb[pid - 1], p["rgb"])
        assert [(rc.track_image[pid - 1], rc.track_p2d[pid - 1])] == p["track"]
    rc.write(str(tmp_path))
    P, n2 = len(p3), [len(rc.images[i]["xys"]) for i in sorted(rc.images)]
    assert os.path.getsize(tmp_path / "cameras.bin") == 8 + 2 * (24 + 32)
    assert os.path.getsize(tmp_path / "points3D.bin") == 8 + P * (8 + 24 + 3 + 8 + 8 + 8)
    assert os.path.getsize(tmp_path / "images.bin") == 8 + sum(4 + 32 + 24 + 4 + len(f"image_{i + 1}") + 1 + 8 + 24 * n
                                                              for i, n in enumerate(n2))
    back = colmap_io.Reconstruction.read(str(tmp_path))
    assert np.array_equal(back.points_xyz, rc.points_xyz) and np.array_equal(back.points_rgb, rc.points_rgb)
    assert np.array_equal(back.track_image, rc.track_image) and np.array_equal(back.track_p2d, rc.track_p2d)
    for iid in rc.images:
        for k in ("qvec", "tvec", "xys", "point3D_ids"):
            assert np.array_equal(back.images[iid][k], rc.images[iid][k])
        assert back.images[iid]["name"] == rc.images[iid]["name"]
    for cid in rc.cameras:
        assert np.array_equal(back.cameras[cid]["params"], rc.cameras[cid]["params"])
        assert (back.cameras[cid]["width"], back.cameras[cid]["height"]) == (518, 518)


def test_rename_and_rescale_follows_the_reference_arithmetic():
    rng = np.random.default_rng(2)
    p3, xyf, rgb, E, K, _ = _scene(rng)
    rc = colmap_io.build_reconstruction_wo_track(p3, xyf, rgb, E, K, np.array([518, 518]))
    before = {i: (rc.cameras[i]["params"].copy(), rc.images[i]["xys"].copy()) for i in rc.images}
    coords = np.array([[0.0, 86.3, 518.0, 431.7, 1500, 1000], [12.0, 0.0, 506.0, 518.0, 800, 840]])
    colmap_io.rename_and_rescale(rc, ["a/b.jpg", "c.png"], coords, img_size=518, shift_point2d_to_original_res=True)
    for iid in rc.images:
        real = coords[iid - 1, -2:]
        ratio = max(real) / 518
        exp = before[iid][0] * ratio
        exp[-2:] = real / 2
        assert np.allclose(rc.cameras[iid]["params"], exp) and rc.cameras[iid]["width"] == int(real[0])
        assert np.allclose(rc.images[iid]["xys"], (before[iid][1] - coords[iid - 1, :2]) * ratio)
    assert rc.images[1]["name"] == "a/b.jpg"


def test_small_helpers_against_the_reference_when_available(golden_dir):
    z = np.load(os.path.join(golden_dir, "host_helpers.npz"))
    assert np.array_equal(stage4.create_pixel_coordinate_grid(2, 5, 4), z["pixel_grid"])
    m = np.random.default_rng(3).random((2, 30, 30)) > 0.3
    np.random.seed(7)
    a = stage4.randomly_limit_trues(m, 100)
    assert np.array_equal(a, z["limited_mask"]) and a.sum() == 100
    # B2P: restated from src/utils/global_utils.py:835-844 (that module imports pytorch3d, absent here): check the
    # published identity instead -- R is B's rotation conjugated by two axis permutations, T = P_T t R
    B = np.eye(4)
    B[:3, :3], B[:3, 3] = _rand_rot(np.random.default_rng(4)), [0.3, -1.2, 2.0]
    R, T = stage4.B2P(B)
    assert np.allclose(R @ R.T, np.eye(3)) and np.isclose(np.linalg.det(R), 1.0)
    assert np.allclose(np.linalg.norm(T), np.linalg.norm(B[:3, 3]))


def test_sparse_model_and_camera_export_end_to_end(tmp_path):
    rng = np.random.default_rng(5)
    S, H, W = 2, 20, 20
    pts = rng.normal(size=(S, H, W, 3))
    conf = rng.random((S, H, W)) * 10
    img = rng.random((S, 3, H, W)).astype(np.float32)
    E = np.stack([np.concatenate([_rand_rot(rng), rng.normal(size=(3, 1))], 1) for _ in range(S)]).astype(np.float32)
    K = np.stack([np.array([[300.0, 0, 10], [0, 310.0, 10], [0, 0, 1]]) for _ in range(S)]).astype(np.float32)
    coords = np.array([[0, 3.3, 20, 16.7, 1500, 1000], [0, 0, 20, 20, 900, 900]], dtype=np.float64)
    out = tmp_path / "sparse"
    cfg = {"output_vggt": str(out), "camera": str(tmp_path / "cam" / "camera.npz"), "conf_thres_value": 5.0,
           "max_points_for_colmap": 150, "vggt_cloud": str(tmp_path / "cloud" / "scene.ply"), "vggt_scene_scale": 5.0}
    os.makedirs(out)
    np.random.seed(0)
    stage4.write_sparse_model(str(out), pts, conf, img, E, K, ["main.jpg", "empty_room.png"], coords, cfg, resolution=H)
    for f in ("cameras.bin", "images.bin", "points3D.bin", "image_list.txt", "points_merged.ply", "points.ply",
              "points_emptyRoom_pre.ply", "points_emptyRoom.ply"):
        assert (out / f).exists(), f
    rc = colmap_io.Reconstruction.read(str(out))
    assert len(rc.points_xyz) == 150 and rc.images[1]["name"] == "main.jpg"
    p0 = stage4.read_ply_vertices(str(out / "points.ply"))
    fit = stage4.read_ply_vertices(str(out / "points_emptyRoom.ply"))
    assert np.allclose(fit.max(0) - fit.min(0), p0.max(0) - p0.min(0), rtol=1e-4)     # bbox fitted to the main cloud
    rec, scene = stage4.export_vggt_data(cfg)
    z = np.load(cfg["camera"])
    assert set(z.files) == {"extrinsic", "focal", "image_size", "camera_angle_x"}
    assert z["extrinsic"].dtype == np.float32 and z["extrinsic"].shape == (4, 4) and z["image_size"].dtype == np.int32
    assert tuple(z["image_size"]) == (1500, 1000)
    ratio = 1500 / H
    focal = (300.0 * ratio + 310.0 * ratio) / 2
    assert np.isclose(z["focal"], focal, rtol=1e-6) and np.isclose(z["camera_angle_x"], 2 * np.arctan(1500 / (2 * focal)), rtol=1e-6)
    R_fix = np.array([[1, 0, 0], [0, 0, -1], [0, 1, 0]], dtype=np.float32)
    assert np.allclose(z["extrinsic"][:3, :3], R_fix @ E[0][:, :3], atol=1e-5)
    assert (tmp_path / "cam" / "camera_emptyRoom.npz").exists()
    Rp, Tp = stage4.B2P(z["extrinsic"])
    exp = ((p0 @ R_fix.T) @ Rp.T + Tp) * np.array([1, -1, 1]) * 5.0
    assert np.allclose(stage4.read_ply_vertices(cfg["vggt_cloud"]), exp, atol=1e-4)


def test_image_loader_against_the_reference_when_available(tmp_path, golden_dir):
    """Row v1: load_and_preprocess_images_square (vggt/vggt/utils/load_fn.py:13-94) -- RGBA on white, centre padding to a
    black square, PIL bicubic resize, ToTensor -- and the original-coordinate table the rescale step consumes.  The
    reference's images are stored as digests of their bytes."""
    import torch
    from make_golden import loader_pngs, sha256
    z = np.load(os.path.join(golden_dir, "host_helpers.npz"))
    paths = loader_pngs(tmp_path)
    for tag, sel in (("3", paths), ("1", paths[:1])):
        a_img, a_xy = stage4.load_and_preprocess_images_square(sel, 256)
        assert tuple(a_img.shape) == tuple(z[f"loader{tag}_shape"]) and a_img.dtype == torch.float32
        assert sha256(a_img) == z[f"loader{tag}_sha256"]
        assert torch.equal(a_xy, torch.from_numpy(z[f"loader{tag}_coords"]))
    with pytest.raises(ValueError):
        stage4.load_and_preprocess_images_square([], 256)
