"""CPU: host-side logic of the pipeline mirror that needs no GPU (mesh export, scheduler mirror, image processor,
stage-script helpers)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_simple_mesh_glb_roundtrip(tmp_path):
    import json
    import struct
    from r3g.pipelines import SimpleMesh
    v = np.random.rand(5, 3).astype(np.float32)
    f = np.array([[0, 1, 2], [2, 3, 4]], np.int32)
    p = SimpleMesh(v, f).export(str(tmp_path / "a.glb"))
    raw = open(p, "rb").read()
    magic, ver, total = struct.unpack("<4sII", raw[:12])
    assert magic == b"glTF" and ver == 2 and total == len(raw)
    jl = struct.unpack("<I", raw[12:16])[0]
    doc = json.loads(raw[20:20 + jl])
    off = 20 + jl + 8
    idx = np.frombuffer(raw[off:off + 24], "<u4").reshape(2, 3)
    pos = np.frombuffer(raw[off + 24:off + 24 + 60], "<f4").reshape(5, 3)
    assert np.array_equal(idx, f) and np.array_equal(pos, v) and doc["accessors"][1]["count"] == 5


def test_scheduler_mirror_matches_reference_fixture(golden_dir):
    from r3g.scheduler import FlowMatchEulerDiscreteScheduler
    z = np.load(os.path.join(golden_dir, "scheduler.npz"))
    sch = FlowMatchEulerDiscreteScheduler(num_train_timesteps=1000)
    for n in (1, 5, 50):
        sch.set_timesteps(sigmas=np.linspace(0, 1, n))
        assert np.array_equal(sch.timesteps.numpy(), z[f"timesteps_{n}"])
        assert np.array_equal(sch.sigmas.numpy(), z[f"sigmas_{n}"])
    sch.set_timesteps(sigmas=np.linspace(0, 1, 5))
    x = torch.from_numpy(z["euler_x"][0])
    for i, t in enumerate(sch.timesteps[:3]):
        x = sch.step(torch.from_numpy(z["euler_v"][i]), t, x).prev_sample
        assert np.array_equal(x.numpy(), z["euler_x"][i + 1])
    with pytest.raises(ValueError):
        sch.step(torch.zeros(1), 3, torch.zeros(1))


def test_image_processor_against_reference_when_available(golden_dir):
    """ImageProcessorV2 (preprocessors.py) bit for bit: the reference's image and mask tensors are stored as digests
    of their bytes (tests/golden/host_helpers.npz)."""
    from PIL import Image
    from make_golden import ellipse_rgba, sha256
    from r3g.preprocessors import ImageProcessorV2
    z = np.load(os.path.join(golden_dir, "host_helpers.npz"))
    a = ImageProcessorV2(512, 0.15)(Image.fromarray(ellipse_rgba(), "RGBA"))
    assert a["image"].shape == (1, 3, 512, 512) and a["mask"].shape == (1, 1, 512, 512)
    assert a["image"].dtype == a["mask"].dtype == torch.float32
    assert sha256(a["image"]) == z["imgproc_image_sha256"] and sha256(a["mask"]) == z["imgproc_mask_sha256"]


def test_stage3_twin_file_contract(tmp_path, monkeypatch):
    """The stage-3 twin's host helpers: config loading, name filter, output clearing (no GPU work here)."""
    sys.path.insert(0, os.path.join(ROOT, "stages", "2d_to_3d_models"))
    import importlib
    run = importlib.import_module("run")
    d = tmp_path / "out"
    (d / "old").mkdir(parents=True)
    (d / "old" / "x.glb").write_bytes(b"1")
    (d / "stale.txt").write_text("x")
    run.clear_output_directory(str(d))
    assert os.listdir(d) == []
    cfg = tmp_path / "c.yaml"
    cfg.write_text("num_inf_steps_hy: 50\noctree_resolution_hy: 256\nuse_banana: false\n")
    assert run.load_config(str(cfg))["octree_resolution_hy"] == 256


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU oracle port on the host cores) prints one JSON line with the contract's keys;
    under torchrun only rank 0 prints."""
    import json
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "objects/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("objects->mesh/sec") and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "objects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=60, cwd=ROOT, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_bench_dump_outputs_stay_within_64_mb(tmp_path):
    """`bench.py --dump-outputs`: float32 stays float32 and other dtypes become float64; small arrays are written whole,
    large ones as the same seeded sample of their rows, in order, on every call; 64 MB in all."""
    sys.path.insert(0, ROOT)
    import bench

    def rows(n, dtype):                 # row i holds i three times: a sampled row shows where it came from
        return np.repeat(np.arange(n, dtype=dtype)[:, None], 3, axis=1)
    arrays = {"v": rows(3_000_000, np.float32), "f": rows(6_000_000, np.int32), "small": torch.arange(10)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    out = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in arrays) <= 64e6
    assert out["v"].dtype == np.float32 and out["f"].dtype == np.float64 and out["small"].dtype == np.float64
    assert np.array_equal(out["small"], np.arange(10))
    for k in ("v", "f"):
        a = out[k]
        assert a.shape[1] == 3 and 0 < len(a) < len(arrays[k])
        assert (a == a[:, :1]).all() and (np.diff(a[:, 0]) > 0).all()
    for k in arrays:
        assert np.array_equal(out[k], np.load(tmp_path / "b" / f"{k}.npy"))


def test_conditioner_mirror_against_reference_when_available(golden_dir):
    """Row a2: DinoImageEncoder (conditioner.py:57-131) -- value-range shift, Resize(bilinear, antialias) + CenterCrop +
    Normalize, HF Dinov2Model, cls token kept; zeros as the unconditional embedding.  Same small seeded model in both;
    the reference's outputs are in tests/golden/host_helpers.npz."""
    sys.path.insert(0, os.path.join(ROOT, "3d-re-gen_b200"))
    from r3g.conditioner import DinoImageEncoder, SingleImageEncoder
    from make_golden import seeded_weights
    cfg = dict(hidden_size=32, num_hidden_layers=2, num_attention_heads=2, mlp_ratio=2, patch_size=14, image_size=56,
               use_swiglu_ffn=True, layerscale_value=1.0, qkv_bias=True, hidden_act="gelu", layer_norm_eps=1e-6)
    z = np.load(os.path.join(golden_dir, "host_helpers.npz"))
    mine = DinoImageEncoder(config=cfg, use_cls_token=True, image_size=56, device="cpu", dtype=torch.float32)
    mine.model.load_state_dict(seeded_weights({k: v.shape for k, v in mine.model.state_dict().items()}))
    g = torch.Generator().manual_seed(0)
    for i, shape in enumerate(((1, 3, 70, 90), (2, 3, 100, 64), (1, 3, 56, 56))):
        img = torch.rand(shape, generator=g) * 2 - 1
        a, b = mine(img), torch.from_numpy(z[f"dino_out{i}"])
        assert a.shape == b.shape == (shape[0], 17, 32)
        assert torch.allclose(a, b, atol=1e-5, rtol=1e-5), (a - b).abs().max()
    u = SingleImageEncoder(mine).unconditional_embedding(2)["main"]
    assert u.shape == (2, 17, 32) and not u.any() and torch.equal(u, torch.from_numpy(z["dino_uncond"]))


def test_near_surface_mask_against_reference_when_available(golden_dir):
    """extract_near_surface_volume_fn (volume_decoders.py:29-119): the point selection of the FlashVDM levels, against
    the reference's masks in tests/golden/host_helpers.npz."""
    from r3g.vae import extract_near_surface_volume_fn
    z = np.load(os.path.join(golden_dir, "host_helpers.npz"))
    torch.manual_seed(0)
    for n in (5, 9):
        x = torch.randn(n, n, n)
        x[torch.rand(n, n, n) < 0.25] = -10000.0
        for j, alpha in enumerate((0.0, 0.3, -0.2)):
            assert torch.equal(extract_near_surface_volume_fn(x, alpha), torch.from_numpy(z[f"near_surface_{n}_{j}"]))


def test_flashvdm_resolution_schedule():
    """volume_decoders.py:310-320: 256 -> [63, 126, 252]; below min_resolution a single level."""
    from r3g.vae import FlashVDMVolumeDecoding
    dec = FlashVDMVolumeDecoding()
    with pytest.raises(ValueError):
        FlashVDMVolumeDecoding("nope")
    with pytest.raises(NotImplementedError):
        FlashVDMVolumeDecoding("merge")
    assert dec._topk(3072) == 1024 and dec._topk(512) == 256 and dec._topk(48) == 16
