"""CPU: pin the oracle restatements (oracle/hy3d_ref.py, oracle/vggt_ref.py) and the VGGT head mirrors against
fixtures generated from the REFERENCE's own modules (oracle/make_golden.py, run where the reference checkout exists)."""
import os

import numpy as np
import torch

import hy3d_ref as R


def load(golden_dir, name):
    z = np.load(os.path.join(golden_dir, name))
    sd = {k[2:]: torch.from_numpy(z[k].astype(np.float32)) for k in z.files if k.startswith("w:")}
    return z, sd


def test_dit_restatement_matches_reference_fixture(golden_dir):
    z, sd = load(golden_dir, "dit_mini.npz")
    taps = []
    y = R.dit_forward(sd, torch.from_numpy(z["x"]), torch.from_numpy(z["t"]), torch.from_numpy(z["cond"]),
                      int(z["cfg_heads"]), int(z["cfg_depth"]), int(z["cfg_depth_single"]), taps=taps)
    for i, tp in enumerate(taps):
        np.testing.assert_allclose(tp.numpy(), z[f"tap{i}"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(y.numpy(), z["y"], rtol=0, atol=2e-5)


def test_timestep_embedding_fp16_bit_exact(golden_dir):
    z, _ = load(golden_dir, "dit_mini.npz")
    out = R.timestep_embedding(torch.from_numpy(z["temb_t"]), 256, max_period=1000.0)
    assert out.dtype == torch.float16
    assert np.array_equal(out.numpy(), z["temb_out"])


def test_vae_and_geo_decoder_match_reference_fixture(golden_dir):
    z, sd = load(golden_dir, "vae_mini.npz")
    heads, layers, Rr = int(z["cfg_heads"]), int(z["cfg_layers"]), int(z["cfg_R"])
    taps = []
    lat = R.vae_forward(sd, torch.from_numpy(z["z"]), heads, layers, taps=taps)
    for i, tp in enumerate(taps):
        np.testing.assert_allclose(tp.numpy(), z[f"tap{i}"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(lat.numpy(), z["latents"], rtol=0, atol=2e-5)
    assert np.array_equal(R.dense_grid_points([-1.01] * 3 + [1.01] * 3, Rr), z["xyz"])
    q = torch.from_numpy(z["xyz"]).half().float()
    np.testing.assert_allclose(R.fourier_embed(q, 8, False).numpy(), z["fourier"], rtol=0, atol=1e-6)
    grid = R.vanilla_volume_decode(sd, torch.from_numpy(z["latents"]), heads, Rr, num_chunks=100)
    np.testing.assert_allclose(grid.numpy(), z["grid"], rtol=0, atol=3e-5)


def test_scheduler_matches_reference_fixture(golden_dir):
    z = np.load(os.path.join(golden_dir, "scheduler.npz"))
    for n in (1, 5, 50):
        ts, sig = R.flow_euler_sigmas(n)
        assert np.array_equal(ts.numpy(), z[f"timesteps_{n}"])
        assert np.array_equal(sig.numpy(), z[f"sigmas_{n}"])
    _, sig = R.flow_euler_sigmas(5)
    x = torch.from_numpy(z["euler_x"][0])
    for i in range(3):
        x = R.flow_euler_step(x, torch.from_numpy(z["euler_v"][i]), sig[i], sig[i + 1])
        assert x.dtype == torch.float16
        assert np.array_equal(x.numpy(), z["euler_x"][i + 1])
    # the reference quirk: the 50th model call has d_sigma = 0 (sigmas[49] == sigmas[50] == 1)
    _, s50 = R.flow_euler_sigmas(50)
    assert float(s50[49]) == 1.0 and float(s50[50]) == 1.0


def test_unproject_matches_reference_fixture(golden_dir):
    z = np.load(os.path.join(golden_dir, "unproject.npz"))
    pts = R.unproject_depth_map_to_point_map(z["depth"], z["extrinsic"], z["intrinsic"])
    assert pts.dtype == np.float64
    np.testing.assert_allclose(pts, z["points"], rtol=0, atol=1e-12)


def test_vggt_restatement_matches_reference_fixture(golden_dir):
    import vggt_ref as V
    z = np.load(os.path.join(golden_dir, "vggt_mini.npz"))
    sd = {k[len("w:agg."):]: torch.from_numpy(z[k].astype(np.float32)) for k in z.files if k.startswith("w:agg.")}
    outs = V.aggregator(sd, torch.from_numpy(z["agg_images"]), depth=2, heads=2)
    for i, o in enumerate(outs):
        np.testing.assert_allclose(o.numpy(), z[f"agg_out{i}"], rtol=0, atol=3e-5)
    vsd = {k[len("w:vit."):]: torch.from_numpy(z[k].astype(np.float32)) for k in z.files if k.startswith("w:vit.")}
    for tag in ("native", "interp"):
        y = V.dino_patch_tokens(vsd, "", torch.from_numpy(z[f"vit_x_{tag}"]), 2, 2, 14, 4)
        np.testing.assert_allclose(y.numpy(), z[f"vit_y_{tag}"], rtol=0, atol=3e-5)


def test_vggt_heads_mirror_matches_reference_modules_live(golden_dir):
    """The torch-operator mirrors of CameraHead / DPTHead / pose utilities against the reference modules' outputs
    (CPU, fp32) on seeded weights of the reference heads' layout (tests/golden/vggt_heads_mini.npz)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "3d-re-gen_b200"))
    from make_golden import seeded_weights, stored_layout
    from r3g import vggt_heads as M
    z = np.load(os.path.join(golden_dir, "vggt_heads_mini.npz"))
    sd = seeded_weights(stored_layout(z))
    C, S, H, W = 128, 2, 56, 70
    ph, pw = H // 14, W // 14
    torch.manual_seed(0)
    toks = [torch.randn(1, S, 5 + ph * pw, C) for _ in range(4)]
    imgs = torch.rand(1, S, 3, H, W)
    mine = M.CameraHead(sd, trunk_depth=2, num_heads=2, device="cpu")(toks)
    assert len(mine) == 4
    for i, a in enumerate(mine):
        np.testing.assert_allclose(a.numpy(), z[f"pose{i}"], rtol=0, atol=2e-5)
    e1, k1 = M.pose_encoding_to_extri_intri(mine[-1], (H, W))
    np.testing.assert_allclose(e1.numpy(), z["extrinsic"], atol=1e-5)
    np.testing.assert_allclose(k1.numpy(), z["intrinsic"], rtol=1e-5)
    md, mc = M.DPTHead(sd, intermediate_layer_idx=(0, 1, 2, 3), device="cpu")(toks, imgs, 5)
    np.testing.assert_allclose(md.numpy(), z["depth"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(mc.numpy(), z["conf"], rtol=1e-4, atol=1e-5)
