#!/usr/bin/env python
"""ORACLE -- test infrastructure only.

Generates tests/golden/*.npz by running the REFERENCE's own Python modules (imported from
/root/reference, see oracle/ref_import.py) on seeded inputs with seeded random weights.
Run in the build container only:  python oracle/make_golden.py
The reference ships no weights and no golden vectors of its own (SURVEY.md section 4), so these
fixtures are the pin: weights are the modules' default initialisation under torch.manual_seed,
rounded through fp16 (what a GPU run holds) and evaluated in fp32 on the CPU.
Where the weights or an output are too large to store, a fixture keeps the state-dict layout (filled by
seeded_weights) or a digest of the output's bytes; the tests import those helpers and the seeded test
inputs from here, so they run without the reference.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_import  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")


def fp16_round_(module, buffers=True):
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(p.half().float())
        for b in module.buffers() if buffers else ():
            if b.is_floating_point():
                b.copy_(b.half().float())


def sd_np(module, prefix=""):
    return {"w:" + prefix + k: v.detach().half().numpy() for k, v in module.state_dict().items()}


def layout_np(module, prefix=""):
    """The state-dict layout of a module (key -> shape) as "shape:<prefix><key>" entries of a fixture."""
    return {"shape:" + prefix + k: np.array(v.shape, np.int64) for k, v in module.state_dict().items()}


def stored_layout(z, prefix=""):
    """{key: shape} of the "shape:<prefix>..." entries of a fixture (or of a dict) written with layout_np."""
    return {k[len("shape:"):]: tuple(int(s) for s in z[k]) for k in z if k.startswith("shape:" + prefix)}


def seeded_weights(shapes, seed=0):
    """float32 tensors for a {key: shape} layout, drawn in sorted key order from one seeded stream, so that a fixture
    only needs to store the layout: matrices and kernels U(-1, 1) / sqrt(fan_in), 1-d norm scales (`*weight`,
    `*scale`) 1 + 0.2 N(0, 1), everything else (biases, LayerScale gammas, tokens) 0.2 N(0, 1)."""
    rng = np.random.default_rng(seed)
    out = {}
    for k in sorted(shapes):
        shape = tuple(shapes[k])
        if len(shape) >= 2:
            v = rng.uniform(-1.0, 1.0, shape) / np.sqrt(np.prod(shape[1:]))
        elif k.endswith(("weight", "scale")):
            v = 1.0 + 0.2 * rng.standard_normal(shape)
        else:
            v = 0.2 * rng.standard_normal(shape)
        out[k] = torch.from_numpy(v.astype(np.float32))
    return out


def sha256(t):
    """Digest of a tensor's or array's bytes: pins a large output that must match bit for bit."""
    import hashlib
    a = t.numpy() if isinstance(t, torch.Tensor) else t
    return np.str_(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


def ellipse_rgba():
    """300x420 RGBA: seeded noise RGB inside an elliptical alpha mask (the image processor's test input)."""
    rng = np.random.default_rng(0)
    rgba = np.zeros((300, 420, 4), np.uint8)
    rgba[..., :3] = rng.integers(0, 256, (300, 420, 3))
    yy, xx = np.mgrid[0:300, 0:420]
    rgba[..., 3] = ((((xx - 200) / 120) ** 2 + ((yy - 160) / 90) ** 2) <= 1) * 255
    return rgba


def loader_pngs(directory):
    """Three seeded PNGs (landscape RGB, portrait RGBA, square RGB) for the square image loader."""
    from PIL import Image
    rng = np.random.default_rng(9)
    paths = []
    for i, (w, h, mode) in enumerate(((150, 100, "RGB"), (64, 97, "RGBA"), (80, 80, "RGB"))):
        arr = rng.integers(0, 256, (h, w, 4 if mode == "RGBA" else 3)).astype(np.uint8)
        path = os.path.join(str(directory), f"im{i}.png")
        Image.fromarray(arr, mode).save(path)
        paths.append(path)
    return paths


def golden_dit():
    m = ref_import.hunyuan_dit()
    cfg = dict(in_channels=64, context_in_dim=96, hidden_size=128, num_heads=2, depth=2, depth_single_blocks=2,
               axes_dim=[64])
    torch.manual_seed(0)
    model = m.Hunyuan3DDiT(**cfg).eval()
    # the default init leaves the RMSNorm scales at 1 and modulation small; perturb so every term matters
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("norm.scale"):
                p.copy_(1 + 0.25 * torch.randn_like(p))
            if ".bias" in n:
                p.copy_(0.1 * torch.randn_like(p))
    fp16_round_(model)
    B, L, Lc = 2, 40, 24
    x = torch.randn(B, L, 64).half().float()
    cond = torch.randn(B, Lc, 96).half().float()
    t = torch.tensor([0.3469, 0.3469]).half().float()
    taps = []
    hooks = [blk.register_forward_hook(lambda mod, i, o: taps.append(
        torch.cat((o[1], o[0]), 1) if isinstance(o, tuple) else o)) for blk in
        list(model.double_blocks) + list(model.single_blocks)]
    with torch.no_grad():
        y = model(x, t, {"main": cond})
    for h in hooks:
        h.remove()
    d = sd_np(model)
    d.update(x=x.numpy(), t=t.numpy(), cond=cond.numpy(), y=y.numpy(), cfg_heads=np.int64(2), cfg_depth=np.int64(2),
             cfg_depth_single=np.int64(2))
    for i, tp in enumerate(taps):
        d[f"tap{i}"] = tp.numpy()
    # timestep embedding in fp16, exactly as the GPU pipeline calls it (pipelines.py:747-749)
    t16 = torch.tensor([0.0, 0.0204, 0.5102, 1.0], dtype=torch.float16)
    d["temb_t"] = t16.numpy()
    d["temb_out"] = m.timestep_embedding(t16, 256, 1000.0).numpy()  # positional, like hunyuan3ddit.py:390
    np.savez_compressed(os.path.join(OUT, "dit_mini.npz"), **d)
    print("dit_mini: y", tuple(y.shape), "taps", len(taps))


def golden_vae():
    ab, ap, vd = ref_import.hunyuan_autoencoders()
    width, heads, layers, n_lat, embed = 128, 2, 2, 48, 64
    torch.manual_seed(1)
    fe = ab.FourierEmbedder(num_freqs=8, include_pi=False)
    post_kl = torch.nn.Linear(embed, width)
    tr = ab.Transformer(n_ctx=n_lat, width=width, layers=layers, heads=heads, qkv_bias=False, qk_norm=True)
    geo = ab.CrossAttentionDecoder(fourier_embedder=fe, out_channels=1, num_latents=n_lat, mlp_expand_ratio=4,
                                   downsample_ratio=1, enable_ln_post=True, width=width, heads=heads,
                                   qkv_bias=False, qk_norm=True, label_type="binary")
    with torch.no_grad():
        for mod in (tr, geo):
            for n, p in mod.named_parameters():
                if "norm" in n or "ln_" in n:
                    p.copy_((1.0 if n.endswith("weight") else 0.0) + 0.2 * torch.randn_like(p))
    for mod in (post_kl, tr, geo):
        mod.eval()
        fp16_round_(mod)
    z = torch.randn(1, n_lat, embed).half().float()
    taps = []
    hooks = [blk.register_forward_hook(lambda mod, i, o: taps.append(o)) for blk in tr.resblocks]
    with torch.no_grad():
        lat = tr(post_kl(z))
        # VanillaVolumeDecoder casts the queries to latents.dtype: run it in fp32 but with fp16-quantised
        # coordinates, the values the fp16 pipeline sees (volume_decoders.py:168)
        R = 8
        xyz, grid_size, _ = vd.generate_dense_grid_points(np.array([-1.01] * 3), np.array([1.01] * 3), R, "ij")
        q = torch.from_numpy(xyz).half().float().reshape(1, -1, 3)
        logits = geo(queries=q, latents=lat)
        grid = logits.view(1, *grid_size).float()
        emb = fe(q)
    for h in hooks:
        h.remove()
    d = {}
    d.update(sd_np(post_kl, "post_kl."))
    d.update(sd_np(tr, "transformer."))
    d.update(sd_np(geo, "geo_decoder."))
    d = {k: v for k, v in d.items() if "fourier_embedder" not in k}
    d.update(z=z.numpy(), latents=lat.numpy(), grid=grid.numpy(), xyz=xyz.reshape(-1, 3), fourier=emb.numpy()[0],
             cfg_heads=np.int64(heads), cfg_layers=np.int64(layers), cfg_R=np.int64(R))
    for i, tp in enumerate(taps):
        d[f"tap{i}"] = tp.numpy()
    np.savez_compressed(os.path.join(OUT, "vae_mini.npz"), **d)
    print("vae_mini: grid", tuple(grid.shape), "range", float(grid.min()), float(grid.max()))


def golden_flashvdm():
    """FlashVDMVolumeDecoding (volume_decoders.py:280-435) with FlashVDMCrossAttentionProcessor (attention_processors.py:
    35-79) on a mini geo-decoder, two levels (31 -> 62): the reference CLASS is run in fp32.  Its level-0 queries are
    `xyz.to(dtype)`; the fp16 pipeline therefore sees fp16-quantised coordinates there, so generate_dense_grid_points is
    wrapped to hand the class fp16-representable float32 coordinates (levels >= 1 build float32 queries in both)."""
    ab, ap, vd = ref_import.hunyuan_autoencoders()
    width, heads, n_lat = 128, 2, 48
    torch.manual_seed(4)
    fe = ab.FourierEmbedder(num_freqs=8, include_pi=False)
    geo = ab.CrossAttentionDecoder(fourier_embedder=fe, out_channels=1, num_latents=n_lat, mlp_expand_ratio=4,
                                   downsample_ratio=1, enable_ln_post=True, width=width, heads=heads,
                                   qkv_bias=False, qk_norm=True, label_type="binary")
    with torch.no_grad():
        for n, p in geo.named_parameters():
            if "norm" in n or "ln_" in n:
                p.copy_((1.0 if n.endswith("weight") else 0.0) + 0.2 * torch.randn_like(p))
        geo.output_proj.weight.mul_(6.0)       # logits of a few units: the |logit| < 0.95 band is a fraction of the volume
    geo.eval()
    fp16_round_(geo)
    lat = (torch.randn(1, n_lat, width) * 0.7).half().float()
    orig = vd.generate_dense_grid_points

    def fp16_points(*a, **kw):
        xyz, gs, ln = orig(*a, **kw)
        return xyz.astype(np.float16).astype(np.float32), gs, ln
    vd.generate_dense_grid_points = fp16_points
    try:
        dec = vd.FlashVDMVolumeDecoding(topk_mode="mean")
        with torch.no_grad():
            grid = dec(lat, geo, bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=64, min_resolution=31,
                       mini_grid_num=4, enable_pbar=False)
            grid0 = dec(lat, geo, bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=31, min_resolution=31,
                        mini_grid_num=4, enable_pbar=False)
    finally:
        vd.generate_dense_grid_points = orig
    d = sd_np(geo, "geo_decoder.")
    d = {k: v for k, v in d.items() if "fourier_embedder" not in k}
    g = grid.numpy()
    d.update(latents=lat.numpy(), grid=g, grid_level0=grid0.numpy(), cfg_heads=np.int64(heads),
             cfg_octree=np.int64(64), cfg_min_resolution=np.int64(31), cfg_num_chunks=np.int64(3000))
    np.savez_compressed(os.path.join(OUT, "flashvdm_mini.npz"), **d)
    print("flashvdm_mini: grid", g.shape, "finite", float(np.isfinite(g).mean()), "range", float(np.nanmin(g)),
          float(np.nanmax(g)), "level0", grid0.shape)


def golden_scheduler():
    s = ref_import.hunyuan_scheduler()
    sch = s.FlowMatchEulerDiscreteScheduler(num_train_timesteps=1000)
    d = {}
    for n in (1, 5, 50):
        sch.set_timesteps(sigmas=np.linspace(0, 1, n))
        d[f"timesteps_{n}"] = sch.timesteps.numpy()
        d[f"sigmas_{n}"] = sch.sigmas.numpy()
    # three Euler steps on an fp16 sample, the dtype flow of pipelines.py:755-756
    torch.manual_seed(2)
    sch.set_timesteps(sigmas=np.linspace(0, 1, 5))
    x = torch.randn(1, 16, 64).half()
    xs = [x.numpy()]
    vs = []
    for t in sch.timesteps[:3]:
        v = torch.randn(1, 16, 64).half()
        x = sch.step(v, t, x).prev_sample
        vs.append(v.numpy())
        xs.append(x.numpy())
    d["euler_x"] = np.stack(xs)
    d["euler_v"] = np.stack(vs)
    np.savez_compressed(os.path.join(OUT, "scheduler.npz"), **d)
    print("scheduler: ok", d["sigmas_5"])


def golden_unproject():
    ref_import.vggt_package()
    from vggt.utils.geometry import unproject_depth_map_to_point_map
    rng = np.random.default_rng(3)
    S, H, W = 3, 13, 18
    depth = (0.5 + rng.random((S, H, W, 1))).astype(np.float32)
    depth[0, 0, 0, 0] = 0.0
    ang = rng.normal(size=(S, 3))
    E = np.zeros((S, 3, 4), np.float32)
    for s in range(S):
        a, b, c = ang[s]
        Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
        Ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
        Rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
        E[s, :, :3] = (Rz @ Ry @ Rx).astype(np.float32)
        E[s, :, 3] = rng.normal(size=3).astype(np.float32)
    K = np.zeros((S, 3, 3), np.float32)
    K[:, 0, 0] = 300 + 50 * rng.random(S)
    K[:, 1, 1] = 310 + 50 * rng.random(S)
    K[:, 0, 2] = W / 2
    K[:, 1, 2] = H / 2
    K[:, 2, 2] = 1
    pts = unproject_depth_map_to_point_map(depth, E, K)
    assert pts.dtype == np.float64
    np.savez_compressed(os.path.join(OUT, "unproject.npz"), depth=depth, extrinsic=E, intrinsic=K, points=pts)
    print("unproject:", pts.shape, pts.dtype)


def golden_vggt():
    ref_import.vggt_package()
    from vggt.models.aggregator import Aggregator
    from vggt.layers.vision_transformer import DinoVisionTransformer
    from vggt.layers.block import Block
    torch.manual_seed(4)
    agg = Aggregator(img_size=56, patch_size=14, embed_dim=128, depth=2, num_heads=2, patch_embed="conv",
                     qk_norm=True, rope_freq=100, init_values=0.01).eval()
    with torch.no_grad():
        for n, prm in agg.named_parameters():
            if "gamma" in n:
                prm.copy_(0.5 + 0.2 * torch.randn_like(prm))      # LayerScale that matters
            elif "norm" in n:
                prm.copy_((1.0 if n.endswith("weight") else 0.0) + 0.2 * torch.randn_like(prm))
            elif n in ("camera_token", "register_token"):
                prm.copy_(0.5 * torch.randn_like(prm))
            elif n.endswith("bias"):
                prm.copy_(0.1 * torch.randn_like(prm))
    fp16_round_(agg, buffers=False)  # the ImageNet mean/std buffers are constants, not checkpoint weights
    imgs = torch.rand(1, 2, 3, 56, 70)
    with torch.no_grad():
        outs, psi = agg(imgs)
    d = sd_np(agg, "agg.")
    d.update(agg_images=imgs.numpy(), agg_psi=np.int64(psi))
    for i, o in enumerate(outs):
        d[f"agg_out{i}"] = o.numpy()
    torch.manual_seed(5)
    vit = DinoVisionTransformer(img_size=56, patch_size=14, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4,
                                num_register_tokens=4, init_values=1.0, block_fn=Block, interpolate_antialias=True,
                                interpolate_offset=0.0, block_chunks=0).eval()
    with torch.no_grad():
        for n, prm in vit.named_parameters():
            if "gamma" in n:
                prm.copy_(0.5 + 0.2 * torch.randn_like(prm))
            elif n in ("cls_token", "register_tokens", "pos_embed"):
                prm.copy_(0.3 * torch.randn_like(prm))
            elif n.endswith("bias"):
                prm.copy_(0.1 * torch.randn_like(prm))
    fp16_round_(vit)
    for tag, shape in (("native", (2, 3, 56, 56)), ("interp", (2, 3, 70, 56))):
        x = torch.randn(*shape)
        with torch.no_grad():
            y = vit.forward_features(x)["x_norm_patchtokens"]
        d[f"vit_x_{tag}"], d[f"vit_y_{tag}"] = x.numpy(), y.numpy()
    d.update(sd_np(vit, "vit."))
    np.savez_compressed(os.path.join(OUT, "vggt_mini.npz"), **d)
    print("vggt_mini: outs", len(outs), tuple(outs[0].shape))


def golden_checkpoint_layout():
    """State-dict layout of a `model.fp16.safetensors` (pipelines.py:140-232) at the small sizes of
    tests/test_checkpoint_loading.py: the reference's Hunyuan3DDiT ("model."), ShapeVAE transformer and geo-decoder
    ("vae.").  The test fills it with seeded_weights."""
    m = ref_import.hunyuan_dit()
    ab, _, _ = ref_import.hunyuan_autoencoders()
    dit = m.Hunyuan3DDiT(in_channels=64, context_in_dim=96, hidden_size=128, mlp_ratio=4.0, num_heads=2, depth=2,
                         depth_single_blocks=3, axes_dim=[64], theta=10000, qkv_bias=True, time_factor=1000,
                         guidance_embed=False)
    tr = ab.Transformer(n_ctx=48, width=128, layers=2, heads=2, qkv_bias=False, qk_norm=True)
    geo = ab.CrossAttentionDecoder(out_channels=1, num_latents=48, mlp_expand_ratio=4, downsample_ratio=1,
                                   enable_ln_post=True, fourier_embedder=ab.FourierEmbedder(num_freqs=8, include_pi=False),
                                   width=128, heads=2, qkv_bias=False, qk_norm=True, label_type="binary")
    d = layout_np(dit, "model.")
    d.update(layout_np(torch.nn.Linear(64, 128), "vae.post_kl."))
    d.update(layout_np(tr, "vae.transformer."))
    d.update(layout_np(geo, "vae.geo_decoder."))
    np.savez_compressed(os.path.join(OUT, "checkpoint_layout.npz"), **d)
    print("checkpoint_layout:", len(d), "tensors")


def golden_vggt_heads():
    """CameraHead / DPTHead (vggt/heads/camera_head.py, dpt_head.py) and pose_encoding_to_extri_intri (pose_enc.py) in
    fp32 on the CPU: seeded_weights of the heads' layout, tokens and images from torch.manual_seed(0)."""
    ref_import.vggt_package()
    from vggt.heads.camera_head import CameraHead
    from vggt.heads.dpt_head import DPTHead
    from vggt.utils.pose_enc import pose_encoding_to_extri_intri
    C, S, H, W = 128, 2, 56, 70
    torch.manual_seed(0)
    toks = [torch.randn(1, S, 5 + (H // 14) * (W // 14), C) for _ in range(4)]
    imgs = torch.rand(1, S, 3, H, W)
    cam = CameraHead(dim_in=C, trunk_depth=2, num_heads=2).eval()
    dpt = DPTHead(dim_in=C, output_dim=2, activation="exp", conf_activation="expp1", features=32,
                  out_channels=[16, 32, 64, 64], intermediate_layer_idx=[0, 1, 2, 3]).eval()
    d = layout_np(cam, "camera_head.")
    d.update(layout_np(dpt, "depth_head."))
    w = seeded_weights(stored_layout(d))
    for prefix, mod in (("camera_head.", cam), ("depth_head.", dpt)):
        mod.load_state_dict({k[len(prefix):]: v for k, v in w.items() if k.startswith(prefix)})
    with torch.no_grad():
        poses = cam(toks)
        depth, conf = dpt(toks, images=imgs, patch_start_idx=5)
    extrinsic, intrinsic = pose_encoding_to_extri_intri(poses[-1], (H, W))
    for i, p in enumerate(poses):
        d[f"pose{i}"] = p.numpy()
    d.update(extrinsic=extrinsic.numpy(), intrinsic=intrinsic.numpy(), depth=depth.numpy(), conf=conf.numpy())
    np.savez_compressed(os.path.join(OUT, "vggt_heads_mini.npz"), **d)
    print("vggt_heads_mini: depth", tuple(depth.shape), "range", float(depth.min()), float(depth.max()))


def golden_host_helpers():
    """Host-side helpers of the pipeline and the stage scripts, on the inputs of tests/test_host_logic.py and
    tests/test_stage4_tail.py: ImageProcessorV2 (preprocessors.py), DinoImageEncoder (conditioner.py:57-131) with
    seeded_weights, extract_near_surface_volume_fn (volume_decoders.py:29-119), vggt/utils/helper.py and
    load_and_preprocess_images_square (vggt/utils/load_fn.py:13-94).  The two image outputs that must match bit for
    bit are stored as digests of their bytes."""
    import tempfile
    import warnings
    from PIL import Image
    d = {}
    out = ref_import.hunyuan_preprocessors().ImageProcessorV2(size=512, border_ratio=0.15)(
        Image.fromarray(ellipse_rgba(), "RGBA"))
    d["imgproc_image_sha256"], d["imgproc_mask_sha256"] = sha256(out["image"]), sha256(out["mask"])

    cfg = dict(hidden_size=32, num_hidden_layers=2, num_attention_heads=2, mlp_ratio=2, patch_size=14, image_size=56,
               use_swiglu_ffn=True, layerscale_value=1.0, qkv_bias=True, hidden_act="gelu", layer_norm_eps=1e-6)
    enc = ref_import.hunyuan_conditioner().DinoImageEncoder(config=cfg, use_cls_token=True, image_size=56)
    enc.model.load_state_dict(seeded_weights({k: v.shape for k, v in enc.model.state_dict().items()}))
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for i, shape in enumerate(((1, 3, 70, 90), (2, 3, 100, 64), (1, 3, 56, 56))):
            d[f"dino_out{i}"] = enc(torch.rand(shape, generator=g) * 2 - 1).numpy()
    d["dino_uncond"] = enc.unconditional_embedding(2).numpy()

    _, _, vd = ref_import.hunyuan_autoencoders()
    torch.manual_seed(0)
    for n in (5, 9):
        x = torch.randn(n, n, n)
        x[torch.rand(n, n, n) < 0.25] = -10000.0
        for j, alpha in enumerate((0.0, 0.3, -0.2)):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                d[f"near_surface_{n}_{j}"] = vd.extract_near_surface_volume_fn(x.clone(), alpha).numpy()

    ref_import.vggt_package()
    from vggt.utils import helper
    from vggt.utils.load_fn import load_and_preprocess_images_square
    d["pixel_grid"] = helper.create_pixel_coordinate_grid(2, 5, 4)
    np.random.seed(7)
    d["limited_mask"] = helper.randomly_limit_trues(np.random.default_rng(3).random((2, 30, 30)) > 0.3, 100)
    with tempfile.TemporaryDirectory() as tmp:
        paths = loader_pngs(tmp)
        for tag, sel in (("3", paths), ("1", paths[:1])):
            img, xy = load_and_preprocess_images_square(sel, 256)
            d[f"loader{tag}_sha256"], d[f"loader{tag}_shape"], d[f"loader{tag}_coords"] = (
                sha256(img), np.array(img.shape, np.int64), xy.numpy())
    np.savez_compressed(os.path.join(OUT, "host_helpers.npz"), **d)
    print("host_helpers:", len(d), "arrays")


if __name__ == "__main__":
    assert ref_import.available(), "reference checkout not found"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    golden_dit()
    golden_vae()
    golden_flashvdm()
    golden_scheduler()
    golden_unproject()
    golden_vggt()
    golden_checkpoint_layout()
    golden_vggt_heads()
    golden_host_helpers()
