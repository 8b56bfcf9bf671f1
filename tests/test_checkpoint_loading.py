"""CPU: `Hunyuan3DDiTFlowMatchingPipeline.from_pretrained` on a fabricated checkpoint in the reference's layout
($HY3DGEN_MODELS/<repo>/<subfolder>/config.yaml + model.fp16.safetensors with `model.` / `vae.` / `conditioner.` key
prefixes, pipelines.py:140-232).  The DiT / VAE key names and shapes are the state-dict layout of the reference's own
classes at small sizes (tests/golden/checkpoint_layout.npz, oracle/make_golden.py) filled with seeded values, so the
test pins the state-dict key mapping, the linear1 row permutation and the modulation packing -- the part of the drop-in
that no GPU test can reach because no real checkpoint is reachable here."""
import os
import sys

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-re-gen_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def test_from_pretrained_maps_a_reference_layout_checkpoint(tmp_path, monkeypatch, golden_dir):
    import safetensors.torch
    from make_golden import seeded_weights, stored_layout
    from transformers import Dinov2Config, Dinov2Model
    H, Mh, nh = 128, 512, 2
    dit_p = dict(in_channels=64, context_in_dim=96, hidden_size=H, mlp_ratio=4.0, num_heads=nh, depth=2,
                 depth_single_blocks=3, axes_dim=[64], theta=10000, qkv_bias=True, time_factor=1000, guidance_embed=False)
    vae_p = dict(num_latents=48, embed_dim=64, width=128, heads=2, num_decoder_layers=2, num_freqs=8, include_pi=False,
                 qkv_bias=False, qk_norm=True, scale_factor=0.999)
    dino_p = dict(hidden_size=96, num_hidden_layers=2, num_attention_heads=2, mlp_ratio=2, patch_size=14, image_size=56,
                  use_swiglu_ffn=True, layerscale_value=1.0, qkv_bias=True, hidden_act="gelu", layer_norm_eps=1e-6)
    layout = stored_layout(np.load(os.path.join(golden_dir, "checkpoint_layout.npz")))
    flat = {k: v.half() for k, v in seeded_weights(layout).items()}
    torch.manual_seed(0)
    dino = Dinov2Model(Dinov2Config(**dino_p))
    for k, v in dino.state_dict().items():
        flat["conditioner.main_image_encoder.model." + k] = v.half().contiguous()
    base = tmp_path / "tencent" / "Hunyuan3D-2" / "hunyuan3d-dit-v2-0"
    base.mkdir(parents=True)
    safetensors.torch.save_file(flat, str(base / "model.fp16.safetensors"))
    cfg = {"model": {"target": "hy3dgen.shapegen.models.Hunyuan3DDiT", "params": dit_p},
           "vae": {"target": "hy3dgen.shapegen.models.ShapeVAE", "params": vae_p},
           "conditioner": {"target": "hy3dgen.shapegen.models.SingleImageEncoder",
                           "params": {"main_image_encoder": {"type": "DinoImageEncoder",
                                                             "kwargs": {"config": dino_p, "use_cls_token": True,
                                                                        "image_size": 56}}}},
           "scheduler": {"target": "hy3dgen.shapegen.schedulers.FlowMatchEulerDiscreteScheduler",
                         "params": {"num_train_timesteps": 1000}},
           "image_processor": {"target": "hy3dgen.shapegen.preprocessors.ImageProcessorV2",
                               "params": {"size": 512, "border_ratio": 0.15}}}
    (base / "config.yaml").write_text(yaml.safe_dump(cfg))
    monkeypatch.setenv("HY3DGEN_MODELS", str(tmp_path))
    from r3g.pipelines import Hunyuan3DDiTFlowMatchingPipeline
    pipe = Hunyuan3DDiTFlowMatchingPipeline.from_pretrained("tencent/Hunyuan3D-2", device="cpu")
    w, sd = pipe.model.w, {k[len("model."):]: v for k, v in flat.items() if k.startswith("model.")}
    # plain tensors keep their keys
    for k in ("latent_in.weight", "cond_in.bias", "double_blocks.1.img_attn.qkv.weight", "double_blocks.0.txt_mlp.2.bias",
              "single_blocks.2.linear2.weight", "single_blocks.0.norm.key_norm.scale", "final_layer.linear.weight"):
        assert torch.equal(w[k], sd[k]), k
    # linear1 rows (q, k, v, mlp) -> (q, mlp, k, v)
    l1, ref1 = w["single_blocks.1.linear1.weight"], sd["single_blocks.1.linear1.weight"]
    assert torch.equal(l1[:H], ref1[:H]) and torch.equal(l1[H:H + Mh], ref1[3 * H:]) and torch.equal(l1[H + Mh:], ref1[H:3 * H])
    b1, refb = w["single_blocks.1.linear1.bias"], sd["single_blocks.1.linear1.bias"]
    assert torch.equal(b1[H:H + Mh], refb[3 * H:])
    # every Modulation.lin packed into one matrix, at the recorded offsets
    for key, name in (((1, "img"), "double_blocks.1.img_mod.lin"), ((0, "txt"), "double_blocks.0.txt_mod.lin"),
                      (("s", 2), "single_blocks.2.modulation.lin"), ("final", "final_layer.adaLN_modulation.1")):
        off, n = pipe.model.mod_off[key]
        assert torch.equal(w["mod.weight"][off:off + n], sd[name + ".weight"]), name
        assert torch.equal(w["mod.bias"][off:off + n], sd[name + ".bias"]), name
    assert pipe.model.mod_total == 2 * 2 * 6 * H + 3 * 3 * H + 2 * H
    # VAE / geo-decoder / conditioner
    assert torch.equal(pipe.vae.w["post_kl.weight"], flat["vae.post_kl.weight"])
    assert torch.equal(pipe.vae.w["transformer.resblocks.1.attn.c_qkv.weight"],
                       flat["vae.transformer.resblocks.1.attn.c_qkv.weight"])
    assert torch.equal(pipe.vae.geo_decoder.w["c_kv.weight"], flat["vae.geo_decoder.cross_attn_decoder.attn.c_kv.weight"])
    assert torch.equal(pipe.vae.geo_decoder.w["query_proj.weight"][:, :51], flat["vae.geo_decoder.query_proj.weight"])
    assert not pipe.vae.geo_decoder.w["query_proj.weight"][:, 51:].any()      # K padded 51 -> 64 with zeros
    enc = pipe.conditioner.main_image_encoder.model
    assert torch.equal(enc.state_dict()["encoder.layer.1.mlp.weights_in.weight"],
                       dino.state_dict()["encoder.layer.1.mlp.weights_in.weight"].half())
    assert pipe.scheduler.config.num_train_timesteps == 1000 and pipe.image_processor.size == 512
    assert abs(pipe.vae.scale_factor - 0.999) < 1e-9 and pipe.vae.latent_shape == (48, 64)
