"""-m "not gpu": the drop-in boundary as the reference's own script reaches it (SURVEY.md §8b, §3.5).

tests/golden/init_models_calls.json records every call the reference's `init_models` (MOFA-Video-Traj/run_gradio.py:
90-159) makes on the names it imports, in order (oracle/make_goldens.py --init-models ran the function itself against
recording stand-ins).  The test replays those calls against this package: its `from models... import`,
`from pipeline.pipeline import` names resolve to mofa_video_b200/ (first on sys.path, INTEGRATION.md),
`CLIPVisionModelWithProjection` / `AutoencoderKLTemporalDecoder` (transformers / diffusers loaders, absent here) are
stand-ins that read the same checkpoint folders, and the checkpoint tree is synthetic but laid out per the reference's
MOFA-Video-Hybrid/ckpt_tree.md:60-84.  Checks: the calls run unmodified; the VAE they hand over (an
AutoencoderKLTemporalDecoder-layout nn.Module) is re-hosted on the engine, so decode does not fall to eager PyTorch; a
clip through the resulting pipeline matches the oracle.  Also `FlowControlNet.from_unet` (models/controlnet_sdv.py:
572-628).  CPU backend = tests/ref_ops.py via models._base.default_backend."""
import importlib
import json
import os
import sys

import pytest
import torch
from safetensors.torch import save_file

import ref_ops
from mofa_video_b200 import synthetic
from mofa_video_b200.models import _base
from mofa_video_b200.models.autoencoder_kl_temporal_decoder import AutoencoderKLTemporalDecoder as VaeModule
from oracle import fixtures
from oracle import pipeline as opipe
from oracle import scheduler as osched

CALLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "init_models_calls.json")
PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "mofa_video_b200")


def _write_model(d, cfg, sd, name):
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump({"_class_name": "X", "_diffusers_version": "0.24.0",
                   **{k: (list(v) if isinstance(v, tuple) else v) for k, v in cfg.items()}}, f)
    save_file({k: v.contiguous() for k, v in sd.items()}, os.path.join(d, name))


class TinyClip(torch.nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.proj = torch.nn.Linear(3 * 8 * 8, dim)

    def forward(self, x):
        from types import SimpleNamespace
        return SimpleNamespace(image_embeds=self.proj(torch.nn.functional.adaptive_avg_pool2d(x, 8).flatten(1)))


VAE_CH = (64, 64, 128, 128)


def _checkpoint_tree(root, cfg):
    """ckpt_tree.md:60-84: stable-video-diffusion-img2vid-xt-1-1/{image_encoder,vae,unet,scheduler} + controlnet/."""
    svd = os.path.join(root, "ckpts", "stable-video-diffusion-img2vid-xt-1-1")
    ctrl = os.path.join(root, "ckpts", "controlnet")
    unet, adapter = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    _write_model(os.path.join(svd, "unet"), {**cfg, **{k: v for k, v in unet.config.__dict__.items() if k != "get"}},
                 {k: v.half() for k, v in unet.state_dict().items()}, "diffusion_pytorch_model.fp16.safetensors")
    _write_model(ctrl, {k: v for k, v in adapter.config.__dict__.items() if k != "get"},
                 {k: v.half() for k, v in adapter.state_dict().items()}, "diffusion_pytorch_model.safetensors")
    torch.manual_seed(5)
    vae = VaeModule(block_out_channels=VAE_CH).eval()
    with torch.no_grad():
        for p in vae.parameters():
            p.copy_(p.half().float())
    _write_model(os.path.join(svd, "vae"), {"block_out_channels": VAE_CH, "latent_channels": 4,
                                            "scaling_factor": 0.18215, "force_upcast": True},
                 {k: v.half() for k, v in vae.state_dict().items()}, "diffusion_pytorch_model.fp16.safetensors")
    clip = TinyClip(cfg["cross_attention_dim"]).eval()
    with torch.no_grad():
        for p in clip.parameters():
            p.copy_(p.half().float())
    os.makedirs(os.path.join(svd, "image_encoder"))
    save_file({k: v.half() for k, v in clip.state_dict().items()},
              os.path.join(svd, "image_encoder", "model.fp16.safetensors"))
    os.makedirs(os.path.join(svd, "scheduler"))
    with open(os.path.join(svd, "scheduler", "scheduler_config.json"), "w") as f:
        json.dump({"_class_name": "EulerDiscreteScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear",
                   "beta_start": 0.00085, "interpolation_type": "linear", "num_train_timesteps": 1000,
                   "prediction_type": "v_prediction", "sigma_max": 700.0, "sigma_min": 0.002, "steps_offset": 1,
                   "timestep_spacing": "leading", "timestep_type": "continuous", "use_karras_sigmas": True}, f)
    # CMP experiment folder the script hard-codes relative to the CWD (run_gradio.py:113-116)
    import yaml
    exp = os.path.join(root, "models", "cmp", "experiments", "semiauto_annot", "resnet50_vip+mpii_liteflow")
    os.makedirs(os.path.join(exp, "checkpoints"))
    with open(os.path.join(exp, "config.yaml"), "w") as f:
        yaml.safe_dump({"model": {"arch": "CMP", "module": {
            "arch": "CMP", "image_encoder": "resnet50", "sparse_encoder": "shallownet8x",
            "flow_decoder": "MotionDecoderSkipLayer", "skip_layer": True, "img_enc_dim": 256, "sparse_enc_dim": 16,
            "output_dim": 198, "decoder_combo": [1, 2, 4], "nbins": 99, "fmax": 50}}}, f)
    torch.save({"step": 42000, "state_dict": synthetic.cmp_state_dict()},
               os.path.join(exp, "checkpoints", "ckpt_iter_42000.pth.tar"))
    return svd, ctrl, unet, adapter, vae, clip


def _loader_stubs(cfg):
    """Stand-ins for the two third-party loaders the script imports at module level (run_gradio.py:23-25)."""
    from safetensors.torch import load_file

    class CLIPVisionModelWithProjection:
        @staticmethod
        def from_pretrained(path, subfolder=None, revision=None, variant=None):
            m = TinyClip(cfg["cross_attention_dim"]).eval()
            m.load_state_dict({k: v.float() for k, v in load_file(
                os.path.join(path, subfolder, f"model.{variant}.safetensors")).items()})
            return m

    class AutoencoderKLTemporalDecoder:
        @staticmethod
        def from_pretrained(path, subfolder=None, revision=None, variant=None):
            with open(os.path.join(path, subfolder, "config.json")) as f:
                c = {k: v for k, v in json.load(f).items() if not k.startswith("_")}
            m = VaeModule(block_out_channels=tuple(c["block_out_channels"]), latent_channels=c["latent_channels"],
                          scaling_factor=c["scaling_factor"], force_upcast=c["force_upcast"]).eval()
            m.load_state_dict({k: v.float() for k, v in load_file(
                os.path.join(path, subfolder, f"diffusion_pytorch_model.{variant}.safetensors")).items()})
            return m

    return CLIPVisionModelWithProjection, AutoencoderKLTemporalDecoder


def _replay_init_models(names, *args):
    """Run the recorded calls of the reference's init_models(*args); `names` answers its non-package imports."""
    with open(CALLS) as f:
        rec = json.load(f)
    argv = dict(zip(rec["args"], args))
    objs = {}

    def dec(v):
        if isinstance(v, list):
            return [dec(x) for x in v]
        if isinstance(v, dict):
            return objs[v["ref"]] if "ref" in v else argv[v["arg"]]
        return v

    for op in rec["ops"]:
        if op["op"] == "name":
            obj = names[op["name"]] if op["module"] is None else getattr(importlib.import_module(op["module"]), op["name"])
        else:
            fn = objs[op["obj"]] if op["method"] is None else getattr(objs[op["obj"]], op["method"])
            obj = fn(*dec(op["args"]), **{k: dec(v) for k, v in op["kwargs"].items()})
        objs[op["out"]] = obj
    return tuple(dec(rec["returns"]))


def test_reference_init_models_runs_unmodified_against_the_shim(tmp_path, monkeypatch):
    cfg = dict(fixtures.TINY_CONFIG)
    svd, ctrl, unet, adapter, vae, clip = _checkpoint_tree(str(tmp_path), cfg)
    clip_cls, vae_cls = _loader_stubs(cfg)
    names = {"CLIPVisionModelWithProjection": clip_cls, "AutoencoderKLTemporalDecoder": vae_cls}
    monkeypatch.chdir(tmp_path)
    monkeypatch.syspath_prepend(PKG)                      # INTEGRATION.md: mofa_video_b200/ first on sys.path
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k.split(".")[0] in ("models", "pipeline", "utils")}
    try:
        with _base.default_backend(ref_ops, "cpu"):
            # weight_dtype: the script passes torch.float16 on its CUDA device (run_gradio.py:223); the third-party CLIP /
            # VAE stand-ins stay fp32 on this CPU backend, the engine models accept only fp16 (checked below)
            pipeline, cmp = _replay_init_models(names, svd, ctrl, None, "cpu")
            assert type(pipeline).__module__ == "pipeline.pipeline" and type(pipeline.unet).__module__.startswith("models.")
            with pytest.raises(ValueError):
                pipeline.unet.to("cpu", dtype=torch.float32)
            assert pipeline.unet.to("cpu", dtype=torch.float16) is pipeline.unet
            # the VAE the script built (an nn.Module in the diffusers layout) now runs on the engine
            from mofa_video_b200.vae_engine import NativeTemporalDecoderVAE
            assert isinstance(pipeline.vae, NativeTemporalDecoderVAE) and hasattr(pipeline.vae, "decode_uint8")
            assert abs(pipeline.scheduler.config.sigma_max - 700.0) < 1e-6
            H, W, T = 128, 128, cfg["num_frames"]
            image, flow = fixtures.make_image(H, W), fixtures.make_flow(T, H, W)
            lat0 = torch.randn(1, T, 4, H // 8, W // 8, generator=torch.Generator().manual_seed(9))
            out = pipeline(image, image, flow, height=H, width=W, num_inference_steps=2, latents=lat0.clone(),
                           generator=torch.Generator().manual_seed(11), output_type="latent")
            ref = opipe.run_pipeline(vae, clip, unet, adapter, osched.EulerDiscreteScheduler(), image, image, flow,
                                     height=H, width=W, num_inference_steps=2, latents=lat0.clone(),
                                     generator=torch.Generator().manual_seed(11), output_type="latent")
            err = ((out.frames.float() - ref).abs().max() / ref.abs().max()).item()
            assert err < 1.5e-2, err
            frames = pipeline(image, image, flow, height=H, width=W, num_inference_steps=1, latents=lat0.clone(),
                              output_type="pil", decode_chunk_size=2).frames
            assert len(frames) == 1 and len(frames[0]) == T and frames[0][0].size == (W, H)
            # the CMP object the script also returns: same entry point (FCN.py:51-62)
            g = torch.Generator().manual_seed(1)
            img = torch.rand(1, 3, 128, 128, generator=g)
            sparse = torch.zeros(1, 2, 128, 128)
            mask = torch.zeros(1, 2, 128, 128)
            sparse[:, :, 40, 50], mask[:, :, 40, 50] = 5.0, 1.0
            assert cmp.run(img, sparse, mask).shape == (1, 2, 128, 128)
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] in ("models", "pipeline", "utils")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_from_unet_copies_trunk_and_zeroes_the_zero_convs():
    from mofa_video_b200.models.svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine import FlowControlNet
    from mofa_video_b200.models.unet_spatio_temporal_condition_controlnet import \
        UNetSpatioTemporalConditionControlNetModel
    cfg = dict(fixtures.TINY_CONFIG)
    cu, su = synthetic.unet_state_dict(cfg)
    unet = UNetSpatioTemporalConditionControlNetModel.from_state_dict(su, cu, device="cpu", ops=ref_ops)
    ad = FlowControlNet.from_unet(unet)
    sd = ad.state_dict()
    assert ad.config.num_frames == cfg["num_frames"] and tuple(ad.config.block_out_channels) == (64, 128, 256, 256)
    assert tuple(ad.config.conditioning_embedding_out_channels) == (16, 32, 96, 256)
    for k in sd:
        if k.startswith(("conv_in.", "time_embedding.", "down_blocks.", "mid_block.")):
            assert sd[k] is su[k], k                       # the UNet's tensors, by reference (:617-626)
        if k.startswith(("controlnet_down_blocks.", "controlnet_mid_block.", "flow_encoder.zeroconvs.",
                         "controlnet_cond_embedding.conv_out.")):
            assert float(sd[k].abs().max()) == 0.0, k      # zero_module
    assert not torch.equal(sd["add_embedding.linear_1.weight"], su["add_embedding.linear_1.weight"])  # not copied
    # zero-convs => the adapter is an exact no-op on the UNet (12 zero residuals), as right after from_unet in training
    inp = fixtures.make_step_inputs(cfg, 16, 16)
    down, mid, _, _ = ad.forward(inp["sample"], 1.0, inp["encoder_hidden_states"], inp["added_time_ids"],
                                 controlnet_cond=inp["controlnet_cond"], controlnet_flow=inp["controlnet_flow"],
                                 return_dict=False)
    assert len(down) == 12 and all(float(d.abs().max()) == 0.0 for d in down) and float(mid.abs().max()) == 0.0
    # the oracle UNet module is accepted too (anything with .config and .state_dict())
    ounet, _ = fixtures.make_models(cfg, seed=0)
    ad2 = FlowControlNet.from_unet(ounet, load_weights_from_unet=True, device="cpu", ops=ref_ops)
    assert torch.equal(ad2.state_dict()["conv_in.weight"], ounet.state_dict()["conv_in.weight"])
