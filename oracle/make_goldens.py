"""ORACLE tooling: generate tests/golden/*.pt by EXECUTING THE REFERENCE'S OWN CODE from /root/reference.

Runs only in the builder container (the GPU box has no /root/reference); the produced fixtures are committed.
The reference modules import diffusers 0.24 / cupy, which are absent, so minimal import stubs are installed
for the *base classes and helpers only* (ConfigMixin, register_to_config, SchedulerMixin, BaseOutput,
randn_tensor, logging, ModelMixin ...).  The arithmetic executed is the reference's:
  * utils/scheduling_euler_discrete_karras_fix.py : EulerDiscreteScheduler (whole class)
  * models/svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py :
        FlowControlNetConditioningEmbeddingSVD, FlowControlNetFirstFrameEncoder
  * models/cmp/models/modules/* + backbone/resnet.py + utils/visualize_utils.py (CMP forward, see make_cmp)

    python -m oracle.make_goldens
"""
import functools
import inspect
import os
import sys
import types
from collections import OrderedDict

import torch

REF = "/root/reference/MOFA-Video-Traj"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_stubs():
    class ConfigMixin:
        # diffusers' ConfigMixin.__getattr__ falls back to the registered config (the reference's scheduler
        # reads self.use_karras_sigmas before assigning it, SCHED.py:225 vs :246)
        def __getattr__(self, name):
            cfg = self.__dict__.get("config")
            if cfg is not None and name in cfg.__dict__:
                return cfg.__dict__[name]
            raise AttributeError(name)

    def register_to_config(init):
        @functools.wraps(init)
        def wrapper(self, *args, **kwargs):
            sig = inspect.signature(init)
            bound = sig.bind(self, *args, **kwargs)
            bound.apply_defaults()
            cfg = {k: v for k, v in bound.arguments.items() if k != "self"}
            self.config = types.SimpleNamespace(**cfg)
            self.config.__dict__["get"] = cfg.get
            init(self, *args, **kwargs)
        return wrapper

    class BaseOutput(OrderedDict):
        def __post_init__(self):
            pass

    class _Logger:
        def warning(self, *a, **k):
            pass

        info = debug = warning

    logging = types.SimpleNamespace(get_logger=lambda name=None: _Logger())

    def randn_tensor(shape, generator=None, device=None, dtype=None, layout=None):
        return torch.randn(shape, generator=generator, device=device, dtype=dtype)

    class SchedulerMixin:
        pass

    class _Dummy(torch.nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

    _mod("diffusers")
    _mod("diffusers.configuration_utils", ConfigMixin=ConfigMixin, register_to_config=register_to_config)
    _mod("diffusers.utils", BaseOutput=BaseOutput, logging=logging)
    _mod("diffusers.utils.torch_utils", randn_tensor=randn_tensor)
    _mod("diffusers.schedulers")
    _mod("diffusers.schedulers.scheduling_utils", KarrasDiffusionSchedulers=[], SchedulerMixin=SchedulerMixin)
    _mod("diffusers.loaders", FromOriginalControlnetMixin=type("FromOriginalControlnetMixin", (), {}))
    names = ["ADDED_KV_ATTENTION_PROCESSORS", "CROSS_ATTENTION_PROCESSORS", "AttentionProcessor",
             "AttnAddedKVProcessor", "AttnProcessor"]
    _mod("diffusers.models", UNetSpatioTemporalConditionModel=_Dummy)
    _mod("diffusers.models.attention_processor", **{n: _Dummy for n in names})
    _mod("diffusers.models.embeddings", TextImageProjection=_Dummy, TextImageTimeEmbedding=_Dummy,
         TextTimeEmbedding=_Dummy, TimestepEmbedding=_Dummy, Timesteps=_Dummy)
    _mod("diffusers.models.modeling_utils", ModelMixin=torch.nn.Module)
    _mod("diffusers.models.unet_3d_blocks", get_down_block=None, get_up_block=None,
         UNetMidBlockSpatioTemporal=_Dummy)
    # cupy-backed kernel module: not executable here
    _mod("cupy")


def load_reference_scheduler():
    install_stubs()
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_sched", os.path.join(REF, "utils",
                                                                              "scheduling_euler_discrete_karras_fix.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def make_scheduler():
    m = load_reference_scheduler()
    from oracle.scheduler import SVD_XT_SCHEDULER_CONFIG
    s = m.EulerDiscreteScheduler(**SVD_XT_SCHEDULER_CONFIG)
    g = {"init_noise_sigma_initial": float(s.init_noise_sigma)}
    for n in (25, 2):
        s.set_timesteps(n)
        g[f"sigmas_{n}"] = s.sigmas.clone()
        g[f"timesteps_{n}"] = s.timesteps.clone()
        g[f"init_noise_sigma_{n}"] = float(s.init_noise_sigma)
    s.set_timesteps(25)
    gen = torch.Generator().manual_seed(123)
    x = torch.randn(1, 3, 4, 6, 5, generator=gen) * float(s.init_noise_sigma)
    g["x0"] = x.clone()
    g["model_out"], g["scaled"], g["traj"] = [], [], []
    for t in s.timesteps:
        mo = torch.randn(1, 3, 4, 6, 5, generator=gen)
        g["model_out"].append(mo)
        g["scaled"].append(s.scale_model_input(x, t).clone())
        x = s.step(mo, t, x).prev_sample
        g["traj"].append(x.clone())
    torch.save(g, os.path.join(OUT, "scheduler_svdxt.pt"))
    print("scheduler golden written;", "sigma[0..2] =", g["sigmas_25"][:3].tolist())


def make_adapter_encoders():
    install_stubs()
    sys.path.insert(0, REF)
    # neighbours of FCN.py that cannot be imported here (diffusers blocks / cupy): give it what it names
    import torch.nn as nn

    def zero_module(module):  # same contract as controlnet_sdv.py:779-782
        for p in module.parameters():
            nn.init.zeros_(p)
        return module

    _mod("models.controlnet_sdv", ControlNetSDVModel=torch.nn.Module, zero_module=zero_module)
    _mod("models.softsplat", softsplat=None)
    _mod("models.cmp")
    _mod("models.cmp.models")
    _mod("models.cmp.utils")
    _mod("torchvision")
    _mod("torchvision.transforms")
    import importlib.util
    fn = os.path.join(REF, "models", "svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py")
    spec = importlib.util.spec_from_file_location("ref_fcn", fn)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    from oracle.cmp import seeded_state_dict
    ce = m.FlowControlNetConditioningEmbeddingSVD(conditioning_embedding_channels=32)   # small: keeps the fixture < 1 MB
    fe = m.FlowControlNetFirstFrameEncoder(c_in=32, channels=[32, 64, 128])
    # seeded weights (no zero-convs left, so the fixture exercises them) are rebuilt by the test from the seeds:
    # only inputs and outputs are stored
    ce.load_state_dict(seeded_state_dict(ce, seed=11))
    fe.load_state_dict(seeded_state_dict(fe, seed=12))
    gen = torch.Generator().manual_seed(1)
    with torch.no_grad():
        cond_in = torch.randn(1, 3, 64, 64, generator=gen)
        cond_out = ce(cond_in)
        flow_out = fe(cond_out)
    g = {"cond_embedding_seed": 11, "flow_encoder_seed": 12, "cond_in": cond_in, "cond_out": cond_out,
         "flow_out": flow_out}
    torch.save(g, os.path.join(OUT, "adapter_encoders.pt"))
    print("adapter encoder golden written:", [tuple(t.shape) for t in flow_out])


def make_cmp():
    """Run the reference's CMP module files (pure PyTorch) on CPU: ResNet-50-dilated + ShallowNet +
    MotionDecoderSkipLayer + Fuser arithmetic, with weights from oracle.cmp.seeded_state_dict."""
    import importlib.util
    import torch.nn.functional as F
    base = os.path.join(REF, "models", "cmp")

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(base, rel))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m

    resnet = load("ref_cmp_resnet", "models/backbone/resnet.py")
    shallow = load("ref_cmp_shallow", "models/modules/shallownet.py")
    decoder = load("ref_cmp_decoder", "models/modules/decoder.py")
    # modules/cmp.py looks its parts up through `models.cmp.models`: give it exactly those namespaces
    pkg = _mod("models")
    _mod("models.cmp")
    parts = _mod("models.cmp.models.modules", shallownet8x=shallow.shallownet8x,
                 MotionDecoderSkipLayer=decoder.MotionDecoderSkipLayer)
    mm = _mod("models.cmp.models", backbone=resnet, modules=parts)
    pkg.cmp = sys.modules["models.cmp"]
    sys.modules["models.cmp"].models = mm
    cmpmod = load("ref_cmp_module", "models/modules/cmp.py")
    params = dict(img_enc_dim=256, sparse_enc_dim=16, output_dim=198, pretrained_image_encoder=False,
                  decoder_combo=[1, 2, 4], skip_layer=True, image_encoder="resnet50", sparse_encoder="shallownet8x",
                  flow_decoder="MotionDecoderSkipLayer")
    torch.manual_seed(0)
    ref = cmpmod.CMP(params).eval()
    from oracle import cmp as ocmp
    ref.load_state_dict(ocmp.seeded_state_dict(ref, seed=3))
    g = torch.Generator().manual_seed(5)
    image = torch.rand(2, 3, 128, 128, generator=g)
    sparse = torch.zeros(2, 2, 128, 128)
    mask = torch.zeros(2, 2, 128, 128)
    idx = torch.randint(0, 128, (2, 12, 2), generator=g)
    for b in range(2):
        for (y, x) in idx[b].tolist():
            sparse[b, :, y, x] = torch.randn(2, generator=g) * 10
            mask[b, :, y, x] = 1
    with torch.no_grad():
        logits = ref((image * 2 - 1), torch.cat([sparse, mask], dim=1))
        # Fuser.convert_flow arithmetic (visualize_utils.py:13-19; its mesh is built with .cuda() so the lines are
        # restated on CPU here) + CMP_demo.run's align_corners upsample (FCN.py:56-60)
        nb, fmax = 99, 50
        step = 2 * fmax / float(nb)
        mesh = torch.arange(nb).view(1, -1, 1, 1).float() * step - fmax + step / 2
        px = F.softmax(logits[:, :nb], dim=1) * mesh
        py = F.softmax(logits[:, nb:], dim=1) * mesh
        flow = torch.cat([px.sum(1, keepdim=True), py.sum(1, keepdim=True)], dim=1)
        flow_up = F.interpolate(flow, size=(128, 128), mode="bilinear", align_corners=True)
    # the hints as (batch, y, x) points and their flow values: the dense sparse / mask tensors are rebuilt from them
    points = mask[:, 0].nonzero()
    values = sparse[points[:, 0], :, points[:, 1], points[:, 2]]
    torch.save({"image": image, "points": points, "values": values, "logits_sub": logits[:, ::9, ::4, ::4].clone(),
                "flow": flow_up, "seed": 3}, os.path.join(OUT, "cmp_small.pt"))
    print("cmp golden written:", tuple(logits.shape), float(flow_up.abs().mean()))


def make_hourglass():
    """ForegroundMatting of the Keypoint adapter, executed from the reference file (pure PyTorch)."""
    import importlib.util
    fn = "/root/reference/MOFA-Video-Keypoint/models/occlusion/hourglass.py"
    spec = importlib.util.spec_from_file_location("ref_hourglass", fn)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    from oracle import cmp as ocmp
    fm = m.ForegroundMatting(64).eval()
    fm.load_state_dict(ocmp.seeded_state_dict(fm, seed=7))   # weights regenerated from the seed by the test
    g = torch.Generator().manual_seed(2)
    ref_img, flow, warped = (torch.randn(2, 64, 12, 10, generator=g), torch.randn(2, 2, 12, 10, generator=g),
                             torch.randn(2, 64, 12, 10, generator=g))
    with torch.no_grad():
        out, mask = fm(ref_img, flow, warped)
    torch.save({"seed": 7, "ref": ref_img, "flow": flow, "warped": warped, "out": out, "mask": mask},
               os.path.join(OUT, "hourglass_small.pt"))
    print("hourglass golden written:", tuple(out.shape), tuple(mask.shape))


def make_networks():
    """Execute the reference's OWN network definitions and forward graphs -- models/unet_spatio_temporal_condition_
    controlnet.py (UNet: residual injection, Q1), models/controlnet_sdv.py (ControlNetSDVModel base class) and
    models/svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py (FlowControlNet.forward, get_warped_frames, Q2)
    -- on CPU.  The diffusers 0.24 *blocks* they instantiate are absent here, so the module names they import
    (diffusers.models.unet_3d_blocks / embeddings) are bound to oracle/d24_blocks.py; models.softsplat (CuPy) is bound
    to oracle/softsplat.py.  What this pins: the constructors' channel bookkeeping and state-dict layout (the oracle's
    state dict must load strictly), and every line of the two forward graphs.  What stays unpinned: the arithmetic
    inside the diffusers blocks."""
    install_stubs()
    import importlib.util

    from oracle import d24_blocks as D
    from oracle import fixtures
    from oracle.softsplat import softsplat as oracle_softsplat

    class ModelMixin(torch.nn.Module):
        @property
        def dtype(self):
            return next(self.parameters()).dtype

        @property
        def device(self):
            return next(self.parameters()).device

    _mod("diffusers.models.modeling_utils", ModelMixin=ModelMixin)
    _mod("diffusers.loaders", FromOriginalControlnetMixin=type("FromOriginalControlnetMixin", (), {}),
         UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}))
    _mod("diffusers.models.embeddings", TimestepEmbedding=D.TimestepEmbedding, Timesteps=D.Timesteps,
         TextImageProjection=None, TextImageTimeEmbedding=None, TextTimeEmbedding=None)
    _mod("diffusers.models.unet_3d_blocks", get_down_block=D.get_down_block, get_up_block=D.get_up_block,
         UNetMidBlockSpatioTemporal=D.UNetMidBlockSpatioTemporal,
         CrossAttnDownBlockSpatioTemporal=D.CrossAttnDownBlockSpatioTemporal,
         DownBlockSpatioTemporal=D.DownBlockSpatioTemporal)
    _mod("diffusers.models", UNetSpatioTemporalConditionModel=ModelMixin)
    sys.path.insert(0, REF)

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    ref_unet = load("ref_unet", "models/unet_spatio_temporal_condition_controlnet.py")
    ref_cn = load("models.controlnet_sdv", "models/controlnet_sdv.py")
    _mod("models.softsplat", softsplat=oracle_softsplat)
    _mod("models.cmp")
    _mod("models.cmp.models")
    _mod("models.cmp.utils")
    ref_fcn = load("ref_fcn_full", "models/svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py")

    cfg = dict(fixtures.TINY_CONFIG)
    o_unet, o_ad = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    torch.manual_seed(0)
    r_unet = ref_unet.UNetSpatioTemporalConditionControlNetModel(**cfg).eval()
    # FlowControlNet.__init__ (FCN.py:183-221) calls super().__init__() and FlowControlNetFirstFrameEncoder() WITHOUT
    # arguments, so the reference adapter only exists at the SVD-XT widths (1.4 GB).  For a fixture of test size the
    # two constructors' *default sizes* are overridden here; no forward code is touched.
    base_init = ref_cn.ControlNetSDVModel.__init__
    enc_init = ref_fcn.FlowControlNetFirstFrameEncoder.__init__
    boc = cfg["block_out_channels"]
    ref_cn.ControlNetSDVModel.__init__ = lambda self, *a, **k: base_init(self, *a, **{**cfg, **k})
    ref_fcn.FlowControlNetFirstFrameEncoder.__init__ = \
        lambda self, *a, **k: enc_init(self, *a, **{"c_in": boc[0], "channels": list(boc[:3]), **k})
    try:
        r_ad = ref_fcn.FlowControlNet(**cfg).eval()
    finally:
        ref_cn.ControlNetSDVModel.__init__ = base_init
        ref_fcn.FlowControlNetFirstFrameEncoder.__init__ = enc_init
    r_unet.load_state_dict(o_unet.state_dict(), strict=True)
    r_ad.load_state_dict(o_ad.state_dict(), strict=True)
    inp = fixtures.make_step_inputs(cfg, 16, 16)
    t = torch.tensor(1.6377)
    with torch.no_grad():
        dres, mid, _, _ = r_ad(inp["sample"], t, inp["encoder_hidden_states"], inp["added_time_ids"],
                               controlnet_cond=inp["controlnet_cond"], controlnet_flow=inp["controlnet_flow"],
                               conditioning_scale=0.8, return_dict=False)
        out = r_unet(inp["sample"], t, inp["encoder_hidden_states"], down_block_additional_residuals=dres,
                     mid_block_additional_residual=mid, added_time_ids=inp["added_time_ids"], return_dict=False)[0]

    def digest(x):  # compact fingerprint of a tensor: moments + a strided sample
        f = x.flatten()
        return {"shape": tuple(x.shape), "mean": f.mean().item(), "abs_mean": f.abs().mean().item(),
                "sample": f[:: max(1, f.numel() // 64)][:64].clone()}

    g = {"config": cfg, "seed": 0, "adapter_gain": 20.0, "latent_hw": (16, 16), "timestep": float(t),
         "conditioning_scale": 0.8, "unet_out": out.clone(),
         "mid": mid.clone(), "down_digests": [digest(d) for d in dres],
         "n_params": {"unet": sum(p.numel() for p in r_unet.parameters()),
                      "adapter": sum(p.numel() for p in r_ad.parameters())}}
    torch.save(g, os.path.join(OUT, "networks_tiny.pt"))
    print("network golden written:", tuple(out.shape), float(out.abs().mean()), g["n_params"])


def make_pipeline(H=128, W=128, steps=2, cond_scale=0.8, name="pipeline_tiny.pt"):
    """Execute the reference's FlowControlNetPipeline.__call__ (/root/reference/MOFA-Video-Traj/pipeline/pipeline.py:
    282-527, with _encode_image, _encode_vae_image, _get_add_time_ids, prepare_latents, _resize_with_antialiasing ...)
    on CPU for 2 steps at 128x128x3 frames with the reference UNet / FlowControlNet (see make_networks), the
    reference scheduler, and small seeded VAE / CLIP stand-ins.  Absent base classes are stubbed minimally:
    DiffusionPipeline (register_modules, _execution_device, progress_bar, maybe_free_model_hooks) and
    VaeImageProcessor (pil_to_numpy / numpy_to_pt / preprocess: PIL -> [0,1] -> NCHW -> 2x-1, diffusers 0.24 behaviour)."""
    install_stubs()
    import contextlib
    import importlib.util

    import numpy as np
    import PIL.Image

    from oracle import d24_blocks as D
    from oracle import fixtures
    from oracle.softsplat import softsplat as oracle_softsplat

    class ModelMixin(torch.nn.Module):
        @property
        def dtype(self):
            return next(self.parameters()).dtype

    class DiffusionPipeline:
        def __init__(self):
            pass

        def register_modules(self, **kw):
            for k, v in kw.items():
                setattr(self, k, v)

        @property
        def _execution_device(self):
            return torch.device("cpu")

        @contextlib.contextmanager
        def progress_bar(self, total=None):
            class _Bar:
                def update(self, *a):
                    pass
            yield _Bar()

        def maybe_free_model_hooks(self):
            pass

    class VaeImageProcessor:
        def __init__(self, vae_scale_factor=8, do_resize=True, do_normalize=True):
            self.vae_scale_factor = vae_scale_factor

        @staticmethod
        def pil_to_numpy(images):
            if not isinstance(images, list):
                images = [images]
            return np.stack([np.array(im).astype(np.float32) / 255.0 for im in images], axis=0)

        @staticmethod
        def numpy_to_pt(images):
            if images.ndim == 3:
                images = images[..., None]
            return torch.from_numpy(images.transpose(0, 3, 1, 2))

        def preprocess(self, image, height=None, width=None):
            if isinstance(image, PIL.Image.Image):
                image = [image]
            image = [im.resize((width, height), resample=PIL.Image.LANCZOS) if im.size != (width, height) else im
                     for im in image]
            return 2.0 * self.numpy_to_pt(self.pil_to_numpy(image)) - 1.0

    _mod("diffusers.models.modeling_utils", ModelMixin=ModelMixin)
    _mod("diffusers.loaders", FromOriginalControlnetMixin=type("FromOriginalControlnetMixin", (), {}),
         UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}))
    _mod("diffusers.models.embeddings", TimestepEmbedding=D.TimestepEmbedding, Timesteps=D.Timesteps,
         TextImageProjection=None, TextImageTimeEmbedding=None, TextTimeEmbedding=None)
    _mod("diffusers.models.unet_3d_blocks", get_down_block=D.get_down_block, get_up_block=D.get_up_block,
         UNetMidBlockSpatioTemporal=D.UNetMidBlockSpatioTemporal,
         CrossAttnDownBlockSpatioTemporal=D.CrossAttnDownBlockSpatioTemporal,
         DownBlockSpatioTemporal=D.DownBlockSpatioTemporal)
    _mod("diffusers.models", UNetSpatioTemporalConditionModel=ModelMixin, AutoencoderKLTemporalDecoder=ModelMixin)
    _mod("diffusers.image_processor", VaeImageProcessor=VaeImageProcessor)
    _mod("diffusers.pipelines")
    _mod("diffusers.pipelines.pipeline_utils", DiffusionPipeline=DiffusionPipeline)

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    _mod("models")
    ref_unet = load("models.unet_spatio_temporal_condition_controlnet",
                    "models/unet_spatio_temporal_condition_controlnet.py")
    ref_cn = load("models.controlnet_sdv", "models/controlnet_sdv.py")
    _mod("models.softsplat", softsplat=oracle_softsplat)
    _mod("models.cmp")
    _mod("models.cmp.models")
    _mod("models.cmp.utils")
    ref_fcn = load("models.svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine",
                   "models/svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine.py")
    _mod("utils")
    ref_sched = load("utils.scheduling_euler_discrete_karras_fix", "utils/scheduling_euler_discrete_karras_fix.py")
    ref_pipe = load("ref_pipeline", "pipeline/pipeline.py")

    cfg = dict(fixtures.TINY_CONFIG)
    boc = cfg["block_out_channels"]
    o_unet, o_ad = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    r_unet = ref_unet.UNetSpatioTemporalConditionControlNetModel(**cfg).eval()
    base_init = ref_cn.ControlNetSDVModel.__init__
    enc_init = ref_fcn.FlowControlNetFirstFrameEncoder.__init__
    ref_cn.ControlNetSDVModel.__init__ = lambda self, *a, **k: base_init(self, *a, **{**cfg, **k})
    ref_fcn.FlowControlNetFirstFrameEncoder.__init__ = \
        lambda self, *a, **k: enc_init(self, *a, **{"c_in": boc[0], "channels": list(boc[:3]), **k})
    try:
        r_ad = ref_fcn.FlowControlNet(**cfg).eval()
    finally:
        ref_cn.ControlNetSDVModel.__init__ = base_init
        ref_fcn.FlowControlNetFirstFrameEncoder.__init__ = enc_init
    r_unet.load_state_dict(o_unet.state_dict(), strict=True)
    r_ad.load_state_dict(o_ad.state_dict(), strict=True)
    from oracle.scheduler import SVD_XT_SCHEDULER_CONFIG
    sched = ref_sched.EulerDiscreteScheduler(**SVD_XT_SCHEDULER_CONFIG)
    vae, clip = fixtures.make_vae_and_clip(cfg["cross_attention_dim"])
    pipe = ref_pipe.FlowControlNetPipeline(vae=vae, image_encoder=clip, unet=r_unet, controlnet=r_ad, scheduler=sched,
                                           feature_extractor=None)
    T = cfg["num_frames"]
    img = fixtures.make_image(H, W)
    pil = PIL.Image.fromarray((img.permute(1, 2, 0) * 255).round().to(torch.uint8).numpy())
    flow = fixtures.make_flow(T, H, W)
    lat0 = torch.randn(1, T, 4, H // 8, W // 8, generator=torch.Generator().manual_seed(9))
    seen = []
    out = pipe(pil, pil, flow, height=H, width=W, num_frames=T, num_inference_steps=steps, latents=lat0.clone(),
               generator=torch.Generator().manual_seed(11), output_type="latent", controlnet_cond_scale=cond_scale,
               callback_on_step_end=lambda p_, i, t, kw: seen.append(float(t)) or {})
    g = {"config": cfg, "hw": (H, W), "steps": steps, "latent_seed": 9, "generator_seed": 11, "cond_scale": cond_scale,
         "image_u8": torch.from_numpy(np.array(pil)), "latents": out.frames.clone(), "timesteps_seen": seen}
    torch.save(g, os.path.join(OUT, name))
    print("pipeline golden written:", tuple(out.frames.shape), float(out.frames.abs().mean()), seen)


def _reference_tree(root):
    """Install the stubs and return a loader for files of one reference sub-project (Traj / Keypoint / Hybrid): the
    diffusers block / embedding modules are bound to oracle/d24_blocks.py, models.softsplat to oracle/softsplat.py,
    DiffusionPipeline / VaeImageProcessor to minimal stand-ins (see make_pipeline)."""
    install_stubs()
    import contextlib
    import importlib.util

    import numpy as np
    import PIL.Image

    from oracle import d24_blocks as D
    from oracle.softsplat import softsplat as oracle_softsplat

    class ModelMixin(torch.nn.Module):
        @property
        def dtype(self):
            return next(self.parameters()).dtype

    class DiffusionPipeline:
        def __init__(self):
            pass

        def register_modules(self, **kw):
            for k, v in kw.items():
                setattr(self, k, v)

        @property
        def _execution_device(self):
            return torch.device("cpu")

        @contextlib.contextmanager
        def progress_bar(self, total=None):
            class _Bar:
                def update(self, *a):
                    pass
            yield _Bar()

        def maybe_free_model_hooks(self):
            pass

    class VaeImageProcessor:
        def __init__(self, vae_scale_factor=8, do_resize=True, do_normalize=True):
            self.vae_scale_factor = vae_scale_factor

        @staticmethod
        def pil_to_numpy(images):
            if not isinstance(images, list):
                images = [images]
            return np.stack([np.array(im).astype(np.float32) / 255.0 for im in images], axis=0)

        @staticmethod
        def numpy_to_pt(images):
            if images.ndim == 3:
                images = images[..., None]
            return torch.from_numpy(images.transpose(0, 3, 1, 2))

        def preprocess(self, image, height=None, width=None):
            if isinstance(image, PIL.Image.Image):
                image = [image]
            image = [im.resize((width, height), resample=PIL.Image.LANCZOS) if im.size != (width, height) else im
                     for im in image]
            return 2.0 * self.numpy_to_pt(self.pil_to_numpy(image)) - 1.0

    _mod("diffusers.models.modeling_utils", ModelMixin=ModelMixin)
    _mod("diffusers.loaders", FromOriginalControlnetMixin=type("FromOriginalControlnetMixin", (), {}),
         UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}))
    _mod("diffusers.models.embeddings", TimestepEmbedding=D.TimestepEmbedding, Timesteps=D.Timesteps,
         TextImageProjection=None, TextImageTimeEmbedding=None, TextTimeEmbedding=None)
    _mod("diffusers.models.unet_3d_blocks", get_down_block=D.get_down_block, get_up_block=D.get_up_block,
         UNetMidBlockSpatioTemporal=D.UNetMidBlockSpatioTemporal,
         CrossAttnDownBlockSpatioTemporal=D.CrossAttnDownBlockSpatioTemporal,
         DownBlockSpatioTemporal=D.DownBlockSpatioTemporal)
    _mod("diffusers.models", UNetSpatioTemporalConditionModel=ModelMixin, AutoencoderKLTemporalDecoder=ModelMixin)
    _mod("diffusers.image_processor", VaeImageProcessor=VaeImageProcessor)
    _mod("diffusers.pipelines")
    _mod("diffusers.pipelines.pipeline_utils", DiffusionPipeline=DiffusionPipeline)
    _mod("models")
    _mod("models.softsplat", softsplat=oracle_softsplat)
    _mod("models.cmp")
    _mod("models.cmp.models")
    _mod("models.cmp.utils")
    _mod("models.occlusion")
    _mod("utils")

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(root, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m
    return load


def _build_reference_adapter(ref_cn, mod, cfg, state_dict, hourglass=None):
    """Instantiate a reference FlowControlNet at the test widths (its constructor hard-codes the SVD-XT sizes: default
    sizes overridden, zero_outs / occlusions re-created from the reference's own classes) and load the oracle weights."""
    import torch.nn as nn
    boc = cfg["block_out_channels"]
    base_init = ref_cn.ControlNetSDVModel.__init__
    enc_init = mod.FlowControlNetFirstFrameEncoder.__init__
    ref_cn.ControlNetSDVModel.__init__ = lambda self, *a, **k: base_init(self, *a, **{**cfg, **k})
    mod.FlowControlNetFirstFrameEncoder.__init__ = \
        lambda self, *a, **k: enc_init(self, *a, **{"c_in": boc[0], "channels": list(boc[:3]), **k})
    try:
        net = mod.FlowControlNet(**cfg)
    finally:
        ref_cn.ControlNetSDVModel.__init__ = base_init
        mod.FlowControlNetFirstFrameEncoder.__init__ = enc_init
    if hourglass is not None:
        chans = {"8": boc[0], "16": boc[0], "32": boc[1], "64": boc[2]}
        net.zero_outs = nn.ModuleDict({k: nn.Conv2d(c, c, kernel_size=1) for k, c in chans.items()})
        net.occlusions = nn.ModuleDict({k: hourglass.ForegroundMatting(c) for k, c in chans.items()})
    net.load_state_dict(state_dict, strict=True)
    return net.eval()


KP_CONFIG_UPDATE = dict(block_out_channels=(320, 128, 256, 256), num_attention_heads=(5, 2, 4, 4))


def _kp_inputs(cfg, H, W, F_frames):
    import numpy as np
    import PIL.Image

    from oracle import fixtures
    g = torch.Generator().manual_seed(3)
    img = fixtures.make_image(H, W)
    pil = PIL.Image.fromarray((img.permute(1, 2, 0) * 255).round().to(torch.uint8).numpy())
    flow = fixtures.make_flow(F_frames, H, W)
    ldmk = torch.rand(1, F_frames, 3, H, W, generator=g).half().float()
    lat0 = torch.randn(1, F_frames, 4, H // 8, W // 8, generator=g)
    return pil, torch.from_numpy(np.array(pil)), flow, ldmk, lat0


def make_keypoint_pipeline():
    """Execute /root/reference/MOFA-Video-Keypoint/pipeline/svdxt_pipeline_ctrlnet_loop.py FlowControlNetPipeline.__call__
    (windowed views, per-view denoise, _step_index rewind, value / count averaging, :287-664) for a 5-frame clip with
    window_size 3, stride 1, 2 steps, with the Keypoint tree's own UNet / ldmk_ctrlnet / hourglass / scheduler files."""
    K = "/root/reference/MOFA-Video-Keypoint"
    load = _reference_tree(K)
    from oracle import fixtures
    from oracle.scheduler import SVD_XT_SCHEDULER_CONFIG
    ref_unet = load("models.unet_spatio_temporal_condition_controlnet", "models/unet_spatio_temporal_condition_controlnet.py")
    ref_cn = load("models.controlnet_sdv", "models/controlnet_sdv.py")
    ref_hg = load("models.occlusion.hourglass", "models/occlusion/hourglass.py")
    ref_ldmk = load("models.ldmk_ctrlnet", "models/ldmk_ctrlnet.py")
    ref_sched = load("utils.scheduling_euler_discrete_karras_fix", "utils/scheduling_euler_discrete_karras_fix.py")
    ref_pipe = load("ref_kp_pipeline", "pipeline/svdxt_pipeline_ctrlnet_loop.py")
    cfg = dict(fixtures.TINY_CONFIG)
    cfg.update(KP_CONFIG_UPDATE)
    o_unet, _ = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    o_face = fixtures.make_ldmk_adapter(cfg)
    r_unet = ref_unet.UNetSpatioTemporalConditionControlNetModel(**cfg).eval()
    r_unet.load_state_dict(o_unet.state_dict(), strict=True)
    r_face = _build_reference_adapter(ref_cn, ref_ldmk, cfg, o_face.state_dict(), hourglass=ref_hg)
    vae, clip = fixtures.make_vae_and_clip(cfg["cross_attention_dim"])
    pipe = ref_pipe.FlowControlNetPipeline(vae=vae, image_encoder=clip, unet=r_unet, controlnet=r_face,
                                           scheduler=ref_sched.EulerDiscreteScheduler(**SVD_XT_SCHEDULER_CONFIG),
                                           feature_extractor=None)
    H = W = 128
    T, F_frames, stride = cfg["num_frames"], 5, 1
    pil, u8, flow, ldmk, lat0 = _kp_inputs(cfg, H, W, F_frames)
    out = pipe(pil, pil, flow, ldmk, height=H, width=W, num_frames=F_frames, num_inference_steps=2,
               latents=lat0.clone(), generator=torch.Generator().manual_seed(11), output_type="latent",
               window_size=T, stride=stride)
    g = {"config": cfg, "hw": (H, W), "frames": F_frames, "stride": stride, "steps": 2, "generator_seed": 11,
         "image_u8": u8, "latents": out.frames.clone()}
    torch.save(g, os.path.join(OUT, "keypoint_pipeline_tiny.pt"))
    print("keypoint pipeline golden written:", tuple(out.frames.shape), float(out.frames.abs().mean()))


def make_hybrid_pipeline():
    """Execute /root/reference/MOFA-Video-Hybrid/pipeline/pipeline.py FlowControlNetPipeline.__call__ (face adapter
    inside the mask, drag adapter outside, nearest-resized mask per level, :291-520) with the Hybrid tree's own files."""
    Hy = "/root/reference/MOFA-Video-Hybrid"
    load = _reference_tree(Hy)
    from oracle import fixtures
    from oracle.scheduler import SVD_XT_SCHEDULER_CONFIG
    ref_unet = load("models.unet_spatio_temporal_condition_controlnet", "models/unet_spatio_temporal_condition_controlnet.py")
    ref_cn = load("models.controlnet_sdv", "models/controlnet_sdv.py")
    ref_hg = load("models.occlusion.hourglass", "models/occlusion/hourglass.py")
    ref_traj = load("models.traj_ctrlnet", "models/traj_ctrlnet.py")
    ref_ldmk = load("models.ldmk_ctrlnet", "models/ldmk_ctrlnet.py")
    ref_sched = load("utils.scheduling_euler_discrete_karras_fix", "utils/scheduling_euler_discrete_karras_fix.py")
    ref_pipe = load("ref_hybrid_pipeline", "pipeline/pipeline.py")
    cfg = dict(fixtures.TINY_CONFIG)
    cfg.update(KP_CONFIG_UPDATE)
    o_unet, o_drag = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    o_face = fixtures.make_ldmk_adapter(cfg)
    r_unet = ref_unet.UNetSpatioTemporalConditionControlNetModel(**cfg).eval()
    r_unet.load_state_dict(o_unet.state_dict(), strict=True)
    r_drag = _build_reference_adapter(ref_cn, ref_traj, cfg, o_drag.state_dict())
    r_face = _build_reference_adapter(ref_cn, ref_ldmk, cfg, o_face.state_dict(), hourglass=ref_hg)
    vae, clip = fixtures.make_vae_and_clip(cfg["cross_attention_dim"])
    pipe = ref_pipe.FlowControlNetPipeline(vae=vae, image_encoder=clip, unet=r_unet, drag_controlnet=r_drag,
                                           face_controlnet=r_face,
                                           scheduler=ref_sched.EulerDiscreteScheduler(**SVD_XT_SCHEDULER_CONFIG),
                                           feature_extractor=None)
    H = W = 128
    T = cfg["num_frames"]
    pil, u8, flow, ldmk, lat0 = _kp_inputs(cfg, H, W, T)
    drag_flow = (fixtures.make_flow(T, H, W, seed=99) * 0.5).half().float()
    mask = torch.zeros(1, 1, H, W)
    mask[..., 20:90, 30:100] = 1.0
    out = pipe(pil, pil, flow, ldmk, drag_flow, mask, height=H, width=W, num_frames=T, num_inference_steps=2,
               latents=lat0.clone(), generator=torch.Generator().manual_seed(11), output_type="latent",
               ctrl_scale_traj=1.1, ctrl_scale_ldmk=0.9)
    g = {"config": cfg, "hw": (H, W), "steps": 2, "generator_seed": 11, "image_u8": u8, "latents": out.frames.clone(),
         "scale_traj": 1.1, "scale_ldmk": 0.9}
    torch.save(g, os.path.join(OUT, "hybrid_pipeline_tiny.pt"))
    print("hybrid pipeline golden written:", tuple(out.frames.shape), float(out.frames.abs().mean()))


def make_keypoint_network():
    """Same as make_networks for the Keypoint adapter: executes /root/reference/MOFA-Video-Keypoint/models/ldmk_ctrlnet.py
    (FlowControlNet.__init__ / get_warped_frames / forward with landmarks, :187-575), its controlnet_sdv.py and its
    occlusion/hourglass.py.  The constructor hard-codes the SVD-XT widths (super().__init__() without arguments,
    Conv2d(320, 320) ..., ForegroundMatting(1280)); the default sizes are overridden and the four zero_outs /
    occlusions entries re-created from the reference's own classes at the test widths.  No forward code is touched."""
    install_stubs()
    import importlib.util

    import torch.nn as nn

    from oracle import d24_blocks as D
    from oracle import fixtures
    from oracle.softsplat import softsplat as oracle_softsplat
    K = "/root/reference/MOFA-Video-Keypoint"

    class ModelMixin(torch.nn.Module):
        @property
        def dtype(self):
            return next(self.parameters()).dtype

    _mod("diffusers.models.modeling_utils", ModelMixin=ModelMixin)
    _mod("diffusers.loaders", FromOriginalControlnetMixin=type("FromOriginalControlnetMixin", (), {}),
         UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}))
    _mod("diffusers.models.embeddings", TimestepEmbedding=D.TimestepEmbedding, Timesteps=D.Timesteps,
         TextImageProjection=None, TextImageTimeEmbedding=None, TextTimeEmbedding=None)
    _mod("diffusers.models.unet_3d_blocks", get_down_block=D.get_down_block, get_up_block=D.get_up_block,
         UNetMidBlockSpatioTemporal=D.UNetMidBlockSpatioTemporal,
         CrossAttnDownBlockSpatioTemporal=D.CrossAttnDownBlockSpatioTemporal,
         DownBlockSpatioTemporal=D.DownBlockSpatioTemporal)
    _mod("diffusers.models", UNetSpatioTemporalConditionModel=ModelMixin)

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(K, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
        return m

    _mod("models")
    ref_cn = load("models.controlnet_sdv", "models/controlnet_sdv.py")
    _mod("models.softsplat", softsplat=oracle_softsplat)
    _mod("models.cmp")
    _mod("models.cmp.models")
    _mod("models.cmp.utils")
    _mod("models.occlusion")
    ref_hg = load("models.occlusion.hourglass", "models/occlusion/hourglass.py")
    ref_ldmk = load("ref_ldmk", "models/ldmk_ctrlnet.py")

    # forward() adds the landmark embedding where `sample.shape[1] == 320` (a literal, :501): the first level keeps the
    # SVD-XT width so that branch is exercised; the deeper levels are shrunk
    cfg = dict(fixtures.TINY_CONFIG)
    cfg.update(block_out_channels=(320, 128, 256, 256), num_attention_heads=(5, 2, 4, 4))
    boc = cfg["block_out_channels"]
    o_ad = fixtures.make_ldmk_adapter(cfg)
    base_init = ref_cn.ControlNetSDVModel.__init__
    enc_init = ref_ldmk.FlowControlNetFirstFrameEncoder.__init__
    ref_cn.ControlNetSDVModel.__init__ = lambda self, *a, **k: base_init(self, *a, **{**cfg, **k})
    ref_ldmk.FlowControlNetFirstFrameEncoder.__init__ = \
        lambda self, *a, **k: enc_init(self, *a, **{"c_in": boc[0], "channels": list(boc[:3]), **k})
    try:
        r_ad = ref_ldmk.FlowControlNet(**cfg)
    finally:
        ref_cn.ControlNetSDVModel.__init__ = base_init
        ref_ldmk.FlowControlNetFirstFrameEncoder.__init__ = enc_init
    chans = {"8": boc[0], "16": boc[0], "32": boc[1], "64": boc[2]}
    r_ad.zero_outs = nn.ModuleDict({k: nn.Conv2d(c, c, kernel_size=1) for k, c in chans.items()})
    r_ad.occlusions = nn.ModuleDict({k: ref_hg.ForegroundMatting(c) for k, c in chans.items()})
    r_ad.load_state_dict(o_ad.state_dict(), strict=True)
    r_ad.eval()
    H = W = 16
    T = cfg["num_frames"]
    inp = fixtures.make_step_inputs(cfg, H, W)
    landmarks = torch.rand(1, T, 3, 8 * H, 8 * W, generator=torch.Generator().manual_seed(11)).half().float()
    landmarks = landmarks.repeat(2, 1, 1, 1, 1)
    t = torch.tensor(1.6377)
    with torch.no_grad():
        dres, mid, _, occ = r_ad(inp["sample"], t, inp["encoder_hidden_states"], inp["added_time_ids"],
                                 controlnet_cond=inp["controlnet_cond"], controlnet_flow=inp["controlnet_flow"],
                                 landmarks=landmarks, conditioning_scale=0.9, return_dict=False)

    def digest(x):
        f = x.flatten()
        return {"shape": tuple(x.shape), "mean": f.mean().item(), "abs_mean": f.abs().mean().item(),
                "sample": f[:: max(1, f.numel() // 64)][:64].clone()}

    g = {"config": cfg, "latent_hw": (H, W), "timestep": float(t), "conditioning_scale": 0.9, "landmark_seed": 11,
         "mid": mid.clone(), "down_digests": [digest(d) for d in dres], "occ_digests": [digest(m) for m in occ],
         "n_params": sum(p.numel() for p in r_ad.parameters())}
    torch.save(g, os.path.join(OUT, "keypoint_network_tiny.pt"))
    print("keypoint network golden written:", tuple(mid.shape), float(mid.abs().mean()), g["n_params"])


def _extract_functions(path, names, namespace):
    """exec() the named top-level function definitions of a reference file, verbatim (ast), into `namespace`."""
    import ast
    with open(path) as f:
        tree = ast.parse(f.read())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    assert len(body) == len(names), (path, names)
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), namespace)
    return namespace


def sparse_flow_cases():
    """Seeded inputs of the control-signal rasterisation goldens (shared with the tests)."""
    import numpy as np
    rng = np.random.default_rng(0)
    K, n, H, W = 7, 5, 24, 32
    pts = np.zeros((K, n + 1, 2))
    pts[:, 0, 0] = rng.uniform(0, W - 1, K)
    pts[:, 0, 1] = rng.uniform(0, H - 1, K)
    pts[5, 0] = pts[2, 0]                                    # two tracks from the same pixel: their flows add
    pts[:, 1:] = pts[:, 0:1] + rng.normal(0, 6, (K, n, 2))
    g = torch.Generator().manual_seed(4)
    lm = torch.rand(2, 4, 9, 2, generator=g) * torch.tensor([W + 4.0, H + 4.0]) - 2   # some landmarks off the image
    lm[:, 0, 3] = lm[:, 0, 6]                                # two landmarks on the same pixel: the later one wins
    return {"points": pts, "n_steps": n, "H": H, "W": W, "landmarks": lm, "t": 4}


def make_sparse_flow():
    """tests/golden/sparse_flow_ref.pt: outputs of the reference's OWN get_sparseflow_and_mask_forward
    (MOFA-Video-Traj/run_gradio.py:61-86) and get_sparse_flow / sample_optical_flow (MOFA-Video-Keypoint/utils/utils.py:
    81-119), both extracted verbatim from their files."""
    import numpy as np
    c = sparse_flow_cases()
    t_ns = _extract_functions("/root/reference/MOFA-Video-Traj/run_gradio.py", ["get_sparseflow_and_mask_forward"],
                              {"np": np})
    k_ns = _extract_functions("/root/reference/MOFA-Video-Keypoint/utils/utils.py",
                              ["sample_optical_flow", "get_sparse_flow"], {"torch": torch})
    out = {}
    for back in (False, True):
        f, m = t_ns["get_sparseflow_and_mask_forward"](c["points"], c["n_steps"], c["H"], c["W"], is_backward_flow=back)
        out[f"traj_flow_back{int(back)}"] = torch.from_numpy(f)
        out[f"traj_mask_back{int(back)}"] = torch.from_numpy(m)
    f, m = k_ns["get_sparse_flow"](c["landmarks"].clone(), c["H"], c["W"], c["t"])
    out["ldmk_flow"], out["ldmk_mask"] = f.contiguous(), m.contiguous()
    torch.save(out, os.path.join(OUT, "sparse_flow_ref.pt"))
    print("sparse-flow golden written:", {k: tuple(v.shape) for k, v in out.items()})


def make_init_models_calls():
    """tests/golden/init_models_calls.json: every call the reference's model-loading function `init_models`
    (MOFA-Video-Traj/run_gradio.py:90-159, extracted verbatim) makes on the names it imports, in order, recorded by
    running it against recording stand-ins with its default options.  tests/test_boundary_init_models_cpu.py replays the
    calls against this package.  Encoding: {"ref": n} is the object op n returned, {"arg": name} an argument of
    init_models, anything else a literal."""
    import json
    ops = []

    def enc(v):
        if isinstance(v, _Rec):
            return {"ref": v.ref}
        if isinstance(v, _Arg):
            return {"arg": v.name}
        if isinstance(v, (tuple, list)):
            return [enc(x) for x in v]
        assert v is None or isinstance(v, (str, int, float, bool)), type(v)
        return v

    class _Arg:
        def __init__(self, name):
            self.name = name

    class _Rec:
        def __init__(self, op):
            ops.append({**op, "out": len(ops)})
            self.ref = len(ops) - 1

        def __getattr__(self, method):
            if method.startswith("__"):
                raise AttributeError(method)
            return lambda *a, **k: _Rec({"op": "call", "obj": self.ref, "method": method, "args": enc(a),
                                         "kwargs": {n: enc(v) for n, v in k.items()}})

        def __call__(self, *a, **k):
            return _Rec({"op": "call", "obj": self.ref, "method": None, "args": enc(a),
                         "kwargs": {n: enc(v) for n, v in k.items()}})

    def module(name):
        m = _mod(name)

        def getattr_(attr):        # the import machinery probes dunders and looks a name up more than once
            if attr.startswith("__"):
                raise AttributeError(attr)
            rec = _Rec({"op": "name", "module": name, "name": attr})
            setattr(m, attr, rec)
            return rec
        m.__getattr__ = getattr_
        return m

    for name in ("models", "pipeline", "models.unet_spatio_temporal_condition_controlnet", "pipeline.pipeline",
                 "models.svdxt_featureflow_forward_controlnet_s2d_fixcmp_norefine"):
        module(name)
    ns = {n: _Rec({"op": "name", "module": None, "name": n})
          for n in ("CLIPVisionModelWithProjection", "AutoencoderKLTemporalDecoder")}
    _extract_functions(os.path.join(REF, "run_gradio.py"), ["init_models"], ns)
    args = ("pretrained_model_name_or_path", "resume_from_checkpoint", "weight_dtype", "device")
    ret = ns["init_models"](*[_Arg(a) for a in args])
    out ={"args": list(args), "ops": ops, "returns": enc(ret)}
    with open(os.path.join(OUT, "init_models_calls.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("init_models call trace written:", len(ops), "ops")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--sparse-flow" in sys.argv:
        make_sparse_flow()
        sys.exit(0)
    if "--init-models" in sys.argv:
        make_init_models_calls()
        sys.exit(0)
    make_scheduler()
    if "--networks" in sys.argv or "--all" in sys.argv:
        make_networks()
    if "--pipeline" in sys.argv:
        make_pipeline()           # separate process as well
    if "--pipeline-rect" in sys.argv:
        make_pipeline(H=128, W=192, steps=3, cond_scale=1.0, name="pipeline_tiny_rect.pt")
    if "--keypoint-pipeline" in sys.argv:
        make_keypoint_pipeline()
    if "--hybrid-pipeline" in sys.argv:
        make_hybrid_pipeline()
    if "--keypoint" in sys.argv:
        make_keypoint_network()   # separate process from --networks: both bind sys.modules["models.*"]
    if "--all" in sys.argv:
        make_adapter_encoders()
        make_cmp()
        make_hourglass()
