"""-m "not gpu": the oracle against (i) fixtures generated from the reference's own code
(tests/golden/*.pt, made by oracle/make_goldens.py) and (ii) algebraic identities (SURVEY.md §4)."""
import os

import pytest
import torch

from oracle import fixtures
from oracle import scheduler as osched
from oracle.softsplat import softsplat

GOLD = os.path.join(os.path.dirname(__file__), "golden")
FIXTURE_THREADS = 8   # torch intra-op threads of the host that generated the pipeline fixtures


def _gold(name):
    fn = os.path.join(GOLD, name)
    if not os.path.exists(fn):
        pytest.skip(f"{name} not generated")
    return torch.load(fn)


def test_scheduler_matches_reference_fixture():
    g = _gold("scheduler_svdxt.pt")
    s = osched.EulerDiscreteScheduler()
    assert abs(float(s.init_noise_sigma) - g["init_noise_sigma_initial"]) < 1e-4
    for n in (25, 2):
        s.set_timesteps(n)
        assert torch.allclose(s.sigmas, g[f"sigmas_{n}"], rtol=1e-6, atol=0)
        assert torch.allclose(s.timesteps, g[f"timesteps_{n}"], rtol=1e-6, atol=0)
        assert abs(float(s.init_noise_sigma) - g[f"init_noise_sigma_{n}"]) < 1e-3
    # one full trajectory of scale_model_input + step on seeded tensors
    s.set_timesteps(25)
    x = g["x0"].clone()
    for i, t in enumerate(s.timesteps):
        xin = s.scale_model_input(x, t)
        assert torch.allclose(xin, g["scaled"][i], rtol=1e-5, atol=1e-6)
        x = s.step(g["model_out"][i], t, x)
        assert torch.allclose(x, g["traj"][i], rtol=1e-5, atol=1e-5)


def test_product_scheduler_matches_reference_fixture():
    from mofa_video_b200.utils.scheduling_euler_discrete_karras_fix import EulerDiscreteScheduler
    g = _gold("scheduler_svdxt.pt")
    s = EulerDiscreteScheduler()
    for n in (25, 2):
        s.set_timesteps(n)
        assert torch.allclose(s.sigmas, g[f"sigmas_{n}"], rtol=1e-6, atol=0)
        assert torch.allclose(s.timesteps, g[f"timesteps_{n}"], rtol=1e-6, atol=0)
    s.set_timesteps(25)
    x = g["x0"].clone()
    for i, t in enumerate(s.timesteps):
        assert torch.allclose(s.scale_model_input(x, t), g["scaled"][i], rtol=1e-5, atol=1e-6)
        x = s.step(g["model_out"][i], t, x).prev_sample
        assert torch.allclose(x, g["traj"][i], rtol=1e-5, atol=1e-5)


def test_adapter_encoders_match_reference_fixture():
    from oracle.cmp import seeded_state_dict
    from oracle.models import FlowControlNetConditioningEmbeddingSVD, FlowControlNetFirstFrameEncoder
    g = _gold("adapter_encoders.pt")
    ce = FlowControlNetConditioningEmbeddingSVD(32)
    ce.load_state_dict(seeded_state_dict(ce, seed=g["cond_embedding_seed"]))
    fe = FlowControlNetFirstFrameEncoder(c_in=32, channels=(32, 64, 128))
    fe.load_state_dict(seeded_state_dict(fe, seed=g["flow_encoder_seed"]))
    with torch.no_grad():
        c = ce(g["cond_in"])
        assert torch.allclose(c, g["cond_out"], rtol=1e-5, atol=1e-6)
        for a, b in zip(fe(g["cond_out"]), g["flow_out"]):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)


def test_softsplat_identities():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 5, 7, 9, generator=g)
    zero = torch.zeros(2, 2, 7, 9)
    assert torch.allclose(softsplat(x, zero, None, "avg"), x / (1 + 1e-7), rtol=1e-6, atol=1e-7)
    # integer shift by (+2, +1): out[y+1, x+2] = in[y, x]; vacated pixels are empty -> 0
    fl = torch.zeros(2, 2, 7, 9)
    fl[:, 0], fl[:, 1] = 2.0, 1.0
    o = softsplat(x, fl, None, "avg")
    assert torch.allclose(o[:, :, 1:, 2:], x[:, :, :-1, :-2] / (1 + 1e-7), rtol=1e-6, atol=1e-7)
    assert o[:, :, 0].abs().max() == 0 and o[:, :, :, :2].abs().max() == 0
    # 'sum' mode conserves mass for flows that stay in bounds
    fl = torch.rand(2, 2, 7, 9, generator=g) * 0.9
    inner = torch.zeros_like(x)
    inner[:, :, 1:-2, 1:-2] = x[:, :, 1:-2, 1:-2]
    assert torch.allclose(softsplat(inner, fl, None, "sum").sum((2, 3)), inner.sum((2, 3)), rtol=1e-4, atol=1e-4)
    # non-finite flow is skipped (softsplat.py:301-302)
    fl = torch.zeros(1, 2, 4, 4)
    fl[0, 0, 1, 1] = float("nan")
    o = softsplat(torch.ones(1, 1, 4, 4), fl, None, "sum")
    assert o[0, 0, 1, 1] == 0 and o.sum() == 15


def test_zero_convs_make_adapter_a_noop():
    """Q19: with the reference's zero-initialised output convs every residual is exactly zero."""
    from oracle import fixtures
    from oracle.models import FlowControlNet
    cfg = dict(fixtures.TINY_CONFIG)
    torch.manual_seed(0)
    ad = FlowControlNet(**cfg).eval()
    inp = fixtures.make_step_inputs(cfg, 16, 16)
    with torch.no_grad():
        dres, mid, _, _ = ad(inp["sample"], torch.tensor(1.0), inp["encoder_hidden_states"], inp["added_time_ids"],
                             controlnet_cond=inp["controlnet_cond"], controlnet_flow=inp["controlnet_flow"])
    assert all(d.abs().max() == 0 for d in dres) and mid.abs().max() == 0


def test_network_forward_graphs_match_reference_fixture():
    """tests/golden/networks_tiny.pt comes from EXECUTING the reference's own UNet / ControlNetSDVModel / FlowControlNet
    definitions and forward code (oracle/make_goldens.py:make_networks; the absent diffusers block classes are bound to
    oracle/d24_blocks.py).  The oracle's restated forward graphs must reproduce it exactly: residual injection with the
    Q1 multiplicities, warp-add placement (Q2), conditioning scale, time-embedding plumbing, state-dict layout."""
    g = _gold("networks_tiny.pt")
    cfg = g["config"]
    unet, ad = fixtures.make_models(cfg, seed=g["seed"], adapter_gain=g["adapter_gain"])
    assert sum(p.numel() for p in unet.parameters()) == g["n_params"]["unet"]
    assert sum(p.numel() for p in ad.parameters()) == g["n_params"]["adapter"]
    inp = fixtures.make_step_inputs(cfg, *g["latent_hw"])
    t = torch.tensor(g["timestep"])
    with torch.no_grad():
        dres, mid, _, _ = ad(inp["sample"], t, inp["encoder_hidden_states"], inp["added_time_ids"],
                             controlnet_cond=inp["controlnet_cond"], controlnet_flow=inp["controlnet_flow"],
                             conditioning_scale=g["conditioning_scale"])
        out = unet(inp["sample"], t, inp["encoder_hidden_states"], dres, mid, added_time_ids=inp["added_time_ids"])[0]
    assert (out - g["unet_out"]).abs().max().item() <= 1e-6 * g["unet_out"].abs().max().item()
    assert (mid - g["mid"]).abs().max().item() <= 1e-6 * g["mid"].abs().max().item()
    assert len(dres) == len(g["down_digests"]) == 12
    for d, dg in zip(dres, g["down_digests"]):
        f = d.flatten()
        assert tuple(d.shape) == dg["shape"]
        assert (f[:: max(1, f.numel() // 64)][:64] - dg["sample"]).abs().max().item() <= 1e-6
        assert abs(f.abs().mean().item() - dg["abs_mean"]) <= 1e-6


@pytest.mark.parametrize("fixture", ["pipeline_tiny.pt", "pipeline_tiny_rect.pt"])
def test_pipeline_call_matches_reference_fixture(fixture):
    """tests/golden/pipeline_tiny.pt comes from EXECUTING the reference's FlowControlNetPipeline.__call__ (with its own
    UNet / FlowControlNet / scheduler files; DiffusionPipeline and VaeImageProcessor stubbed, oracle/make_goldens.py:
    make_pipeline).  oracle.pipeline.run_pipeline -- the oracle every engine pipeline test compares against -- must
    reproduce the 2-step latents: PIL conversion, CLIP resize path (Q3), VAE encode of the noise-augmented frame (Q7),
    added-time-id constants (Q4), CFG with the per-frame scale, Karras-sigma Euler steps.

    Runs with the FIXTURE_THREADS intra-op threads the fixtures were generated with: the square clip's latents move by
    ~7e-5 of their max when the CPU reductions are split across another thread count (3 or 16), beyond the 1e-5 below."""
    import PIL.Image

    from oracle import pipeline as opipe
    g = _gold(fixture)          # square 128x128 / 2 steps / scale 0.8, and rectangular 128x192 / 3 steps / scale 1.0
    cfg = g["config"]
    H, W = g["hw"]
    T = cfg["num_frames"]
    unet, ad = fixtures.make_models(cfg, seed=0, adapter_gain=20.0)
    vae, clip = fixtures.make_vae_and_clip(cfg["cross_attention_dim"])
    pil = PIL.Image.fromarray(g["image_u8"].numpy())
    flow = fixtures.make_flow(T, H, W)
    lat0 = torch.randn(1, T, 4, H // 8, W // 8, generator=torch.Generator().manual_seed(g["latent_seed"]))
    threads = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    try:
        out = opipe.run_pipeline(vae, clip, unet, ad, osched.EulerDiscreteScheduler(), pil, pil, flow, height=H, width=W,
                                 num_inference_steps=g["steps"], latents=lat0.clone(),
                                 generator=torch.Generator().manual_seed(g["generator_seed"]), output_type="latent",
                                 controlnet_cond_scale=g["cond_scale"])
    finally:
        torch.set_num_threads(threads)
    assert out.shape == g["latents"].shape
    assert (out - g["latents"]).abs().max().item() <= 1e-5 * g["latents"].abs().max().item()


def test_adapter_parameter_names_match_the_reference_training_dump():
    """The reference's Training/rec_para_train.txt is its own dump of `controlnet.named_parameters()` names
    (train_stage1.py:846-856) -- 683 names produced by the REAL diffusers 0.24 blocks.  The oracle adapter (hence
    oracle/d24_blocks.py's module structure: resnets / attentions / transformer_blocks / temporal blocks / mixers) must
    have exactly that name set.  Compared through a digest of that file so no reference file is copied:
    sha256 of its sorted non-empty lines joined by newlines."""
    import hashlib
    from oracle.models import FlowControlNet
    with torch.device("meta"):
        names = sorted(n for n, _ in FlowControlNet().named_parameters())
    assert len(names) == 683
    digest = hashlib.sha256("\n".join(names).encode()).hexdigest()
    assert digest == "dde7b69aad4901bc3ef3bcd4f1301973a7749dd83d6f843e466b3b599d358dd5"


def test_softsplat_oracle_matches_reference_kernel_golden():
    """oracle/softsplat.py vs outputs of the reference's OWN CUDA-C kernel + Python wrapper (softsplat.py:232-335), run on a
    B200 (oracle/make_softsplat_ref.py; fp32 atomics => summation order differs: 1e-5 relative)."""
    import os
    import pytest
    from oracle import make_softsplat_ref as msr
    from oracle.softsplat import softsplat, softsplat_out
    if not os.path.exists(msr.GOLDEN):
        pytest.skip("tests/golden/softsplat_ref.pt not generated yet")
    gold = torch.load(msr.GOLDEN)
    assert len(gold["cases"]) == len(msr.CASES)
    for i, c in enumerate(gold["cases"]):
        x, fl = c["x"].float(), c["flow"].float()
        x2, fl2 = msr.make_case(i)
        assert torch.equal(x, x2) and torch.equal(fl.nan_to_num(7.0, 8.0, 9.0), fl2.nan_to_num(7.0, 8.0, 9.0))
        ones = torch.cat([x, x.new_ones(x.shape[0], 1, x.shape[2], x.shape[3])], 1)
        s = softsplat_out(ones, fl)
        assert (s - c["out_sum"]).abs().max().item() <= 1e-5 * max(1.0, c["out_sum"].abs().max().item()), i
        a = softsplat(x, fl, None, "avg")
        assert (a - c["out_avg"]).abs().max().item() <= 1e-4 * max(1.0, c["out_avg"].abs().max().item()), i
