"""Pins the oracle (oracle/*.py, a restatement) against fixtures produced by the reference
implementation itself (tests/golden/gen_golden.py). CPU only."""
import numpy as np
import torch

from diffbir_b200 import arch
from diffbir_b200.utils.synth import make_state_dict
from oracle import cldm as ocl
from oracle import sampling as osm
from oracle import swinir as osw
from tests.small_cfg import CN_SMALL, SWIN_SMALL, UNET_SMALL, VAE_SMALL


def close(a, b, rtol=2e-5):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item() / scale
    assert err < rtol, f"max rel-to-max err {err:.3e}"


def test_cldm_forward_matches_reference(golden_dir):
    g = np.load(golden_dir / "cldm_small.npz")
    usd = make_state_dict(arch.unet_shapes(UNET_SMALL), 1, arch.is_zero_init)
    csd = make_state_dict(arch.unet_shapes(CN_SMALL, True), 2, arch.is_zero_init)
    x, hint, ctx = (torch.from_numpy(g[k]) for k in ("x", "hint", "ctx"))
    t = torch.from_numpy(g["t"])
    with torch.no_grad():
        control = ocl.controlnet_forward(csd, x, hint, t, ctx)
        close(control[0], g["control0"])
        close(control[12], g["control12"])
        eps = ocl.cldm_forward(usd, csd, x, t, ctx, hint, list(g["scales"]))
    close(eps, g["eps"])


def test_vae_matches_reference(golden_dir):
    g = np.load(golden_dir / "vae_small.npz")
    sd = make_state_dict(arch.vae_shapes(VAE_SMALL), 3)
    with torch.no_grad():
        close(ocl.vae_decode(sd, torch.from_numpy(g["z"])), g["dec"])
        close(ocl.vae_encode_moments(sd, torch.from_numpy(g["img"])), g["moments"])


def test_swinir_matches_reference(golden_dir):
    g = np.load(golden_dir / "swinir_small.npz")
    sd = make_state_dict(arch.swinir_shapes(SWIN_SMALL), 4)
    with torch.no_grad():
        y = osw.swinir_forward(sd, torch.from_numpy(g["x"]))
    ref = torch.from_numpy(g["y"])
    assert y.shape == ref.shape
    # compare against the signal's own spread (random-init output is nearly constant)
    err = (y - ref).abs().max().item() / ref.std().item()
    assert err < 1e-3, err


def test_schedules_match_reference(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    for name, zero_snr in (("eps", False), ("v", True)):
        betas = osm.make_betas(zero_snr=zero_snr)
        np.testing.assert_allclose(betas, g[f"betas_{name}"], rtol=1e-12, atol=1e-15)
        betas = g[f"betas_{name}"]
        with np.errstate(divide="ignore"):
            tb = osm.spaced_tables(betas, 50)
        assert (tb["timesteps"] == g[f"spaced_ts_{name}"]).all()
        for k in ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
                  "posterior_mean_coef1", "posterior_mean_coef2", "sqrt_alphas_cumprod",
                  "sqrt_one_minus_alphas_cumprod"):
            np.testing.assert_array_equal(tb[k].astype(np.float32), g[f"spaced_{k}_{name}"])
        td = osm.ddim_tables(betas, 50)
        assert (td["timesteps"] == g[f"ddim_ts_{name}"]).all()
        np.testing.assert_array_equal(td["alphas"].astype(np.float32), g[f"ddim_alphas_{name}"])
        np.testing.assert_array_equal(td["alphas_prev"].astype(np.float32), g[f"ddim_alphas_prev_{name}"])
        np.testing.assert_array_equal(td["sqrt_one_minus_alphas"].astype(np.float32),
                                      g[f"ddim_sqrt_one_minus_alphas_{name}"])


def _stub(x, t, cond):
    return (0.3 * torch.tanh(x) + 0.05 * cond["c_img"]
            + 0.01 * cond["c_txt"].mean(dim=(1, 2)).view(-1, 1, 1, 1)
            + 1e-4 * t.float().view(-1, 1, 1, 1))


def test_sampler_trajectories_bit_exact(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    xT = torch.from_numpy(g["xT"])
    cond = dict(c_txt=torch.from_numpy(g["cond_c_txt"]), c_img=torch.from_numpy(g["cond_c_img"]))
    uncond = dict(c_txt=torch.from_numpy(g["uncond_c_txt"]), c_img=torch.from_numpy(g["uncond_c_img"]))
    noises = [torch.from_numpy(n) for n in g["noises"]]
    for name in ("eps", "v"):
        betas = g[f"betas_{name}"]
        for sname, fn in (("spaced", osm.spaced_sample), ("ddim", osm.ddim_sample)):
            for tiled in (False, True):
                with np.errstate(divide="ignore"):
                    z = fn(_stub, betas, name, 10, xT.clone(), cond, uncond, 4.0, noises=noises,
                           tiled=tiled, tile_size=16, tile_stride=8)
                ref = g[f"traj_{sname}_{name}_{'tiled' if tiled else 'full'}"]
                np.testing.assert_array_equal(z.numpy(), ref, err_msg=f"{sname} {name} tiled={tiled}")


def test_tiling_and_colour_fix(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    np.testing.assert_array_equal(osm.gaussian_weights(16, 16), g["gauss_16"])
    assert (np.array(osm.sliding_windows(24, 40, 16, 8)) == g["windows_24_40_16_8"]).all()
    assert (np.array(osm.sliding_windows(30, 30, 16, 12)) == g["windows_30_30_16_12"]).all()
    a, b = torch.from_numpy(g["wavelet_a"]), torch.from_numpy(g["wavelet_b"])
    np.testing.assert_allclose(osm.wavelet_reconstruction(a, b).numpy(), g["wavelet_out"], atol=1e-6)
    np.testing.assert_array_equal(osm.resize_short_edge(a, 64).numpy(), g["resize_out"])


def test_tiled_image_fn_and_tiled_cleaner_match_reference():
    """Image tiling wrapper + the tiled stage-1 branch: oracle AND product host code against the
    fixture produced by the reference (tests/golden/gen_golden_tiled_fn.py), bit-exact on CPU."""
    from oracle import sampling as osm
    from diffbir_b200.pipeline import SwinIRPipeline
    from diffbir_b200.utils.common import make_tiled_fn
    from pathlib import Path
    import pytest
    g = np.load(Path(__file__).resolve().parent / "golden" / "tiled_fn.npz")

    def stand_in(t):
        return torch.tanh(t) * 0.5 + t.mean(dim=(2, 3), keepdim=True) * 0.25

    x = torch.tensor(g["x"])
    for size, stride in ((32, 16), (40, 24)):
        ref = g[f"tiled_{size}_{stride}"]
        np.testing.assert_array_equal(osm.make_tiled_image_fn(stand_in, size, stride)(x).numpy(), ref)
        np.testing.assert_array_equal(make_tiled_fn(stand_in, size, stride)(x).numpy(), ref)
    lq = torch.tensor(g["lq"])
    pipe = SwinIRPipeline(stand_in, None, None, None, "cpu")
    for name, inp in (("cleaner_tiled_128_64", lq), ("cleaner_tiny_untiled", lq[..., :100, :90])):
        for out in (osm.apply_cleaner(stand_in, inp, True, 128, 64), pipe.apply_cleaner(inp, True, 128, 64)):
            assert tuple(out.shape) == tuple(g[name + "_shape"])
            np.testing.assert_array_equal(out[..., ::8, ::8].numpy(), g[name + "_sub8"])
    with pytest.raises(ValueError):
        pipe.apply_cleaner(torch.zeros(1, 3, 256, 256), True, 100, 50)
    # x4 up-scaling tiles and the tiled branches of BSRNetPipeline (both output-size regimes) and SCUNetPipeline
    from diffbir_b200.pipeline import BSRNetPipeline, SCUNetPipeline

    def stand_in_up4(t):
        return torch.nn.functional.interpolate(stand_in(t), scale_factor=4, mode="bilinear", align_corners=False)

    ref = g["tiled_up4_24_16_sub4"]
    np.testing.assert_array_equal(make_tiled_fn(stand_in_up4, 24, 16, scale_type="up", scale=4)(x)[..., ::4, ::4].numpy(), ref)
    np.testing.assert_array_equal(osm.make_tiled_image_fn(stand_in_up4, 24, 16, scale=4)(x)[..., ::4, ::4].numpy(), ref)
    for scale, key in ((2.0, "bsr_tiled_small"), (4.0, "bsr_tiled_big")):
        bp = BSRNetPipeline(stand_in_up4, None, None, None, "cpu", upscale=scale)
        bp.set_output_size(lq.size())
        y = bp.apply_cleaner(lq, True, 64, 48)
        assert tuple(y.shape) == tuple(g[key + "_shape"])
        np.testing.assert_array_equal(y[..., ::8, ::8].numpy(), g[key + "_sub8"])
    y = SCUNetPipeline(stand_in, None, None, None, "cpu").apply_cleaner(lq, True, 64, 48)
    assert tuple(y.shape) == tuple(g["scunet_tiled_shape"])
    np.testing.assert_array_equal(y[..., ::8, ::8].numpy(), g["scunet_tiled_sub8"])


def test_clip_text_tower_matches_reference(golden_dir):
    """OpenCLIP text tower (penultimate layer, causal mask): the oracle's restatement AND the product's
    TextTower (plain torch, run here on CPU) against the reference's FrozenOpenCLIPEmbedder output."""
    from diffbir_b200.model.clip import TextTower
    from tests.small_cfg import CLIP_SMALL
    g = np.load(golden_dir / "clip_small.npz")
    sd = make_state_dict(arch.clip_text_shapes(CLIP_SMALL), 7)
    tokens = torch.tensor(g["tokens"])
    ref = torch.tensor(g["out"])
    with torch.no_grad():
        o = ocl.clip_text_encode(sd, tokens, heads=CLIP_SMALL["heads"])
        p = TextTower(sd, heads=CLIP_SMALL["heads"], layer="penultimate", device="cpu")(tokens)
    assert (o - ref).abs().max() < 2e-5 * ref.abs().max()
    assert (p - ref).abs().max() < 2e-5 * ref.abs().max()


def test_q_sample_matches_reference(golden_dir):
    """Diffusion.q_sample (start point "cond", noise augmentation): oracle and product, bit-exact."""
    from diffbir_b200.model import Diffusion
    g = np.load(golden_dir / "qsample.npz")
    x0, noise, t = torch.tensor(g["x0"]), torch.tensor(g["noise"]), torch.tensor(g["t"])
    for name, kw in (("eps", {}), ("v", dict(parameterization="v", zero_snr=True))):
        d = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, **kw)
        np.testing.assert_array_equal(d.q_sample(x0, t, noise).numpy(), g[f"q_{name}"])
        np.testing.assert_array_equal(osm.q_sample(osm.make_betas(zero_snr=bool(kw)), x0, t, noise).numpy(), g[f"q_{name}"])


def test_rrdbnet_and_bsrnet_cleaner_match_reference(golden_dir):
    """oracle.bsrnet (RRDBNet forward, BSRNetPipeline.apply_cleaner) and the product's BSRNetPipeline host code
    (driven by the oracle network on the CPU) against a fixture the reference produced: bit-exact."""
    from diffbir_b200.pipeline import BSRNetPipeline
    from oracle import bsrnet as ob
    from tests.small_cfg import RRDB_SMALL
    g = np.load(golden_dir / "bsrnet_small.npz")
    sd = make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 7)
    net = lambda im: ob.rrdbnet_forward(sd, im)               # noqa: E731
    lq = torch.from_numpy(g["lq"])
    with torch.no_grad():
        np.testing.assert_array_equal(net(torch.from_numpy(g["x"])).numpy(), g["y"])
        for scale, key in ((4.0, "cond_small"), (45.0, "cond_big")):
            a = ob.bsrnet_apply_cleaner(net, lq, scale)
            assert tuple(a.shape) == tuple(g[key + "_shape"])
            np.testing.assert_array_equal(a[..., ::6, ::6].numpy(), g[key])
            pipe = BSRNetPipeline(net, None, None, None, "cpu", upscale=scale)
            pipe.set_output_size(lq.size())
            b = pipe.apply_cleaner(lq, False, 512, 256)
            np.testing.assert_array_equal(b.numpy(), a.numpy())


def test_scunet_matches_reference(golden_dir):
    """oracle.scunet (SCUNet.forward incl. the replicate pad / crop and both block types) against a fixture the
    reference module produced, bit-exact; SCUNetPipeline's host code on top of it."""
    from diffbir_b200.pipeline import SCUNetPipeline
    from oracle import scunet as osc
    from tests.small_cfg import SCUNET_SMALL
    g = np.load(golden_dir / "scunet_small.npz")
    sd = make_state_dict(arch.scunet_shapes(SCUNET_SMALL), 9)
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        y = osc.scunet_forward(sd, x)
        np.testing.assert_array_equal(y.numpy(), g["y"])
        net = lambda im: osc.scunet_forward(sd, im)           # noqa: E731
        pipe = SCUNetPipeline(net, None, None, None, "cpu")
        a, b = pipe.apply_cleaner(x, False, 512, 256), osc.scunet_apply_cleaner(net, x)
        assert a.shape[2:] == (853, 512) and torch.equal(a, b)


def test_whole_pipeline_matches_reference_run(golden_dir):
    """The oracle's restatement of SwinIRPipeline.run (stage 1, resize, VAE encode, text tower, CFG sampler loop,
    VAE decode, wavelet colour fix, resize back, uint8 truncation) against the uint8 output of the REFERENCE's own
    `Pipeline.run` on the reduced networks (tests/golden/gen_golden_pipeline.py): spaced / eps and DDIM / v + zero SNR."""
    from diffbir_b200.model import Diffusion
    from diffbir_b200.model.clip import SyntheticTokenizer
    from diffbir_b200.utils.synth import synthetic_sd_checkpoint
    from tests.small_cfg import CLIP_SMALL
    g = np.load(golden_dir / "pipeline_small.npz")
    sd = synthetic_sd_checkpoint(UNET_SMALL, VAE_SMALL, CLIP_SMALL, 1234)
    usd = {k[len("model.diffusion_model."):]: v for k, v in sd.items() if k.startswith("model.diffusion_model.")}
    vsd = {k[len("first_stage_model."):]: v for k, v in sd.items() if k.startswith("first_stage_model.")}
    clipsd = {k[len("cond_stage_model.model."):]: v for k, v in sd.items() if k.startswith("cond_stage_model.model.")}
    csd = make_state_dict(arch.unet_shapes(CN_SMALL, True), 1237, arch.is_zero_init)
    ssd = make_state_dict(arch.swinir_shapes(SWIN_SMALL), 1238)
    tok = SyntheticTokenizer(CLIP_SMALL["vocab_size"])
    scales = {"s": [1.0] * 13}
    neg = "low quality, blurry, low-resolution, noisy, unsharp, weird textures"
    for sampler, steps, pname, zs in (("spaced", 3, "eps", False), ("ddim", 4, "v", True)):
        d = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, parameterization=pname, zero_snr=zs)
        torch.manual_seed(231)
        with torch.no_grad():
            out = osm.swinir_pipeline_run(
                g["lq"], cleaner=lambda im: osw.swinir_forward(ssd, im), encode_img=lambda im: ocl.vae_encode_mode(vsd, im, 0.18215),
                encode_txt=lambda txt: ocl.clip_text_encode(clipsd, tok(txt), heads=CLIP_SMALL["heads"]),
                decode=lambda z: ocl.vae_decode(vsd, z / 0.18215),
                model=lambda x, t, c: ocl.cldm_forward(usd, csd, x, t, c["c_txt"], c["c_img"], scales["s"]),
                betas=d.betas, parameterization=pname, steps=steps, strength=1.0, pos_prompt="a photo", neg_prompt=neg,
                cfg_scale=4.0, sampler=sampler, set_strength=lambda s: scales.update(s=[s] * 13))
        ref = g[f"out_{sampler}_{pname}"]
        diff = np.abs(out.astype(int) - ref.astype(int))
        mse = (diff.astype(np.float64) ** 2).mean()
        psnr = float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        print(f"whole pipeline {sampler}/{pname}: {100 * (diff > 0).mean():.3f} % of pixels differ, max |diff| {diff.max()}, PSNR {psnr:.1f} dB")
        assert out.shape == ref.shape and diff.max() <= 1 and psnr > 70.0


def test_whole_bsrnet_and_scunet_pipelines_match_reference_run(golden_dir):
    """The two other stage-1 pipelines with the two other sampler families, end to end against the reference's own
    uint8 output: BSRNetPipeline + EDM dpm++_2m (v, zero SNR) and SCUNetPipeline + DPM-Solver++ m2 (eps). Networks are
    the oracle's; the sampler loops are the product's host code (itself bit-exact vs the reference, test_host_logic.py)
    driving the oracle network on the CPU."""
    from diffbir_b200.model import Diffusion
    from diffbir_b200.model.clip import SyntheticTokenizer
    from diffbir_b200.sampler import DPMSolverSampler, EDMSampler
    from diffbir_b200.utils.synth import synthetic_sd_checkpoint
    from oracle import bsrnet as ob
    from oracle import scunet as osc
    from tests.small_cfg import CLIP_SMALL, RRDB_SMALL, SCUNET_SMALL
    g = np.load(golden_dir / "pipeline_small.npz")
    sd = synthetic_sd_checkpoint(UNET_SMALL, VAE_SMALL, CLIP_SMALL, 1234)
    usd = {k[len("model.diffusion_model."):]: v for k, v in sd.items() if k.startswith("model.diffusion_model.")}
    vsd = {k[len("first_stage_model."):]: v for k, v in sd.items() if k.startswith("first_stage_model.")}
    clipsd = {k[len("cond_stage_model.model."):]: v for k, v in sd.items() if k.startswith("cond_stage_model.model.")}
    csd = make_state_dict(arch.unet_shapes(CN_SMALL, True), 1237, arch.is_zero_init)
    rsd = make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 91)
    scsd = make_state_dict(arch.scunet_shapes(SCUNET_SMALL), 9)
    tok = SyntheticTokenizer(CLIP_SMALL["vocab_size"])
    neg = "low quality, blurry, low-resolution, noisy, unsharp, weird textures"
    cases = (("bsrnet", "lq_bsr", "edm_dpm++_2m", "v", True, (512, 640),
              lambda im: ob.bsrnet_apply_cleaner(lambda t: ob.rrdbnet_forward(rsd, t), im, 4.0)),
             ("scunet", "lq", "dpm++_m2", "eps", False, None,
              lambda im: osc.scunet_apply_cleaner(lambda t: osc.scunet_forward(scsd, t), im)))
    for tag, lqk, sampler, pname, zs, out_size, stage1 in cases:
        d = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, parameterization=pname, zero_snr=zs)

        def sample_fn(model, x_T, cond, uncond):
            if sampler.startswith("edm"):
                smp = EDMSampler(d.betas, pname, False, sampler, 0, 0, 300, 1, 1, 1)
            else:
                smp = DPMSolverSampler(d.betas, pname, False, sampler)
            return smp.sample(model, "cpu", 6, tuple(x_T.shape), cond, uncond, 4.0, x_T=x_T, progress=False)

        torch.manual_seed(231)
        with torch.no_grad():
            out = osm.swinir_pipeline_run(
                g[lqk], cleaner=None, encode_img=lambda im: ocl.vae_encode_mode(vsd, im, 0.18215),
                encode_txt=lambda txt: ocl.clip_text_encode(clipsd, tok(txt), heads=CLIP_SMALL["heads"]),
                decode=lambda z: ocl.vae_decode(vsd, z / 0.18215),
                model=lambda x, t, c: ocl.cldm_forward(usd, csd, x, t, c["c_txt"], c["c_img"], [1.0] * 13),
                betas=d.betas, parameterization=pname, steps=6, strength=1.0, pos_prompt="a photo", neg_prompt=neg,
                cfg_scale=4.0, stage1=stage1, out_size=out_size, sample_fn=sample_fn)
        ref = g[f"out_{tag}"]
        diff = np.abs(out.astype(int) - ref.astype(int))
        mse = (diff.astype(np.float64) ** 2).mean()
        psnr = float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        print(f"whole {tag} pipeline {sampler}/{pname}: {100 * (diff > 0).mean():.3f} % of pixels differ, max |diff| {diff.max()}, PSNR {psnr:.1f} dB")
        assert out.shape == ref.shape and diff.max() <= 1 and psnr > 70.0


def _rel_rms(a, b):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def test_full_config_oracle_matches_reference(golden_dir):
    """The oracle at FULL width (real SD-2.1 UNet + ControlNet, full VAE / SwinIR / RRDBNet / SCUNet of
    configs/inference/*.yaml) against outputs of the reference's own modules on the weights and inputs of the full-config
    GPU tests (tests/golden/gen_golden_full.py): the reference == oracle == CUDA chain is closed at full width too."""
    from oracle import bsrnet as ob
    from oracle import scunet as osc
    g = {k: v for f in ("full_config", "full_config_vae", "full_config_swinir") for k, v in np.load(golden_dir / f"{f}.npz").items()}
    res = {}
    with torch.no_grad():
        usd = make_state_dict(arch.unet_shapes(arch.UNET_CFG), 1234, arch.is_zero_init)
        csd = make_state_dict(arch.unet_shapes(arch.CONTROLNET_CFG, True), 1235, arch.is_zero_init)
        gen = torch.Generator().manual_seed(0)
        x = torch.randn(1, 4, 64, 64, generator=gen).repeat(2, 1, 1, 1)
        hint = (torch.randn(1, 4, 64, 64, generator=gen) * 0.5).repeat(2, 1, 1, 1)
        ctx = torch.randn(2, 77, 1024, generator=gen)
        eps = ocl.cldm_forward(usd, csd, x, torch.full((2,), 500), ctx, hint, [1.0] * 13)
        res["cldm t=500"] = _rel_rms(eps, g["cldm_eps_t500"])
        del usd, csd
        vsd = make_state_dict(arch.vae_shapes(arch.VAE_CFG), 77)
        gen = torch.Generator().manual_seed(31)
        z16 = torch.randn(1, 4, 16, 16, generator=gen)
        img128 = torch.rand(1, 3, 128, 128, generator=gen) * 2 - 1
        res["vae decode 16"] = _rel_rms(ocl.vae_decode(vsd, z16), g["vae_dec16"])
        res["vae encode 128"] = _rel_rms(ocl.vae_encode_moments(vsd, img128), g["vae_moments128"])
        ssd = make_state_dict(arch.swinir_shapes(arch.SWINIR_CFG), 1234)
        xs = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(0))
        res["swinir 256"] = _rel_rms(osw.swinir_forward(ssd, xs), g["swinir_y256"])
        rsd = make_state_dict(arch.rrdbnet_shapes(arch.RRDBNET_CFG), 78)
        xr = torch.rand(1, 3, 128, 160, generator=torch.Generator().manual_seed(4))
        s = int(g["rrdb_stride"])
        res["rrdbnet 128x160"] = _rel_rms(ob.rrdbnet_forward(rsd, xr)[..., ::s, ::s], g["rrdb_y"])
        scsd = make_state_dict(arch.scunet_shapes(arch.SCUNET_CFG), 79)
        xc = torch.rand(1, 3, 256, 320, generator=torch.Generator().manual_seed(6))
        s = int(g["scunet_stride"])
        res["scunet 256x320"] = _rel_rms(osc.scunet_forward(scsd, xc)[..., ::s, ::s], g["scunet_y"])
    print("full-config oracle vs reference (rel. RMS): " + ", ".join(f"{k} {v:.1e}" for k, v in res.items()))
    assert max(res.values()) < 2e-5, res


class _OracleCldm:
    """The ControlLDM surface Pipeline.apply_cldm and the samplers use (prepare_condition_pair, vae_decode,
    control_scales, the model call), backed by the oracle networks on the CPU: lets the PRODUCT's pipeline / sampler host
    code run without the GPU library."""

    def __init__(self, usd, csd, vsd, clipsd, tok, heads):
        self.usd, self.csd, self.vsd, self.clipsd, self.tok, self.heads = usd, csd, vsd, clipsd, tok, heads
        self.control_scales = [1.0] * 13
        self.shard_vae = False

    def _txt(self, prompts):
        return ocl.clip_text_encode(self.clipsd, self.tok(prompts), heads=self.heads)

    def prepare_condition_pair(self, cond_img, pos, neg):
        c_img = ocl.vae_encode_mode(self.vsd, cond_img * 2 - 1, 0.18215)
        return dict(c_txt=self._txt(pos), c_img=c_img), dict(c_txt=self._txt(neg), c_img=c_img.clone())

    def vae_decode(self, z):
        return ocl.vae_decode(self.vsd, z / 0.18215)

    def __call__(self, x, t, cond):
        return ocl.cldm_forward(self.usd, self.csd, x, t, cond["c_txt"], cond["c_img"], self.control_scales)


def test_product_pipeline_host_code_matches_reference_run(golden_dir):
    """The PRODUCT's Pipeline.run / apply_cleaner / apply_cldm and sampler classes (the host code that ships), with the
    oracle networks plugged in where the kernel engines sit, against the uint8 output of whole runs of the reference:
    all three pipeline classes, all four sampler families, incl. the RNG draw order (x_T, per-step noise), the optional
    branches (start point "cond", noise augmentation, control strength, CFG ramp) and both tiled modes."""
    from diffbir_b200.model import Diffusion
    from diffbir_b200.model.clip import SyntheticTokenizer
    from diffbir_b200.pipeline import BSRNetPipeline, SCUNetPipeline, SwinIRPipeline
    from diffbir_b200.utils.synth import RUN_DEFAULTS, synthetic_sd_checkpoint
    from oracle import bsrnet as ob
    from oracle import scunet as osc
    from tests.small_cfg import CLIP_SMALL, RRDB_SMALL, SCUNET_SMALL
    g = np.load(golden_dir / "pipeline_small.npz")
    sd = synthetic_sd_checkpoint(UNET_SMALL, VAE_SMALL, CLIP_SMALL, 1234)
    part = lambda pre: {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}      # noqa: E731
    cldm = _OracleCldm(part("model.diffusion_model."), make_state_dict(arch.unet_shapes(CN_SMALL, True), 1237, arch.is_zero_init),
                       part("first_stage_model."), part("cond_stage_model.model."), SyntheticTokenizer(CLIP_SMALL["vocab_size"]),
                       CLIP_SMALL["heads"])
    ssd = make_state_dict(arch.swinir_shapes(SWIN_SMALL), 1238)
    rsd = make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 91)
    scsd = make_state_dict(arch.scunet_shapes(SCUNET_SMALL), 9)
    swin = lambda im: osw.swinir_forward(ssd, im)                  # noqa: E731
    cases = (("out_spaced_eps", "lq", "spaced", 3, "eps", False, lambda d: SwinIRPipeline(swin, cldm, d, None, "cpu")),
             ("out_ddim_v", "lq", "ddim", 4, "v", True, lambda d: SwinIRPipeline(swin, cldm, d, None, "cpu")),
             ("out_bsrnet", "lq_bsr", "edm_dpm++_2m", 6, "v", True,
              lambda d: BSRNetPipeline(lambda im: ob.rrdbnet_forward(rsd, im), cldm, d, None, "cpu", upscale=4.0)),
             ("out_scunet", "lq", "dpm++_m2", 6, "eps", False,
              lambda d: SCUNetPipeline(lambda im: osc.scunet_forward(scsd, im), cldm, d, None, "cpu")))
    cases = tuple(c + ({},) for c in cases) + (
        # optional branches: start point "cond", noise-augmented condition, control strength, cosine CFG ramp
        ("out_opts", "lq", "spaced", 3, "eps", False, lambda d: SwinIRPipeline(swin, cldm, d, None, "cpu"),
         dict(start_point_type="cond", noise_aug=40, rescale_cfg=True, strength=0.7)),
        # Tiled-VAE flags with tiles larger than the image: un-tiled VAE, but the condition is padded to 8 instead of 64
        ("out_vaetiny", "lq", "spaced", 3, "eps", False, lambda d: SwinIRPipeline(swin, cldm, d, None, "cpu"),
         dict(vae_encoder_tiled=True, vae_encoder_tile_size=1024, vae_decoder_tiled=True, vae_decoder_tile_size=1024)),
        # both tiled modes: Gaussian-blended stage-1 tiles, mixture-of-diffusers latent tiles
        ("out_tiled", "lq", "ddim", 4, "v", True, lambda d: SwinIRPipeline(swin, cldm, d, None, "cpu"),
         dict(cleaner_tiled=True, cleaner_tile_size=64, cleaner_tile_stride=32, cldm_tiled=True, cldm_tile_size=512, cldm_tile_stride=256)))
    for key, lqk, sampler, steps, pname, zs, make, over in cases:
        pipe = make(Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, parameterization=pname, zero_snr=zs))
        torch.manual_seed(231)
        with torch.no_grad():
            out = pipe.run(g[lqk], **dict(RUN_DEFAULTS, steps=steps, sampler_type=sampler, pos_prompt="a photo", **over))
        ref = g[key]
        diff = np.abs(out.astype(int) - ref.astype(int))
        mse = (diff.astype(np.float64) ** 2).mean()
        psnr = float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        print(f"product host code, {type(pipe).__name__} + {sampler}/{pname} {over or ''}: {100 * (diff > 0).mean():.3f} % of pixels differ, "
              f"max |diff| {diff.max()}, PSNR {psnr:.1f} dB")
        assert out.shape == ref.shape and diff.max() <= 1 and psnr > 70.0
        assert cldm.control_scales == [1.0] * 13            # restored after the run (pipeline.py:232)
