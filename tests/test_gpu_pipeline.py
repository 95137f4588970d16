"""-m gpu: end-to-end parity of SwinIRPipeline.run (kernel engines, CUDA-graphed sampler) against
the oracle's restatement of the reference pipeline run in fp32 (TF32 off) on the same device with
the same seed (identical RNG consumption: x_T, then one randn_like per step).

Bar (BASELINE.json north_star): PSNR >= 50 dB between the uint8 outputs of the full 50-step run.
"""
import numpy as np
import pytest
import torch

from diffbir_b200 import arch
from diffbir_b200.utils.synth import RUN_DEFAULTS, build_synthetic_pipeline, make_state_dict, synthetic_lq
from tests.gpu_util import no_tf32, to_dev

pytestmark = pytest.mark.gpu


def _oracle_run_with(pipe, lq, kw, **extra):
    return _oracle_run(pipe, lq, True, _extra=extra, **kw)


def _oracle_run(pipe, lq, small, seed=231, _extra=None, **kw):
    """Oracle pipeline on the GPU in fp32 using the same state dicts the product loaded."""
    from oracle import cldm as ocl
    from oracle import sampling as osm
    from oracle import swinir as osw
    dev = "cuda"
    cl = pipe.cldm
    usd, csd, vsd = to_dev(cl._unet_sd), to_dev(cl._cn_sd), to_dev(cl._vae_sd)
    clipsd = to_dev(cl._clip_sd)
    ssd = to_dev({k: v for k, v in pipe.cleaner.engine_sd.items()})
    heads = cl.clip_cfg["text_cfg"]["heads"]
    scales = {"s": [1.0] * 13}

    def model(x, t, cond):
        return ocl.cldm_forward(usd, csd, x, t, cond["c_txt"], cond["c_img"], scales["s"])

    torch.manual_seed(seed)
    taps = {}
    with torch.no_grad():
        out = osm.swinir_pipeline_run(
            lq, cleaner=lambda im: osw.swinir_forward(ssd, im),
            encode_img=lambda im: ocl.vae_encode_mode(vsd, im, cl.scale_factor),
            encode_txt=lambda txt: ocl.clip_text_encode(clipsd, cl.tokenize(txt).to(dev), heads=heads),
            decode=lambda z: ocl.vae_decode(vsd, z / cl.scale_factor), model=model,
            betas=pipe.diffusion.betas, parameterization=pipe.diffusion.parameterization,
            steps=kw["steps"], strength=kw["strength"], pos_prompt=kw["pos_prompt"], neg_prompt=kw["neg_prompt"],
            cfg_scale=kw["cfg_scale"], sampler=kw["sampler_type"], cldm_tiled=kw["cldm_tiled"],
            rescale_cfg=kw["rescale_cfg"],
            cldm_tile_size=kw["cldm_tile_size"], cldm_tile_stride=kw["cldm_tile_stride"], device=dev,
            cleaner_tiled=kw["cleaner_tiled"], cleaner_tile_size=kw["cleaner_tile_size"],
            cleaner_tile_stride=kw["cleaner_tile_stride"],
            set_strength=lambda s: scales.update(s=[s] * 13), taps=taps, **(_extra or {}))
    return out, taps


def _psnr_u8(a, b):
    mse = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).mean()
    return float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


_PIPES = {}


def _pipe(small, v_prediction=False):
    """One synthetic pipeline per architecture size for the whole module (generating 1.3 G random
    weights costs a minute of host time); the diffusion schedule is swapped per test."""
    no_tf32()
    from diffbir_b200.model import Diffusion
    pipe = _PIPES.get(small)
    if pipe is None:
        pipe = build_synthetic_pipeline("cuda", seed=1234, small=small)
        scfg = dict(arch.SWINIR_CFG, depths=(2, 2), num_heads=(6, 6)) if small else arch.SWINIR_CFG
        pipe.cleaner.engine_sd = make_state_dict(arch.swinir_shapes(scfg), 1234 + 4)
        _PIPES[small] = pipe
    pipe.diffusion = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000,
                               parameterization="v" if v_prediction else "eps", zero_snr=v_prediction)
    pipe.taps = {}
    return pipe


def _report(tag, pipe, out, ref, taps):
    zp, zr = pipe.taps["z"], taps["z"]
    e = ((zp - zr).pow(2).mean().sqrt() / zr.pow(2).mean().sqrt()).item()
    p = _psnr_u8(out, ref)
    print(f"{tag}: latent rel-rms {e:.2e}, uint8 PSNR {p:.2f} dB, differing pixels {(out != ref).mean() * 100:.1f}%, "
          f"max |diff| {np.abs(out.astype(int) - ref.astype(int)).max()}, output mean {out.mean():.1f} std {out.std():.1f}")
    return e, p


@pytest.mark.parametrize("sampler,steps,tiled", [("spaced", 10, False), ("ddim", 10, False), ("spaced", 4, True)])
def test_small_pipeline_matches_oracle(sampler, steps, tiled, cleaner_tiled=False):
    pipe = _pipe(True)
    size = 640 if tiled else 512
    lq = synthetic_lq(size, size, seed=1)
    kw = dict(RUN_DEFAULTS, steps=steps, sampler_type=sampler, cldm_tiled=tiled, cleaner_tiled=cleaner_tiled)
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    ref, taps = _oracle_run(pipe, lq, True, **kw)
    zp, zr = pipe.taps["z"], taps["z"]
    e = ((zp - zr).pow(2).mean().sqrt() / zr.pow(2).mean().sqrt()).item()
    p = _psnr_u8(out, ref)
    print(f"small {sampler} x{steps} tiled={tiled} cleaner_tiled={cleaner_tiled}: latent rel-rms {e:.2e}, uint8 PSNR {p:.1f} dB, "
          f"differing pixels {(out != ref).mean() * 100:.1f}%")
    assert out.shape == ref.shape == lq.shape and out.dtype == np.uint8
    assert e < 2e-2 and p > 45.0


@pytest.mark.parametrize("sampler,rescale", [("spaced", False), ("ddim", True)])
def test_small_pipeline_v_prediction(sampler, rescale):
    """v2.1 settings (BASELINE configs[4]): v-parameterization, zero terminal SNR, optional cfg rescale."""
    pipe = _pipe(True, v_prediction=True)
    lq = synthetic_lq(512, 512, seed=2)
    kw = dict(RUN_DEFAULTS, steps=10, sampler_type=sampler, rescale_cfg=rescale)
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    ref, taps = _oracle_run(pipe, lq, True, **kw)
    zp, zr = pipe.taps["z"], taps["z"]
    e = ((zp - zr).pow(2).mean().sqrt() / zr.pow(2).mean().sqrt()).item()
    p = _psnr_u8(out, ref)
    print(f"small v-pred {sampler} rescale={rescale}: latent rel-rms {e:.2e}, uint8 PSNR {p:.1f} dB")
    assert e < 2e-2 and p > 45.0


def test_full_config_50_step_psnr():
    """BASELINE configs[1]: 512x512, 50-step spaced sampler, cfg 4.0, full SD-2.1 UNet + ControlNet."""
    pipe = _pipe(False)
    lq = synthetic_lq(512, 512, seed=0)
    kw = dict(RUN_DEFAULTS)
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    ref, taps = _oracle_run(pipe, lq, False, **kw)
    e, p = _report("FULL 512^2 50-step spaced", pipe, out, ref, taps)
    assert p >= 50.0, f"PSNR {p:.2f} dB < 50 dB vs the fp32 reference path"


def test_small_pipeline_tiled_cleaner():
    """Tiled stage-1 branch (pipeline.py:389-394): 512-pixel Gaussian-blended SwinIR tiles over a 640^2
    image, followed by the tiled stage 2."""
    test_small_pipeline_matches_oracle("spaced", 4, True, cleaner_tiled=True)


def test_full_config_50_step_ddim():
    """BASELINE configs[2]: 512x512, 50-step DDIM (eta 0, batched CFG), full SD-2.1 UNet + ControlNet
    (the BFR face pipeline's stage 2; the face SwinIR has the same architecture, bfr_loop.py:17-23)."""
    pipe = _pipe(False)
    lq = synthetic_lq(512, 512, seed=3)
    kw = dict(RUN_DEFAULTS, sampler_type="ddim")
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    ref, taps = _oracle_run(pipe, lq, False, **kw)
    e, p = _report("FULL 512^2 50-step DDIM", pipe, out, ref, taps)
    assert p >= 50.0, f"PSNR {p:.2f} dB < 50 dB vs the fp32 reference path"


def test_full_config_50_step_ddim_vs_reference_whole_run(golden_dir):
    """BASELINE configs[2] against the REFERENCE itself: tests/golden/full_pipeline_ddim.npz is the uint8 output of the
    reference's SwinIRPipeline.run at the full configuration (gen_golden_full_pipeline.py: same weights, image, prompts,
    50-step DDIM, cfg 4.0, seed 231, CPU fp32). DDIM with eta 0 draws no per-step noise, so feeding the CPU-drawn x_T makes
    the two runs comparable: the north star's "PSNR >= 50 dB vs reference output" without the oracle in between."""
    g = np.load(golden_dir / "full_pipeline_ddim.npz")
    pipe = _pipe(False)
    lq = synthetic_lq(512, 512, seed=3)
    torch.manual_seed(231)
    x_T = torch.randn((1, 4, 64, 64))
    out = pipe.run(lq, **dict(RUN_DEFAULTS, sampler_type="ddim"), x_T=x_T.cuda())
    ref = g["out"]
    p = _psnr_u8(out, ref)
    print(f"FULL 512^2 50-step DDIM vs the reference's own run: uint8 PSNR {p:.2f} dB, differing pixels {(out != ref).mean() * 100:.1f}%, "
          f"max |diff| {np.abs(out.astype(int) - ref.astype(int)).max()}")
    assert out.shape == ref.shape and p >= 50.0


def test_full_config_tiled_1024():
    """BASELINE configs[3] at 1024^2 (the fp32 oracle of 2048^2 x 49 tiles takes too long for a test):
    full SD-2.1 config, latent 128^2 -> 9 tiles of 64^2 (stride 32), 5 steps, Gaussian-blended in the
    reference's order. Single rank; the multi-rank run is bit-identical to it (tests/test_gpu_multi.py)."""
    pipe = _pipe(False)
    lq = synthetic_lq(1024, 1024, seed=4)
    kw = dict(RUN_DEFAULTS, steps=5, cldm_tiled=True, cldm_tile_size=512, cldm_tile_stride=256)
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    ref, taps = _oracle_run(pipe, lq, False, **kw)
    e, p = _report("FULL tiled 1024^2 (9 tiles) 5-step spaced", pipe, out, ref, taps)
    assert e < 1e-2 and p >= 50.0, f"latent rel-rms {e:.2e}, PSNR {p:.2f} dB"


V21_KW = dict(RUN_DEFAULTS, steps=20, pos_prompt="a photo of a mountain lake at sunrise, sharp, highly detailed",
              rescale_cfg=True)


def test_full_config_v21_1024_batch2_fp16_and_bf16(tmp_path):
    """BASELINE configs[4] (v2.1: v-parameterization, zero terminal SNR, caption prompt, cfg rescale) at
    1024^2 (latent 128^2: 16 384-token self-attention), batch 2, full config, 20 spaced steps.
    The default fp16-operand build must clear 50 dB; the bf16-operand build (DBIR_OPERANDS=bf16, what the
    config names) runs in a subprocess on the same input and its PSNR is reported (the reference's own
    bf16 path is 49.55 dB from its fp32 path, SURVEY headline fact 6, so 50 dB is not demanded of it)."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    pipe = _pipe(False, v_prediction=True)
    lq = synthetic_lq(1024, 1024, batch=2, seed=5)
    torch.manual_seed(231)
    out = pipe.run(lq, **V21_KW)
    ref, taps = _oracle_run(pipe, lq, False, **V21_KW)
    e, p = _report("FULL v2.1 1024^2 batch 2, 20-step spaced, fp16 operands", pipe, out, ref, taps)
    assert p >= 50.0, f"PSNR {p:.2f} dB < 50 dB vs the fp32 reference path"
    # bf16-operand build on the same input / seed
    np.save(tmp_path / "ref.npy", ref)
    env = dict(os.environ, DBIR_OPERANDS="bf16", PYTHONPATH=str(root))
    r = subprocess.run([sys.executable, str(root / "tools" / "run_v21_bf16.py"), str(tmp_path / "ref.npy")],
                       capture_output=True, text=True, env=env, timeout=1500)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0
    res = json.loads(r.stdout.strip().splitlines()[-1])
    print(f"bf16-operand build: uint8 PSNR {res['psnr']:.2f} dB vs the fp32 oracle (fp16-operand build: {p:.2f} dB, "
          f"latent rel-rms {e:.2e})")
    assert res["operand_dtype"] == "torch.bfloat16" and res["psnr"] >= 40.0


@pytest.mark.parametrize("sampler,steps,tiled,vpred", [
    ("edm_euler_a", 8, False, False), ("edm_heun", 6, False, False), ("edm_dpm++_2m", 8, True, False),
    ("edm_dpm++_3m_sde", 8, False, True), ("edm_lms", 6, False, False), ("dpm++_m2", 8, False, False), ("dpm++_m2", 6, True, True)])
def test_edm_dpm_samplers_engine_vs_oracle_model(sampler, steps, tiled, vpred):
    """EDM-family / DPM-Solver++ loops on the kernel engine (EngineEval: batched CFG graph replays, tile
    gather / blend, pre-computed embeddings incl. DPM-Solver's fractional times) against the SAME sampler
    code driven by the fp32 oracle network through the plain-PyTorch path. The loops' arithmetic is pinned
    bit-exactly to the reference on the CPU (test_host_logic.py); this checks the engine wiring."""
    from diffbir_b200.sampler import DPMSolverSampler, EDMSampler
    from oracle import cldm as ocl
    pipe = _pipe(True, v_prediction=vpred)
    cl = pipe.cldm
    cl._build()
    usd, csd = to_dev(cl._unet_sd), to_dev(cl._cn_sd)
    B, L = 2, 80 if tiled else 64
    g = torch.Generator().manual_seed(17)
    ctxd = cl.unet_cfg["context_dim"]
    cond = dict(c_txt=torch.randn(B, 77, ctxd, generator=g).cuda(), c_img=torch.randn(B, 4, L, L, generator=g).cuda())
    unc = dict(c_txt=torch.randn(B, 77, ctxd, generator=g).cuda(), c_img=cond["c_img"].clone())
    xT = torch.randn(B, 4, L, L, generator=g).cuda()
    param = pipe.diffusion.parameterization

    def make():
        if sampler.startswith("edm"):
            return EDMSampler(pipe.diffusion.betas, param, False, sampler, s_churn=0.4, s_tmin=0, s_tmax=300, s_noise=1, eta=1, order=4)
        return DPMSolverSampler(pipe.diffusion.betas, param, False, sampler)

    def oracle_model(x, t, c):
        return ocl.cldm_forward(usd, csd, x, t, c["c_txt"], c["c_img"], [1.0] * 13)

    kw = dict(tiled=tiled, tile_size=64, tile_stride=16)
    torch.manual_seed(5)
    z = make().sample(cl, "cuda", steps, (B, 4, L, L), cond, unc, 4.0, x_T=xT, **kw)
    torch.manual_seed(5)
    with torch.no_grad():
        zr = make().sample(oracle_model, "cuda", steps, (B, 4, L, L), cond, unc, 4.0, x_T=xT, **kw)
    e = ((z - zr).pow(2).mean().sqrt() / zr.pow(2).mean().sqrt()).item()
    print(f"{sampler} x{steps} tiled={tiled} v={vpred}: latent rel-rms {e:.2e} (|z| {zr.abs().mean():.3f})")
    assert torch.isfinite(z).all() and e < 2e-2


def test_small_bsrnet_pipeline_matches_oracle():
    """v2 blind-SR recipe: BSRNetPipeline (RRDBNet x4 stage 1 on the LQ image, pipeline.py:324-366) + the reduced
    stage 2, against the oracle's restatement with the same seed."""
    from diffbir_b200.model import RRDBNet
    from diffbir_b200.pipeline import BSRNetPipeline
    from oracle import bsrnet as ob
    from tests.small_cfg import RRDB_SMALL
    pipe0 = _pipe(True)
    rsd = make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 91)
    net = RRDBNet(**RRDB_SMALL, device="cuda")
    net.load_state_dict(rsd)
    pipe = BSRNetPipeline(net, pipe0.cldm, pipe0.diffusion, None, "cuda", upscale=4.0)
    pipe.taps = {}
    lq = synthetic_lq(128, 160, seed=3)
    kw = dict(RUN_DEFAULTS, steps=6)
    torch.manual_seed(231)
    out = pipe.run(lq, **kw)
    rsd_d = to_dev(rsd)
    pipe0.taps = pipe.taps                       # _oracle_run reads the product taps of `pipe`
    ref, taps = _oracle_run_with(pipe0, lq, kw, stage1=lambda im: ob.bsrnet_apply_cleaner(lambda t: ob.rrdbnet_forward(rsd_d, t), im, 4.0),
                                 out_size=(512, 640))
    e = ((pipe.taps["z"] - taps["z"]).pow(2).mean().sqrt() / taps["z"].pow(2).mean().sqrt()).item()
    p = _psnr_u8(out, ref)
    print(f"small BSRNet pipeline x6: latent rel-rms {e:.2e}, uint8 PSNR {p:.1f} dB, output {out.shape}")
    assert out.shape == ref.shape == (1, 512, 640, 3) and out.dtype == np.uint8
    assert e < 2e-2 and p > 45.0


@pytest.mark.parametrize("case", ["swinir_ddim", "bsrnet_edm", "scunet_dpm"])
def test_small_pipeline_vs_reference_whole_run(golden_dir, case):
    """Product vs the REFERENCE itself, end to end: the uint8 output of the reference's {SwinIR,BSRNet,SCUNet}Pipeline.run
    on the reduced networks (tests/golden/pipeline_small.npz, produced on the CPU by gen_golden_pipeline.py) against the
    same pipeline class of this package on the same weights, input and x_T. The three samplers (DDIM eta 0, EDM dpm++_2m,
    DPM-Solver++ m2) consume no per-step noise, so the CPU-drawn x_T (first draw after the seed, pipeline.py:150-158) is
    the only randomness and can be injected."""
    from diffbir_b200.model import RRDBNet, SCUNet
    from diffbir_b200.pipeline import BSRNetPipeline, SCUNetPipeline
    from tests.small_cfg import RRDB_SMALL, SCUNET_SMALL
    g = np.load(golden_dir / "pipeline_small.npz")
    if case == "swinir_ddim":
        pipe = _pipe(True, v_prediction=True)
        lq, ref, L, kw = g["lq"], g["out_ddim_v"], (64, 88), dict(steps=4, sampler_type="ddim")     # 96 x 128 -> 512 x 683 -> padded 512 x 704
    elif case == "bsrnet_edm":
        p0 = _pipe(True, v_prediction=True)
        net = RRDBNet(**RRDB_SMALL, device="cuda")
        net.load_state_dict(make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 91))
        pipe = BSRNetPipeline(net, p0.cldm, p0.diffusion, None, "cuda", upscale=4.0)
        lq, ref, L, kw = g["lq_bsr"], g["out_bsrnet"], (64, 80), dict(steps=6, sampler_type="edm_dpm++_2m")
    else:
        p0 = _pipe(True, v_prediction=False)
        net = SCUNet(**SCUNET_SMALL, device="cuda")
        net.load_state_dict(make_state_dict(arch.scunet_shapes(SCUNET_SMALL), 9))
        pipe = SCUNetPipeline(net, p0.cldm, p0.diffusion, None, "cuda")
        lq, ref, L, kw = g["lq"], g["out_scunet"], (64, 88), dict(steps=6, sampler_type="dpm++_m2")
    pipe.taps = {}
    torch.manual_seed(231)
    x_T = torch.randn((1, 4) + L)
    out = pipe.run(lq, **dict(RUN_DEFAULTS, pos_prompt="a photo", **kw), x_T=x_T.cuda())
    p = _psnr_u8(out, ref)
    print(f"product vs reference whole run [{case}] (reduced nets): uint8 PSNR {p:.1f} dB, "
          f"differing pixels {(out != ref).mean() * 100:.1f}%, max |diff| {np.abs(out.astype(int) - ref.astype(int)).max()}")
    assert out.shape == ref.shape and p > 45.0
