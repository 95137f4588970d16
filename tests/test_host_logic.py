"""CPU tests of the host-side product code: schedules / samplers (bit-exact against the
reference goldens through the generic model path), tiling helpers, architecture tables,
synthetic checkpoints, GEGLU packing, and the C-ABI surface (library loads and exports every
symbol declared in include/diffbir_b200.h — no compute without a GPU)."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from diffbir_b200 import arch
from diffbir_b200.model import Diffusion
from diffbir_b200.sampler import DDIMSampler, SpacedSampler
from diffbir_b200.utils import common as uc
from diffbir_b200.utils.synth import make_state_dict

ROOT = Path(__file__).resolve().parents[1]


def _stub(x, t, cond):
    return (0.3 * torch.tanh(x) + 0.05 * cond["c_img"]
            + 0.01 * cond["c_txt"].mean(dim=(1, 2)).view(-1, 1, 1, 1) + 1e-4 * t.float().view(-1, 1, 1, 1))


def test_samplers_bit_exact_vs_reference(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    xT = torch.from_numpy(g["xT"])
    cond = dict(c_txt=torch.from_numpy(g["cond_c_txt"]), c_img=torch.from_numpy(g["cond_c_img"]))
    unc = dict(c_txt=torch.from_numpy(g["uncond_c_txt"]), c_img=torch.from_numpy(g["uncond_c_img"]))
    for name, zs in (("eps", False), ("v", True)):
        d = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, zero_snr=zs, parameterization=name)
        np.testing.assert_allclose(d.betas, g[f"betas_{name}"], rtol=1e-12, atol=1e-15)
        for sname, smp in (("spaced", SpacedSampler(g[f"betas_{name}"], name, False)),
                           ("ddim", DDIMSampler(g[f"betas_{name}"], name, False, 0))):
            for tiled in (False, True):
                torch.manual_seed(7)
                z = smp.sample(_stub, "cpu", 10, (1, 4, 24, 40), cond, unc, 4.0, tiled=tiled, tile_size=16,
                               tile_stride=8, x_T=xT.clone())
                ref = g[f"traj_{sname}_{name}_{'tiled' if tiled else 'full'}"]
                np.testing.assert_array_equal(z.numpy(), ref)


def test_edm_dpm_samplers_bit_exact_vs_reference(golden_dir):
    """EDMSampler / DPMSolverSampler (plain-PyTorch path, analytic stand-in model) against trajectories the
    REFERENCE produced for the same calls (tests/golden/gen_golden_samplers.py): every Karras / DPM-Solver++
    step rule reachable from the CLI, eps and v-parameterization (zero terminal SNR), tiled and cosine-rescaled
    CFG cases; the Brownian-tree rules with the fixture's injected noise source."""
    import importlib.util
    from diffbir_b200.sampler import DPMSolverSampler, EDMSampler
    from diffbir_b200.sampler.edm import run_rule
    spec = importlib.util.spec_from_file_location("gen_golden_samplers_cases", golden_dir / "gen_golden_samplers.py")
    src = (golden_dir / "gen_golden_samplers.py").read_text()
    ns = {}
    exec(src[src.index("EDM_CASES = "):src.index("def rnd(")], ns)      # the case tables only (no reference import)
    g = {**np.load(golden_dir / "samplers.npz"), **np.load(golden_dir / "samplers_v.npz")}
    xT = torch.from_numpy(g["xT"])
    cond = dict(c_txt=torch.from_numpy(g["cond_c_txt"]), c_img=torch.from_numpy(g["cond_c_img"]))
    unc = dict(c_txt=torch.from_numpy(g["uncond_c_txt"]), c_img=cond["c_img"].clone())

    def stub(x, t, c):
        tt = t.float().view(-1, 1, 1, 1) / 1000
        return (0.3 * torch.tanh(x) + 0.05 * c["c_img"] + 0.02 * tt * x
                + 0.01 * c["c_txt"].mean(dim=(1, 2)).view(-1, 1, 1, 1))

    HP, STEPS, SHAPE = ns["HP"], ns["STEPS"], tuple(ns["SHAPE"])
    for pname, zs in (("eps", False), ("v", True)):
        d = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, zero_snr=zs, parameterization=pname)
        for solver, tiled, rc in ns["EDM_CASES"]:
            smp = EDMSampler(d.betas, pname, rc, "edm_" + solver, **HP)
            torch.manual_seed(7)
            z = smp.sample(stub, "cpu", STEPS, SHAPE, cond, unc, 4.0, tiled=tiled, tile_size=16, tile_stride=8, x_T=xT.clone())
            np.testing.assert_array_equal(z.numpy(), g[f"edm_{pname}_{solver}_{int(tiled)}_{int(rc)}"], err_msg=f"edm {pname} {solver}")
        np.testing.assert_array_equal(smp.sigmas.numpy(), g[f"edm_sigmas_{pname}"])
        np.testing.assert_array_equal(smp.timesteps.numpy(), g[f"edm_timesteps_{pname}"])
        for spec_, steps, rc in ns["DPM_CASES"]:
            nb = 1 if rc else SHAPE[0]
            smp = DPMSolverSampler(d.betas, pname, rc, spec_)
            z = smp.sample(stub, "cpu", steps, (nb,) + SHAPE[1:], {k: v[:nb] for k, v in cond.items()},
                           {k: v[:nb] for k, v in unc.items()}, 4.0, x_T=xT[:nb].clone())
            np.testing.assert_array_equal(z.numpy(), g[f"dpm_{pname}_{spec_}_{steps}_{int(rc)}"], err_msg=f"dpm {pname} {spec_}")
        smp = EDMSampler(d.betas, pname, False, "edm_euler", **HP)
        smp.make_schedule(STEPS)
        den = smp.convert_to_denoiser(stub, cond, unc, 4.0)
        x0 = xT * torch.sqrt(1.0 + smp.sigmas[0] ** 2.0)
        for solver in ns["SDE_CASES"]:
            gen = torch.Generator().manual_seed(11)
            z = run_rule(solver, den, x0.clone(), smp.sigmas, HP, noise=lambda s0, s1: torch.randn(SHAPE, generator=gen))
            np.testing.assert_array_equal(z.numpy(), g[f"sde_{pname}_{solver}"], err_msg=f"sde {pname} {solver}")
    with pytest.raises(NotImplementedError):
        DPMSolverSampler(d.betas, "eps", False, "dpm++_s2")


def test_schedule_tables_and_timesteps(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    sp = SpacedSampler(g["betas_eps"], "eps", False)
    sp.make_schedule(50)
    assert (sp.timesteps == g["spaced_ts_eps"]).all()
    assert sp.timesteps[0] == 0 and sp.timesteps[-1] == 999 and len(sp.timesteps) == 50
    dd = DDIMSampler(g["betas_eps"], "eps", False, 0)
    dd.make_schedule(50)
    assert (dd.ddim_timesteps == g["ddim_ts_eps"]).all() and dd.ddim_timesteps[0] == 1
    # cosine CFG ramp (sampler/sampler.py:31-38)
    assert SpacedSampler(g["betas_eps"], "eps", True).get_cfg_scale(4.0, 999) == pytest.approx(1.0, abs=1e-6)
    assert SpacedSampler(g["betas_eps"], "eps", False).get_cfg_scale(4.0, 10) == 4.0


def test_tiling_helpers(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    np.testing.assert_array_equal(uc.gaussian_weights(16, 16), g["gauss_16"])
    assert (np.array(uc.sliding_windows(24, 40, 16, 8)) == g["windows_24_40_16_8"]).all()
    assert (np.array(uc.sliding_windows(30, 30, 16, 12)) == g["windows_30_30_16_12"]).all()
    assert len(uc.sliding_windows(256, 256, 64, 32)) == 49         # config 4: 2048^2, tile 512 / 256
    a, b = torch.from_numpy(g["wavelet_a"]), torch.from_numpy(g["wavelet_b"])
    np.testing.assert_allclose(uc.wavelet_reconstruction(a, b).numpy(), g["wavelet_out"], atol=1e-6)


def test_arch_tables_full_config():
    u = arch.unet_shapes(arch.UNET_CFG)
    c = arch.unet_shapes(arch.CONTROLNET_CFG, True)
    n_u = sum(int(np.prod(s)) for s in u.values())
    n_c = sum(int(np.prod(s)) for s in c.values())
    assert abs(n_u - 865.9e6) < 0.1e6 and abs(n_c - 363.2e6) < 0.7e6   # SURVEY.md §8a a13/a14
    assert len(c) == 324                                                # SURVEY.md §8b (strict load)
    plan = arch.unet_plan(arch.UNET_CFG)
    assert len(plan.input_blocks) == 12 and len(plan.output_blocks) == 12
    assert plan.skip_channels == [320] * 4 + [640] * 3 + [1280] * 6
    cins = [b.layers[0].cin for b in plan.output_blocks]
    assert cins == [2560, 2560, 2560, 2560, 2560, 1920, 1920, 1280, 960, 960, 640, 640]
    v = arch.vae_shapes(arch.VAE_CFG)
    assert abs(sum(int(np.prod(s)) for s in v.values()) - 83.65e6) < 0.2e6
    s = arch.swinir_shapes(arch.SWINIR_CFG)
    assert abs(sum(int(np.prod(x)) for x in s.values()) - 15.8e6) < 0.2e6


def test_synth_checkpoint_is_deterministic_and_nonzero():
    sh = arch.unet_shapes(dict(arch.UNET_CFG, model_channels=64, context_dim=128), True)
    a = make_state_dict(sh, 5, arch.is_zero_init)
    b = make_state_dict(sh, 5, arch.is_zero_init)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert all(v.abs().max() > 0 for k, v in a.items() if v.dim() > 1)
    assert not torch.equal(a["zero_convs.0.0.weight"], make_state_dict(sh, 6, arch.is_zero_init)["zero_convs.0.0.weight"])


def test_geglu_packing_roundtrip():
    from diffbir_b200.engine.common import geglu_tile
    for c in (64, 320, 640, 1280):
        bn = geglu_tile(c)
        inner, hb = 4 * c, bn // 2
        assert inner % hb == 0 and (8 * c) % bn == 0
        w = torch.arange(8 * c, dtype=torch.float32)[:, None].repeat(1, 2)
        wv, wg = w[:inner].view(inner // hb, hb, -1), w[inner:].view(inner // hb, hb, -1)
        wp = torch.cat([wv, wg], dim=1).reshape(2 * inner, -1)
        for j in range(inner // hb):          # tile j: values j*hb.., then the matching gates
            assert wp[j * bn, 0] == j * hb and wp[j * bn + hb, 0] == inner + j * hb


def test_c_abi_exports_every_declared_symbol():
    so = ROOT / "diffbir_b200" / "libdiffbir_b200.so"
    if not so.exists():
        from diffbir_b200.build import build_library
        build_library()
    lib = ctypes.CDLL(str(so))
    header = (ROOT / "include" / "diffbir_b200.h").read_text()
    header = re.sub(r"#ifdef DBIR_DEBUG_PROBES.*?#endif", "", header, flags=re.S)      # probe builds only
    names = sorted(set(re.findall(r"\b(dbir_[a-z0-9_]+)\s*\(", header)) - {"dbir_gemm_args"})
    assert not hasattr(lib, "dbir_debug_mma_rate"), "calibration probes must not ship in the product library"
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
    lib.dbir_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.dbir_version()
    assert lib.dbir_operand_kind() in (0, 1)


def test_product_never_imports_oracle():
    for p in (ROOT / "diffbir_b200").rglob("*.py"):
        txt = p.read_text()
        assert "import oracle" not in txt and "from oracle" not in txt, p


def test_gemm_planner_invariants():
    """dbir_gemm's analytic tile planner (host code, no GPU): every plan is runnable by the kernel
    family — known tile widths, no empty split, split-K only with scratch and enough k-blocks, CTA
    pairs only over an even number of M tiles, forced choices honoured, deterministic."""
    import ctypes as C
    import itertools
    from diffbir_b200 import lib
    L = lib.load()
    out = (C.c_int32 * 4)()

    def plan(m_tiles, N, num_kb, geglu=0, fbn=0, split=0, pair=0, ws=16 * 1024 * 1024):
        assert L.dbir_gemm_model_plan(m_tiles, N, num_kb, geglu, fbn, split, pair, C.c_int64(ws), out) == 0
        return tuple(out)

    for m_tiles, N, num_kb in itertools.product((1, 2, 3, 4, 16, 64, 65, 512), (24, 200, 320, 640, 1280, 2560, 10240),
                                                (1, 5, 7, 20, 45, 180, 360)):
        bn, splits, kbs, pair = plan(m_tiles, N, num_kb)
        assert bn in (32, 64, 128, 160, 256)
        assert bn <= 64 or N % bn == 0                       # ragged N only with the narrow tiles
        assert 1 <= splits <= 16 and kbs * splits >= num_kb and kbs * (splits - 1) < num_kb
        assert splits == 1 or (num_kb // splits >= 6 and m_tiles * -(-N // bn) * splits * 128 * bn <= 16 * 1024 * 1024)
        assert pair in (0, 1) and (not pair or (m_tiles % 2 == 0 and bn >= 64))
        assert plan(m_tiles, N, num_kb) == (bn, splits, kbs, pair)
        assert plan(m_tiles, N, num_kb, ws=0)[1] == 1         # no scratch, no split-K
        assert plan(m_tiles, N, num_kb, split=1)[1] == 1
        assert plan(m_tiles, N, num_kb, pair=2)[3] == 0
        if m_tiles % 2 == 0:
            assert plan(m_tiles, N, num_kb, pair=1, fbn=64)[3] == 1
        assert plan(m_tiles, N, num_kb, fbn=64)[0] == 64
    # GEGLU tiles are at least 64 wide and never split
    assert plan(64, 2560, 5, geglu=1, fbn=128)[:2] == (128, 1)
    # long-K, single-tile-row layers (8x8 latents) are split over k
    assert plan(1, 1280, 180)[1] > 1


def test_integration_doc_struct_matches_binding_and_header():
    """The ctypes mirror of dbir_gemm_args in INTEGRATION.md, the one in diffbir_b200/lib.py and the
    C struct in include/diffbir_b200.h list the same fields in the same order."""
    import re
    from pathlib import Path
    from diffbir_b200 import lib
    root = Path(__file__).resolve().parents[1]
    doc = (root / "INTEGRATION.md").read_text()
    block = doc[doc.index("class GemmArgs"):doc.index("def _ck")]
    doc_fields = re.findall(r'\("(\w+)",\s*C\.', block)
    lib_fields = [f[0] for f in lib.GemmArgs._fields_]
    assert doc_fields == lib_fields
    hdr = (root / "include" / "diffbir_b200.h").read_text()
    body = hdr[hdr.index("typedef struct dbir_gemm_args {"):hdr.index("} dbir_gemm_args;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = []
    for decl in body.split("{", 1)[1].split(";"):
        names = re.findall(r"[\*\s,](\w+)\s*(?=,|$)", decl.strip())
        if decl.strip():
            c_fields += [n for n in names if n not in ("const", "void", "float", "int32_t", "int64_t")]
    assert c_fields == lib_fields


def test_diffbir_alias_exposes_the_reference_names():
    """`import diffbir...` (the reference's module paths: sampler/__init__.py:1-4, inference/__init__.py:1-5,
    model/__init__.py:1-12, pipeline.py) resolves to the engine; names outside the path raise at construction."""
    import diffbir.inference as di
    import diffbir.model as dm
    import diffbir.pipeline as dp
    import diffbir.sampler as dsm
    import diffbir_b200
    from diffbir.utils.common import instantiate_from_config, make_tiled_fn, wavelet_reconstruction  # noqa: F401
    assert dp.SwinIRPipeline is diffbir_b200.pipeline.SwinIRPipeline and dp.Pipeline is diffbir_b200.pipeline.Pipeline
    assert dm.ControlLDM is diffbir_b200.model.ControlLDM and dsm.SpacedSampler is diffbir_b200.sampler.SpacedSampler
    for mod, names in ((dsm, ["SpacedSampler", "DDIMSampler", "DPMSolverSampler", "EDMSampler"]),
                       (di, ["BSRInferenceLoop", "BFRInferenceLoop", "BIDInferenceLoop", "UnAlignedBFRInferenceLoop",
                             "CustomInferenceLoop"]),
                       (dm, ["ControlledUnetModel", "ControlNet", "AutoencoderKL", "FrozenOpenCLIPEmbedder", "ControlLDM",
                             "Diffusion", "SwinIR", "RRDBNet", "SCUNet", "config"]),
                       (dp, ["Pipeline", "SwinIRPipeline", "BSRNetPipeline", "SCUNetPipeline"])):
        for n in names:
            assert hasattr(mod, n), f"{mod.__name__}.{n} missing"
    assert dsm.EDMSampler is diffbir_b200.sampler.EDMSampler and dsm.DPMSolverSampler is diffbir_b200.sampler.DPMSolverSampler
    assert dm.RRDBNet is diffbir_b200.model.RRDBNet and dp.BSRNetPipeline is diffbir_b200.pipeline.BSRNetPipeline
    assert dm.SCUNet is diffbir_b200.model.SCUNet and dp.SCUNetPipeline is diffbir_b200.pipeline.SCUNetPipeline
    assert di.BIDInferenceLoop is diffbir_b200.inference.BIDInferenceLoop
    assert di.CustomInferenceLoop is diffbir_b200.inference.CustomInferenceLoop
    for cls in (di.UnAlignedBFRInferenceLoop, dm.ControlNet):
        with pytest.raises(NotImplementedError):
            cls()
    # run_gradio.py-style helpers: registry + local "download", VRAM monitor, nested .to()
    from diffbir.inference.pretrained_models import MODELS
    from diffbir.utils.common import VRAMPeakMonitor, load_model_from_url, to
    assert set(MODELS) >= {"sd_v2.1", "v2.1", "swinir_general", "bsrnet", "scunet_psnr"}
    with pytest.raises(FileNotFoundError, match="v2.pth"):
        load_model_from_url("https://example.invalid/some/path/" + MODELS["v2"])
    with VRAMPeakMonitor("phase"):
        moved = to(dict(a=torch.ones(2), b=[torch.zeros(1), "s"], c=(torch.ones(1),)), "cpu")
    assert moved["b"][1] == "s" and isinstance(moved["c"], tuple) and torch.equal(moved["a"], torch.ones(2))
    # the YAML reflection targets of the reference configs resolve through the alias too
    from diffbir.model.cldm import ControlLDM
    from diffbir.model.gaussian_diffusion import Diffusion
    from diffbir.model.swinir import SwinIR
    assert ControlLDM is dm.ControlLDM and Diffusion is dm.Diffusion and SwinIR is dm.SwinIR
