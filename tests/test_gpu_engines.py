"""-m gpu: network-level parity of the kernel engines against (a) the golden fixtures produced
by the reference itself (reduced configs) and (b) the oracle run in fp32 (TF32 off) on the same
device at the full SD-2.1 / SwinIR configuration.

Tolerance: the engines round tensor-core operands to 16 bit (fp16 by default) and accumulate in
fp32, so a forward differs from the fp32 reference by operand rounding only: relative RMS error
below 4e-3 per network forward (measured ~1e-3), i.e. > 48 dB per forward; the end-to-end
PSNR >= 50 dB target is checked on the uint8 pipeline output in test_gpu_pipeline.py."""
import numpy as np
import pytest
import torch

from diffbir_b200 import arch
from diffbir_b200.utils.synth import make_state_dict
from tests.gpu_util import no_tf32, psnr, rel_rms, to_dev
from tests.small_cfg import CN_SMALL, SWIN_SMALL, UNET_SMALL, VAE_SMALL

pytestmark = pytest.mark.gpu
TOL = 4e-3


def _cldm_engine(ucfg, ccfg, seeds=(1, 2)):
    from diffbir_b200.engine.cldm import CldmEngine
    usd = make_state_dict(arch.unet_shapes(ucfg), seeds[0], arch.is_zero_init)
    csd = make_state_dict(arch.unet_shapes(ccfg, True), seeds[1], arch.is_zero_init)
    return CldmEngine(usd, csd, ucfg, ccfg, "cuda"), usd, csd


def test_cldm_small_vs_reference_golden(golden_dir):
    no_tf32()
    g = np.load(golden_dir / "cldm_small.npz")
    eng, _, _ = _cldm_engine(UNET_SMALL, CN_SMALL)
    x, hint, ctx = (torch.from_numpy(g[k]).cuda() for k in ("x", "hint", "ctx"))
    eng.set_context(ctx)
    eng.set_timesteps([int(g["t"][0])], nb=2)
    eng.load_step(0)
    eps = eng.forward(x, hint, list(g["scales"]))
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["eps"]).cuda()
    e = rel_rms(eps, ref)
    print(f"cldm small vs reference: rel rms {e:.2e}, psnr {psnr(eps, ref):.1f} dB")
    assert e < TOL
    # determinism: same inputs -> same bits
    eps2 = eng.forward(x, hint, list(g["scales"]))
    assert torch.equal(eps, eps2)


@pytest.mark.parametrize("L,nb", [(32, 2), (24, 1), (8, 3)])
def test_cldm_small_vs_oracle_shapes(L, nb):
    from oracle import cldm as ocl
    no_tf32()
    eng, usd, csd = _cldm_engine(UNET_SMALL, CN_SMALL)
    gen = torch.Generator().manual_seed(L)
    x = torch.randn(nb, 4, L, L, generator=gen).cuda()
    hint = torch.randn(nb, 4, L, L, generator=gen).cuda()
    ctx = torch.randn(nb, 77, UNET_SMALL["context_dim"], generator=gen).cuda()
    scales = [1.0] * 13
    import faulthandler
    import os
    import time
    if os.environ.get("DBIR_TEST_FAULTDUMP"):        # where does a slow run spend its time? (stack every N s)
        faulthandler.dump_traceback_later(int(os.environ["DBIR_TEST_FAULTDUMP"]), repeat=True)
    t0 = time.perf_counter()
    eng.set_context(ctx)
    eng.set_timesteps([500], nb=nb)
    eng.load_step(0)
    eps = eng.forward(x, hint, scales)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    with torch.no_grad():
        ref = ocl.cldm_forward(to_dev(usd), to_dev(csd), x, torch.full((nb,), 500, device="cuda"), ctx, hint, scales)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    e = rel_rms(eps, ref)
    faulthandler.cancel_dump_traceback_later()
    print(f"cldm small L={L} nb={nb}: rel rms {e:.2e} (engine {t1 - t0:.1f}s incl. plan tuning, oracle {t2 - t1:.1f}s)")
    assert e < TOL


def test_cldm_full_config_vs_oracle(golden_dir):
    """SD-2.1 UNet + ControlNet (1.23 B parameters, random init), latent 64x64, batch 2 (the
    cond/uncond pair of one 512x512 image) against the fp32 oracle, and against the output of the REFERENCE's own
    modules on the same weights and inputs (tests/golden/full_config.npz, gen_golden_full.py)."""
    from oracle import cldm as ocl
    no_tf32()
    g = np.load(golden_dir / "full_config.npz")
    eng, usd, csd = _cldm_engine(arch.UNET_CFG, arch.CONTROLNET_CFG, seeds=(1234, 1235))
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 64, 64, generator=gen).repeat(2, 1, 1, 1).cuda()
    hint = (torch.randn(1, 4, 64, 64, generator=gen) * 0.5).repeat(2, 1, 1, 1).cuda()
    ctx = torch.randn(2, 77, 1024, generator=gen).cuda()
    scales = [1.0] * 13
    eng.set_context(ctx)
    eng.set_timesteps([999, 500, 0], nb=2)
    usd_d, csd_d = to_dev(usd), to_dev(csd)
    for i, t in enumerate([999, 500, 0]):
        eng.load_step(i)
        eps = eng.forward(x, hint, scales)
        with torch.no_grad():
            ref = ocl.cldm_forward(usd_d, csd_d, x, torch.full((2,), t, device="cuda"), ctx, hint, scales)
        e = rel_rms(eps, ref)
        eg = rel_rms(eps, torch.from_numpy(g[f"cldm_eps_t{t}"]).cuda())
        print(f"cldm full t={t}: rel rms {e:.2e}, psnr {psnr(eps, ref):.1f} dB, |eps| {ref.abs().mean():.3f}; vs reference fixture {eg:.2e}")
        assert e < TOL and eg < TOL


def test_vae_small_vs_reference_golden(golden_dir):
    from diffbir_b200.engine.vae import VaeEngine
    no_tf32()
    g = np.load(golden_dir / "vae_small.npz")
    eng = VaeEngine(make_state_dict(arch.vae_shapes(VAE_SMALL), 3), VAE_SMALL, "cuda")
    dec = eng.decode(torch.from_numpy(g["z"]).cuda())
    mom = eng.encode_moments(torch.from_numpy(g["img"]).cuda())
    e1, e2 = rel_rms(dec, torch.from_numpy(g["dec"]).cuda()), rel_rms(mom, torch.from_numpy(g["moments"]).cuda())
    print(f"vae small vs reference: decode {e1:.2e} encode {e2:.2e}")
    assert e1 < TOL and e2 < TOL


def test_vae_full_config_vs_oracle(golden_dir):
    from diffbir_b200.engine.vae import VaeEngine
    from oracle import cldm as ocl
    no_tf32()
    g = np.load(golden_dir / "full_config_vae.npz")
    sd = make_state_dict(arch.vae_shapes(arch.VAE_CFG), 77)
    eng = VaeEngine(sd, None, "cuda")
    sd_d = to_dev(sd)
    gen = torch.Generator().manual_seed(3)
    z = torch.randn(1, 4, 64, 64, generator=gen).cuda()
    img = (torch.rand(1, 3, 512, 512, generator=gen) * 2 - 1).cuda()
    dec = eng.decode(z)
    mom = eng.encode_moments(img)
    with torch.no_grad():
        rdec, rmom = ocl.vae_decode(sd_d, z), ocl.vae_encode_moments(sd_d, img)
    e1, e2 = rel_rms(dec, rdec), rel_rms(mom, rmom)
    st = int(g["vae_dec_stride"])
    g1 = rel_rms(dec[..., ::st, ::st], torch.from_numpy(g["vae_dec"]).cuda())
    g2 = rel_rms(mom, torch.from_numpy(g["vae_moments"]).cuda())
    print(f"vae full: decode {e1:.2e} ({psnr(dec, rdec):.1f} dB) encode {e2:.2e}; vs reference fixture {g1:.2e} / {g2:.2e}")
    assert e1 < TOL and e2 < TOL and g1 < TOL and g2 < TOL


def test_swinir_small_vs_reference_golden(golden_dir):
    from diffbir_b200.engine.swinir import SwinIREngine
    no_tf32()
    g = np.load(golden_dir / "swinir_small.npz")
    eng = SwinIREngine(make_state_dict(arch.swinir_shapes(SWIN_SMALL), 4), SWIN_SMALL, "cuda")
    x = torch.from_numpy(g["x"])
    xp = torch.nn.functional.pad(x, (0, 0, 0, 0))            # 128 x 192 is already a multiple of 64
    y = eng.forward(xp.cuda().contiguous())
    ref = torch.from_numpy(g["y"]).cuda()
    err = ((y - ref).abs().max() / ref.std()).item()
    print(f"swinir small vs reference: max err / std = {err:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB")
    assert err < 2e-2


@pytest.mark.parametrize("size", [256, 512])
def test_swinir_full_config_vs_oracle(size, golden_dir):
    from diffbir_b200.engine.swinir import SwinIREngine
    from oracle import swinir as osw
    no_tf32()
    sd = make_state_dict(arch.swinir_shapes(arch.SWINIR_CFG), 1234)
    eng = SwinIREngine(sd, None, "cuda")
    x = torch.rand(1, 3, size, size, generator=torch.Generator().manual_seed(0)).cuda()
    y = eng.forward(x)
    with torch.no_grad():
        ref = osw.swinir_forward(to_dev(sd), x)
    err = ((y - ref).abs().max() / ref.std()).item()
    print(f"swinir {size}: max err / std = {err:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB")
    assert err < 3e-2
    if size == 256:                                            # the reference's own output for this weight / input pair
        gref = torch.from_numpy(np.load(golden_dir / "full_config_swinir.npz")["swinir_y256"]).cuda()
        eg = ((y - gref).abs().max() / gref.std()).item()
        print(f"swinir 256 vs reference fixture: max err / std = {eg:.2e}")
        assert eg < 3e-2


def test_rrdbnet_small_vs_reference_golden(golden_dir):
    from diffbir_b200.engine.bsrnet import RRDBNetEngine
    from tests.small_cfg import RRDB_SMALL
    no_tf32()
    g = np.load(golden_dir / "bsrnet_small.npz")
    eng = RRDBNetEngine(make_state_dict(arch.rrdbnet_shapes(RRDB_SMALL), 7), RRDB_SMALL, "cuda")
    y = eng.forward(torch.from_numpy(g["x"]).cuda())
    ref = torch.from_numpy(g["y"]).cuda()
    e = rel_rms(y, ref)
    print(f"rrdbnet small vs reference: rel rms {e:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB")
    assert y.shape == ref.shape and e < TOL
    assert torch.equal(y, eng.forward(torch.from_numpy(g["x"]).cuda()))        # graph replay: same bits


def test_rrdbnet_full_config_vs_oracle(golden_dir):
    """BSRNet (23 RRDB, configs/inference/bsrnet.yaml) on a 128x160 LQ image -> 512x640, against the fp32 oracle and the
    reference's own output (full_config.npz)."""
    from diffbir_b200.engine.bsrnet import RRDBNetEngine
    from oracle import bsrnet as ob
    no_tf32()
    sd = make_state_dict(arch.rrdbnet_shapes(arch.RRDBNET_CFG), 78)
    eng = RRDBNetEngine(sd, None, "cuda")
    x = torch.rand(1, 3, 128, 160, generator=torch.Generator().manual_seed(4)).cuda()
    y = eng.forward(x)
    with torch.no_grad():
        ref = ob.rrdbnet_forward(to_dev(sd), x)
    e = rel_rms(y, ref)
    g = np.load(golden_dir / "full_config.npz")
    st = int(g["rrdb_stride"])
    eg = rel_rms(y[..., ::st, ::st], torch.from_numpy(g["rrdb_y"]).cuda())
    print(f"rrdbnet full: rel rms {e:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB, |y| {ref.abs().mean():.4f}; vs reference fixture {eg:.2e}")
    assert y.shape == (1, 3, 512, 640) and e < TOL and eg < TOL


def test_scunet_small_vs_reference_golden(golden_dir):
    from diffbir_b200.model import SCUNet
    from tests.small_cfg import SCUNET_SMALL
    no_tf32()
    g = np.load(golden_dir / "scunet_small.npz")
    net = SCUNet(**SCUNET_SMALL, device="cuda")
    net.load_state_dict(make_state_dict(arch.scunet_shapes(SCUNET_SMALL), 9))
    y = net(torch.from_numpy(g["x"]).cuda())                 # 120 x 72: replicate-padded to 128 x 128 inside
    ref = torch.from_numpy(g["y"]).cuda()
    e = rel_rms(y, ref)
    print(f"scunet small vs reference: rel rms {e:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB")
    assert y.shape == ref.shape and e < TOL
    assert torch.equal(y, net(torch.from_numpy(g["x"]).cuda()))


def test_scunet_full_config_vs_oracle(golden_dir):
    """SCUNet [4,4,4,4,4,4,4] x dim 64 (configs/inference/scunet.yaml) on a 256 x 320 image against the fp32 oracle and the
    reference's own output (full_config.npz)."""
    from diffbir_b200.engine.scunet import SCUNetEngine
    from oracle import scunet as osc
    no_tf32()
    sd = make_state_dict(arch.scunet_shapes(arch.SCUNET_CFG), 79)
    eng = SCUNetEngine(sd, None, "cuda")
    x = torch.rand(1, 3, 256, 320, generator=torch.Generator().manual_seed(6)).cuda()
    y = eng.forward(x)
    with torch.no_grad():
        ref = osc.scunet_forward(to_dev(sd), x)
    e = rel_rms(y, ref)
    g = np.load(golden_dir / "full_config.npz")
    st = int(g["scunet_stride"])
    eg = rel_rms(y[..., ::st, ::st], torch.from_numpy(g["scunet_y"]).cuda())
    print(f"scunet full: rel rms {e:.2e}, psnr(peak 1) {psnr(y, ref, 1.0):.1f} dB, |y| {ref.abs().mean():.4f}; vs reference fixture {eg:.2e}")
    assert y.shape == x.shape and e < TOL and eg < TOL
