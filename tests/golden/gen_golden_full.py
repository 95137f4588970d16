"""FULL-configuration fixtures from the reference: the real SD-2.1 UNet + ControlNet (1.23 B parameters), the full VAE,
the 8 x 6-block SwinIR, the 23-block RRDBNet and the 28-block SCUNet of configs/inference/*.yaml, random-init weights from
the seeded generator, on EXACTLY the weights and inputs of the full-config `-m gpu` tests (tests/test_gpu_engines.py):

    python tests/golden/gen_golden_full.py        # needs the reference checkout (_ref_import.py), ~10 min of CPU; writes full_config{,_vae,_swinir}.npz

so the chain reference == oracle (tests/test_oracle_golden.py, CPU) and oracle ~ CUDA (GPU) is closed at full width, not
only at the reduced widths of the other fixtures, and the GPU tests can also be read against the reference directly.
Large outputs are stored on a stride (`*_stride` keys).
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle" / "_shims"))
sys.path.insert(0, str(Path(__file__).resolve().parent))
from _ref_import import use_reference  # noqa: E402

use_reference()
from diffbir_b200 import arch  # noqa: E402
from diffbir_b200.utils.synth import make_state_dict  # noqa: E402

OUT = Path(__file__).resolve().parent


def plain(d):
    return {k: (list(v) if isinstance(v, tuple) else v) for k, v in d.items()}


@torch.no_grad()
def main():
    from diffbir.model.bsrnet import RRDBNet
    from diffbir.model.controlnet import ControlledUnetModel, ControlNet
    from diffbir.model.scunet import SCUNet
    from diffbir.model.swinir import SwinIR
    from diffbir.model.vae import AutoencoderKL
    out = {}
    ref_kw = dict(use_checkpoint=False, image_size=32, use_spatial_transformer=True, use_linear_in_transformer=True, legacy=False)

    # ---- ControlLDM.forward (cldm.py:160-172) = test_cldm_full_config_vs_oracle: seeds 1234 / 1235, generator 0
    unet = ControlledUnetModel(**plain(arch.UNET_CFG), **ref_kw).eval()
    cnet = ControlNet(**plain({k: v for k, v in arch.CONTROLNET_CFG.items() if k != "out_channels"}), **ref_kw).eval()
    unet.load_state_dict(make_state_dict(arch.unet_shapes(arch.UNET_CFG), 1234, arch.is_zero_init), strict=True)
    cnet.load_state_dict(make_state_dict(arch.unet_shapes(arch.CONTROLNET_CFG, True), 1235, arch.is_zero_init), strict=True)
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 64, 64, generator=gen).repeat(2, 1, 1, 1)
    hint = (torch.randn(1, 4, 64, 64, generator=gen) * 0.5).repeat(2, 1, 1, 1)
    ctx = torch.randn(2, 77, 1024, generator=gen)
    for t in (999, 500, 0):
        tt = torch.full((2,), t)
        control = cnet(x=x, hint=hint, timesteps=tt, context=ctx)
        eps = unet(x=x, timesteps=tt, context=ctx, control=[c.clone() for c in control], only_mid_control=False)
        out[f"cldm_eps_t{t}"] = eps.numpy()
        print("cldm full t", t, eps.abs().mean().item(), eps.std().item(), flush=True)
    del unet, cnet

    # ---- VAE (vae.py:562-582) = test_vae_full_config_vs_oracle: seed 77, generator 3; plus a 16 x 16 latent case for the CPU suite
    vc = arch.VAE_CFG
    vae = AutoencoderKL(ddconfig=dict(double_z=True, z_channels=vc["z_channels"], resolution=256, in_channels=vc["in_channels"],
                                      out_ch=vc["out_ch"], ch=vc["ch"], ch_mult=list(vc["ch_mult"]),
                                      num_res_blocks=vc["num_res_blocks"], attn_resolutions=[], dropout=0.0), embed_dim=vc["embed_dim"]).eval()
    vae.load_state_dict(make_state_dict(arch.vae_shapes(vc), 77), strict=True)
    gen = torch.Generator().manual_seed(3)
    z = torch.randn(1, 4, 64, 64, generator=gen)
    img = torch.rand(1, 3, 512, 512, generator=gen) * 2 - 1
    out["vae_dec_stride"] = np.int64(4)
    out["vae_dec"] = vae.decode(z)[..., ::4, ::4].numpy()
    out["vae_moments"] = vae.encode(img).parameters.numpy()
    gen = torch.Generator().manual_seed(31)
    z16 = torch.randn(1, 4, 16, 16, generator=gen)
    img128 = torch.rand(1, 3, 128, 128, generator=gen) * 2 - 1
    out["vae_dec16"] = vae.decode(z16).numpy()
    out["vae_moments128"] = vae.encode(img128).parameters.numpy()
    print("vae full", float(np.abs(out["vae_dec"]).mean()), float(np.abs(out["vae_moments"]).mean()), flush=True)
    del vae

    # ---- SwinIR (swinir.py:856-894) = test_swinir_full_config_vs_oracle[256]: seed 1234, generator 0
    sc = arch.SWINIR_CFG
    swin = SwinIR(img_size=sc["img_size"], patch_size=1, in_chans=3, embed_dim=sc["embed_dim"], depths=list(sc["depths"]),
                  num_heads=list(sc["num_heads"]), window_size=8, mlp_ratio=sc["mlp_ratio"], sf=8, img_range=1.0,
                  upsampler="nearest+conv", resi_connection="1conv", unshuffle=True, unshuffle_scale=8).eval()
    missing, unexpected = swin.load_state_dict(make_state_dict(arch.swinir_shapes(sc), 1234), strict=False)
    assert not unexpected and all(k.endswith(("relative_position_index", "attn_mask")) for k in missing)
    xs = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(0))
    out["swinir_y256"] = swin(xs).numpy()
    print("swinir full", float(out["swinir_y256"].mean()), float(out["swinir_y256"].std()), flush=True)
    del swin

    # ---- RRDBNet (bsrnet.py:89-104) = test_rrdbnet_full_config_vs_oracle: seed 78, generator 4
    rr = RRDBNet(**arch.RRDBNET_CFG).eval()
    rr.load_state_dict(make_state_dict(arch.rrdbnet_shapes(arch.RRDBNET_CFG), 78), strict=True)
    xr = torch.rand(1, 3, 128, 160, generator=torch.Generator().manual_seed(4))
    out["rrdb_stride"] = np.int64(4)
    out["rrdb_y"] = rr(xr)[..., ::4, ::4].numpy()
    print("rrdbnet full", float(np.abs(out["rrdb_y"]).mean()), flush=True)
    del rr

    # ---- SCUNet (scunet.py:221-243) = test_scunet_full_config_vs_oracle: seed 79, generator 6
    cfg = arch.SCUNET_CFG
    scu = SCUNet(in_nc=cfg["in_nc"], config=list(cfg["config"]), dim=cfg["dim"]).eval()
    scu.load_state_dict(make_state_dict(arch.scunet_shapes(cfg), 79), strict=True)
    xc = torch.rand(1, 3, 256, 320, generator=torch.Generator().manual_seed(6))
    out["scunet_stride"] = np.int64(2)
    out["scunet_y"] = scu(xc)[..., ::2, ::2].numpy()
    print("scunet full", float(np.abs(out["scunet_y"]).mean()), flush=True)

    # three files, each under 1 MB: the VAE and SwinIR outputs apart from the ControlLDM / RRDBNet / SCUNet ones
    parts = {"full_config_vae": ("vae",), "full_config_swinir": ("swinir",), "full_config": ("cldm", "rrdb", "scunet")}
    for name, prefixes in parts.items():
        np.savez_compressed(OUT / f"{name}.npz", **{k: v for k, v in out.items() if k.startswith(prefixes)})
        print(f"wrote {name}.npz")


if __name__ == "__main__":
    main()
