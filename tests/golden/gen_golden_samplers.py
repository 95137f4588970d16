"""Fixtures for the EDM-family and DPM-Solver samplers, produced by the REFERENCE
(diffbir.sampler.{EDMSampler, DPMSolverSampler} and the k_diffusion step functions) with an analytic
stand-in model on the CPU.

    python tests/golden/gen_golden_samplers.py        # needs the reference checkout (_ref_import.py); writes samplers.npz, samplers_v.npz

tests/test_oracle_golden.py::test_edm_dpm_samplers_match_reference replays the same calls through
diffbir_b200.sampler and asserts bit equality. The stochastic "SDE" rules need torchsde's Brownian tree
inside the reference's EDMSampler (not installed here, the reference itself cannot run them), so their
step functions are driven directly with an injected seeded noise source — the same source is injected
into the product's step rules by the test.
"""
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent))
from _ref_import import use_reference  # noqa: E402

use_reference()
OUT = Path(__file__).resolve().parent

EDM_CASES = [  # (solver, tiled, rescale_cfg)
    ("euler", False, False), ("euler", True, True), ("euler_a", False, False), ("heun", False, True),
    ("dpm_2", True, False), ("dpm_2_a", False, False), ("lms", False, False), ("dpm++_2s_a", False, True),
    ("dpm++_2m", False, False), ("dpm++_2m", True, False),
]
DPM_CASES = [("dpm++_m2", 10, False), ("dpm++_m2", 6, True), ("dpm++_m3", 12, False), ("dpm_m2", 8, False), ("dpm++_m1", 5, False)]
SDE_CASES = ["dpm++_sde", "dpm++_2m_sde", "dpm++_3m_sde"]
HP = dict(s_churn=0.5, s_tmin=0.0, s_tmax=300.0, s_noise=1.003, eta=1.0, order=4)
STEPS, SHAPE = 8, (2, 4, 24, 40)


def rnd(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


class Stub(torch.nn.Module):
    def forward(self, x, t, cond):
        tt = t.float().view(-1, 1, 1, 1) / 1000
        return (0.3 * torch.tanh(x) + 0.05 * cond["c_img"] + 0.02 * tt * x
                + 0.01 * cond["c_txt"].mean(dim=(1, 2)).view(-1, 1, 1, 1))


def seeded_noise(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda s0, s1: torch.randn(SHAPE, generator=g)


@torch.no_grad()
def main():
    from diffbir.model.gaussian_diffusion import Diffusion
    from diffbir.sampler import DPMSolverSampler, EDMSampler
    from diffbir.sampler import k_diffusion as K

    stub = Stub()
    xT = rnd(60, *SHAPE)
    cond = dict(c_txt=rnd(61, 2, 77, 8), c_img=rnd(62, *SHAPE))
    uncond = dict(c_txt=rnd(63, 2, 77, 8), c_img=cond["c_img"].clone())
    out = dict(xT=xT.numpy(), cond_c_txt=cond["c_txt"].numpy(), cond_c_img=cond["c_img"].numpy(),
               uncond_c_txt=uncond["c_txt"].numpy())
    for pname, zero_snr in (("eps", False), ("v", True)):
        diff = Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000, zero_snr=zero_snr, parameterization=pname)
        for solver, tiled, rc in EDM_CASES:
            s = EDMSampler(diff.betas, pname, rc, "edm_" + solver, **HP)
            torch.manual_seed(7)
            z = s.sample(stub, "cpu", STEPS, SHAPE, cond, uncond, 4.0, tiled=tiled, tile_size=16, tile_stride=8,
                         x_T=xT.clone(), progress=False)
            out[f"edm_{pname}_{solver}_{int(tiled)}_{int(rc)}"] = z.numpy()
        out[f"edm_sigmas_{pname}"] = s.sigmas.numpy()
        out[f"edm_timesteps_{pname}"] = s.timesteps.numpy()
        for spec, steps, rc in DPM_CASES:
            s = DPMSolverSampler(diff.betas, pname, rc, spec)
            nb = 1 if rc else SHAPE[0]        # the library's cfg_rescale branch only accepts one sample (math.cos of t)
            c1 = {k: v[:nb] for k, v in cond.items()}
            u1 = {k: v[:nb] for k, v in uncond.items()}
            z = s.sample(stub, "cpu", steps, (nb,) + SHAPE[1:], c1, u1, 4.0, x_T=xT[:nb].clone(), progress=False)
            out[f"dpm_{pname}_{spec}_{steps}_{int(rc)}"] = z.numpy()
        # SDE step functions with an injected noise source, through the reference's own denoiser
        s = EDMSampler(diff.betas, pname, False, "edm_euler", **HP)
        s.make_schedule(STEPS)
        den = s.convert_to_denoiser(stub, cond, uncond, 4.0)
        x0 = xT * torch.sqrt(1.0 + s.sigmas[0] ** 2.0)
        fns = {"dpm++_sde": K.sample_dpmpp_sde, "dpm++_2m_sde": K.sample_dpmpp_2m_sde, "dpm++_3m_sde": K.sample_dpmpp_3m_sde}
        for solver in SDE_CASES:
            z = fns[solver](den, x0.clone(), s.sigmas, disable=True, eta=HP["eta"], s_noise=HP["s_noise"],
                            noise_sampler=seeded_noise(11))
            out[f"sde_{pname}_{solver}"] = z.numpy()
    # two files, each under 1 MB: the inputs and eps-parameterization trajectories, and the v-parameterization ones
    v_keys = [k for k in out if k.startswith(("edm_v_", "edm_sigmas_v", "edm_timesteps_v", "dpm_v_", "sde_v_"))]
    np.savez_compressed(OUT / "samplers.npz", **{k: v for k, v in out.items() if k not in v_keys})
    np.savez_compressed(OUT / "samplers_v.npz", **{k: out[k] for k in v_keys})
    print("wrote", OUT / "samplers.npz", OUT / "samplers_v.npz", len(out), "arrays")


if __name__ == "__main__":
    main()
