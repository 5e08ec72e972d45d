"""CPU: PLMSSampler's schedule check and interface, and the host-side argument checks of sdb_plms_step (every check runs
before any launch, so none of them needs a GPU)."""
import inspect

import numpy as np
import pytest
import torch

from oracle import restate as R


def _shim():
    return R.ModelShim(lambda x, t, c: x, R.sd_alphas_cumprod())


def test_make_schedule_rejects_eta():
    from sdb200.plms import PLMSSampler
    s = PLMSSampler(_shim())
    with pytest.raises(ValueError, match="ddim_eta must be 0 for PLMS"):
        s.make_schedule(50, ddim_eta=0.5, verbose=False)
    with pytest.raises(ValueError):
        s.sample(10, 1, (4, 8, 8), eta=1.0, verbose=False)


def test_schedule_is_ddims():
    from sdb200.ddim import DDIMSampler
    from sdb200.plms import PLMSSampler
    p, d = PLMSSampler(_shim()), DDIMSampler(_shim())
    p.make_schedule(20, verbose=False)
    d.make_schedule(20, verbose=False)
    assert np.array_equal(p.ddim_timesteps, d.ddim_timesteps)
    for i in range(20):
        assert p.derived_coefficients(i) == d.derived_coefficients(i)
        assert p.derived_coefficients(i)[3] == 0.0                      # sigma_t
    assert [int(v) for v in p._time_range(None, False)[0]][:3] == [951, 901, 851]


def test_reference_signatures_and_hidden_img2img():
    from sdb200.ddim import DDIMSampler
    from sdb200.plms import PLMSSampler
    names = lambda f: list(inspect.signature(f).parameters)
    assert names(PLMSSampler.sample) == names(DDIMSampler.sample)
    assert names(PLMSSampler.plms_sampling) == names(DDIMSampler.ddim_sampling)
    assert names(PLMSSampler.p_sample_plms) == ["self", "x", "c", "t", "index", "repeat_noise", "use_original_steps",
                                                "quantize_denoised", "temperature", "noise_dropout", "score_corrector",
                                                "corrector_kwargs", "unconditional_guidance_scale",
                                                "unconditional_conditioning", "old_eps", "t_next"]
    s = PLMSSampler(_shim())
    for name in ("stochastic_encode", "decode", "ddim_sampling", "p_sample_ddim"):
        assert not hasattr(s, name), name
        with pytest.raises(AttributeError, match="PLMSSampler has no"):
            getattr(s, name)
    assert hasattr(DDIMSampler(_shim()), "decode")                     # DDIM keeps its own


def test_txt2img_signature():
    from sdb200.pipeline import LatentDiffusion
    p = inspect.signature(LatentDiffusion.txt2img).parameters
    assert "plms" in p and p["plms"].default is False


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    return _lib.load()


def test_plms_step_no_cpu_fallback(lib):
    from sdb200 import _lib, ops
    z = torch.zeros(4)
    with pytest.raises(_lib.SdbError):
        ops.plms_step(z, z, 1, 0.5, 0.6, 0.3, 0.0, 0.7)


# fake device addresses, 4 KB apart: never dereferenced, the checks reject the call first
X, E, U, O1, O2, O3, NZ, EO, EP, P0, XP = (0x100000 + 0x1000 * k for k in range(11))
N = 16


def _call(lib, x=X, e=E, u=None, o1=O1, o2=O2, o3=O3, order=4, noise=None, sigma=0.0, e_out=EO, ep=EP, p0=P0, xp=XP, n=N):
    return lib.sdb_plms_step(x, e, u, 7.5, o1, o2, o3, order, noise, 0.9, 0.95, 0.3, sigma, 0.4, 1.0, e_out, ep, p0, xp, n, None)


@pytest.mark.parametrize("case", [
    dict(x=None), dict(e=None), dict(n=0),                                           # null inputs, empty problem
    dict(order=-1), dict(order=5),                                                   # order outside 0..4
    dict(e_out=None, ep=None, p0=None, xp=None),                                     # no output
    dict(order=0, o1=None), dict(order=2, o1=None), dict(order=3, o1=None),          # history the order reads
    dict(order=3, o2=None), dict(order=4, o2=None), dict(order=4, o3=None),
    dict(sigma=0.5),                                                                 # sigma != 0 without noise
    dict(xp=X), dict(p0=E), dict(e_out=U, u=U), dict(ep=O1), dict(xp=O3), dict(e_out=NZ, noise=NZ),   # output == input
    dict(xp=X + 4 * (N - 1)), dict(e_out=E - 4 * (N - 1)),                            # output overlaps an input
    dict(p0=XP), dict(ep=EO + 8),                                                    # two outputs overlap
])
def test_plms_step_host_checks(lib, case):
    assert _call(lib, **case) == -1, case
    assert lib.sdb_last_error_string().startswith(b"plms_step: "), case      # rejected by a check, not by a failed launch

