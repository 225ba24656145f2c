"""DPM-Solver++(2M) host logic (schedules.dpmpp_2m_table / dpmpp_timesteps, argument checks,
sample_sharded(method=...)): runs without a GPU."""
import contextlib
import io
import math

import numpy as np
import pytest
import torch

from mri_image_generation_b200 import schedules


def _ac(kind, T):
    betas = (schedules.cosine_beta_schedule(T) if kind == "cosine"
             else schedules.linear_beta_schedule(T, 1e-4, 0.02))
    return schedules.make_buffers(betas, True)["alphas_cumprod"]


def _restated(ac, ts):
    """The table written out independently: fp64 numpy from the fp32 buffer, lambda = log(alpha/sigma)."""
    a = ac.double().numpy()
    alpha = np.array([math.sqrt(a[t]) if t >= 0 else 1.0 for t in ts])
    sigma = np.array([math.sqrt(1.0 - a[t]) if t >= 0 else 0.0 for t in ts])
    rows = []
    for i in range(len(ts) - 1):
        if ts[i + 1] < 0:
            rows.append([sigma[i], 1 / alpha[i], 0.0, 1.0, 0.0])
            continue
        lam = lambda j: math.log(alpha[j] / sigma[j])
        h = lam(i + 1) - lam(i)
        phi = math.expm1(-h)
        c = 0.0 if i == 0 else -0.5 * alpha[i + 1] * phi * h / (lam(i) - lam(i - 1))
        rows.append([sigma[i], 1 / alpha[i], sigma[i + 1] / sigma[i], -alpha[i + 1] * phi, c])
    return np.array(rows)


@pytest.mark.parametrize("kind,T", [("cosine", 1000), ("cosine", 400), ("linear", 1000)])
@pytest.mark.parametrize("M", [1, 2, 7, 20, 50])
def test_table_equals_fp64_restatement(kind, T, M):
    ac = _ac(kind, T)
    ts_list = schedules.dpmpp_timesteps(T - 1, M)
    ts, coef = schedules.dpmpp_2m_table(ac, ts_list)
    assert ts.dtype == torch.int64 and coef.dtype == torch.float32 and coef.shape == (M, 5)
    assert ts.tolist() == ts_list[:-1]
    want = _restated(ac, ts_list)
    # one fp32 rounding of the fp64 value (the two fp64 forms differ by a few fp64 ulps)
    np.testing.assert_allclose(coef.double().numpy(), want, rtol=2 ** -23, atol=0)
    assert coef[0, 4].item() == 0.0
    assert coef[-1, 2:].tolist() == [0.0, 1.0, 0.0]
    if M >= 3:
        assert (coef[1:-1, 4] != 0).all()


def test_interior_target_and_minus_one():
    ac = _ac("cosine", 1000)
    ts, coef = schedules.dpmpp_2m_table(ac, [999, 500, 100])
    assert ts.tolist() == [999, 500] and coef[0, 4].item() == 0.0 and coef[1, 4].item() != 0.0
    assert coef[1, 2].item() != 0.0 and coef[1, 3].item() != 1.0     # no sigma = 0 row here
    _, coef = schedules.dpmpp_2m_table(ac, [999, 500, -1])
    assert coef[1, 2:].tolist() == [0.0, 1.0, 0.0]
    s, r = coef[1, 0].item(), coef[1, 1].item()
    assert s == np.float32(math.sqrt(1 - float(ac[500]))) and r == np.float32(1 / math.sqrt(float(ac[500])))


@pytest.mark.parametrize("start_t", [1, 2, 5, 99, 999])
def test_public_timestep_rule(start_t):
    for M in sorted({1, 2, 3, 7, 20, start_t // 2 or 1, start_t}):
        if M > start_t:
            continue
        ts = schedules.dpmpp_timesteps(start_t, M)
        assert len(ts) == M + 1 and ts[-1] == -1 and ts[0] == start_t
        assert all(a > b for a, b in zip(ts, ts[1:]))
        assert ts[-2] >= 1
        # round(linspace(start_t, 0, M + 1))[:-1] with halves rounded up
        want = [int(math.floor(start_t * (M - i) / M + 0.5)) for i in range(M)]
        assert ts[:-1] == want
    assert schedules.dpmpp_timesteps(999, 20)[:4] == [999, 949, 899, 849]


@pytest.mark.parametrize("bad", [[999], [], [500, 500, -1], [100, 200, -1], [1000, 500, -1],
                                 [999, -1, 0], [999, -2], [999, 500, -3], [-1]])
def test_invalid_lists_raise(bad):
    with pytest.raises(ValueError):
        schedules.dpmpp_2m_table(_ac("cosine", 1000), bad)


@pytest.mark.parametrize("start_t,M", [(10, 0), (10, 11), (0, 1), (5, -1)])
def test_invalid_timestep_rule_raises(start_t, M):
    with pytest.raises(ValueError):
        schedules.dpmpp_timesteps(start_t, M)


def _diffusions():
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import \
        GaussianDiffusion as G25
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion as G2
    with contextlib.redirect_stdout(io.StringIO()):
        return (GaussianDiffusionLatent3D(torch.nn.Identity(), 3, timesteps=50),
                G2(torch.nn.Identity(), 8, timesteps=50), G25(torch.nn.Identity(), 8, timesteps=50))


@pytest.mark.parametrize("num_steps", [0, -3, 50, 51])
def test_invalid_num_steps_raise_before_any_draw(num_steps):
    """ValueError unless 1 <= num_steps <= start_t <= T - 1, raised before x_T is drawn (these CPU
    objects could not draw it)."""
    d3, d2, d25 = _diffusions()
    with pytest.raises(ValueError):
        d3.sample_dpmpp(2, 4, num_steps=num_steps)
    with pytest.raises(ValueError):
        d2.sample_dpmpp(2, num_steps=num_steps)
    with pytest.raises(ValueError):
        d25.sample_dpmpp(2, num_steps=num_steps)


@pytest.mark.parametrize("start_t,num_steps", [(50, 5), (-1, 1), (10, 11), (3, 0)])
def test_invalid_start_t_raises(start_t, num_steps):
    d3, _, _ = _diffusions()
    with pytest.raises(ValueError):
        d3.sample_from_dpmpp(torch.zeros(1, 3, 4, 4, 4), start_t, num_steps)


def test_valid_arguments_give_the_public_table():
    d3, _, _ = _diffusions()
    ts, coef = d3._dpmpp_table(49, 49)
    assert ts.tolist() == list(range(49, 0, -1)) and coef.shape == (49, 5)
    ts, _ = d3._dpmpp_table(1, 1)
    assert ts.tolist() == [1]


class _Stub:
    def sample(self, n, *a, **k):
        return torch.zeros(n)

    def sample_dpmpp(self, n, z_pos=None, num_steps=20):
        return torch.stack([torch.full((n,), float(num_steps)), z_pos, torch.rand(n)])


def test_sample_sharded_dispatches_by_method():
    from mri_image_generation_b200.parallel import sample_sharded
    z = torch.arange(4, dtype=torch.float32)
    got = sample_sharded(_Stub(), 4, base_seed=5, per_sample_kwargs={"z_pos": z},
                         method="sample_dpmpp", num_steps=7)
    torch.manual_seed(5)
    assert torch.equal(got, torch.stack([torch.full((4,), 7.0), z, torch.rand(4)]))
    assert torch.equal(sample_sharded(_Stub(), 3), torch.zeros(3))   # default stays sample()
