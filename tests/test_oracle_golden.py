"""CPU: pin the oracle (oracle/hmc_oracle.py) against fixtures produced by the UNMODIFIED reference
(oracle/gen_golden.py), and against the reference's own output under the same torch RNG state (oracle/ref_pins.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import cases, hmc_oracle as O, ref_pins

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _replay(case, d, ci, seed):
    tgt, kw = case['target'], dict(case['kw'])
    nuts = kw.pop('nuts', False)
    init = torch.from_numpy(d['init_%d' % ci])
    z = torch.from_numpy(d['z_%d' % ci])
    logu = torch.from_numpy(d['logu_%d' % ci])
    return O.sample_hmc(tgt, init, nuts=nuts, normals=z, log_uniforms=logu, **kw)


@pytest.mark.parametrize('name', sorted(cases.plain_cases()))
def test_oracle_reproduces_reference_fixture(name):
    """Oracle driven by the stored random stream returns the reference's chain.  Decisions must be identical;
    samples are compared exactly (same torch build) or to 1e-6 (another CPU's vectorised dot may round differently)."""
    torch.set_num_threads(1)
    case = cases.plain_cases()[name]
    d = np.load(os.path.join(GOLD, name + '.npz'))
    for ci, seed in enumerate(case['seeds']):
        res = _replay(case, d, ci, seed)
        assert list(np.array(res['accepted'], dtype=np.uint8)) == list(d['accepted_%d' % ci])
        got = torch.stack(res['samples']).numpy()
        np.testing.assert_allclose(got, d['samples_%d' % ci], rtol=1e-6, atol=1e-6)
        assert got.shape[0] == case['kw']['num_samples'] - case['kw']['burn']      # samplers.py:959, :1007
        assert np.array_equal(got[0], d['init_%d' % ci])                            # element 0 = params_init
        np.testing.assert_allclose(res['step_size'], d['final_step_size_%d' % ci], rtol=1e-6)


def test_init_recipe_matches_fixture():
    """multi_chain convention (util.py:386-389): manual_seed(seed) -> prior() reproduces the stored inits."""
    for name, case in cases.plain_cases().items():
        d = np.load(os.path.join(GOLD, name + '.npz'))
        for ci, seed in enumerate(case['seeds']):
            init = cases.make_init(case['init'], case['target'].dim, seed)
            assert np.array_equal(init.numpy(), d['init_%d' % ci])


def test_reference_reversibility_case():
    """tests/test_util.py:97-110 of the reference, restated on the oracle: 100 leapfrog steps forward, negate the
    momentum, 100 back.  The reference asserts bitwise return for ITS closure (MultivariateNormal); for the
    descriptor the trajectory must equal the reference's trajectory on the same descriptor and return to the start
    to fp32 round-off."""
    from hamiltorch_b200 import targets as T
    d = np.load(os.path.join(GOLD, 'ref_reversibility.npz'))
    tgt = T.GaussianDiag(torch.zeros(2), torch.tensor([.10, .10]))
    q0, p0, im = torch.tensor([1., 1.]), torch.tensor([1., 1.]), torch.tensor([1., 1.])
    qs, ps = O.leapfrog_hmc(tgt, q0, p0, 100, 0.1, im)
    np.testing.assert_allclose(torch.stack(qs).numpy(), d['fwd_q_desc'], rtol=0, atol=1e-6)
    np.testing.assert_allclose(torch.stack(ps).numpy(), d['fwd_p_desc'], rtol=0, atol=1e-6)
    qb, pb = O.leapfrog_hmc(tgt, qs[-1], -ps[-1], 100, 0.1, im)
    assert torch.allclose(qb[-1], q0, atol=5e-6)
    # the reference's own closure returns bitwise (stored by gen_golden from the reference run)
    assert np.array_equal(d['bwd_q_mvn'][-1], np.array([1., 1.], dtype=np.float32))


def test_dual_average_first_steps():
    """samplers.py:629-674 hand-checked: t=1, rho=0 -> alpha=1, H=(1/11)(delta-1), x=mu-sqrt(1)/.05*H."""
    eps, eps_bar, H = O.dual_average(0.0, 0, 0.1, 0.0, 1.0, 0.8)
    assert abs(H - (0.8 - 1.0) / 11) < 1e-15
    mu = float(torch.log(10 * torch.FloatTensor([0.1])))
    x = mu - (1 ** 0.5) / 0.05 * H
    assert abs(eps - float(torch.exp(torch.FloatTensor([x])))) < 1e-12
    assert abs(eps_bar - eps) < 1e-6          # t^-kappa = 1: eps_bar = exp(x)
    eps2, _, H2 = O.dual_average(float('nan'), 1, 0.1, H, eps_bar, 0.8)     # NaN rho -> alpha = 0 (:660-661)
    assert abs(H2 - ((1 - 1 / 12) * H + (1 / 12) * 0.8)) < 1e-15


def test_oracle_equals_reference_live():
    """Bit-for-bit: oracle.sample_hmc == hamiltorch.sample under the same torch RNG state (HMC and HMC_NUTS), against
    the reference's output stored by oracle/ref_pins.py."""
    torch.set_num_threads(1)
    d = np.load(ref_pins.PINS)
    for nuts in (False, True):
        tag = 'nuts' if nuts else 'hmc'
        o = ref_pins.oracle_gauss12(nuts)
        assert torch.equal(torch.from_numpy(d['gauss12_%s_samples' % tag]), torch.stack(o['samples']))
        if nuts:
            assert float(d['gauss12_nuts_extra']) == o['step_size']
        else:                                # the reference's acceptance rate
            rate = 1 - o['num_rejected'] / ref_pins.GAUSS12_KW['num_samples']
            assert abs(float(d['gauss12_hmc_extra']) - rate) < 1e-12


# ---- sampler=RMHMC: oracle/rmhmc_oracle.py ---------------------------------------------------------------------
@pytest.mark.parametrize('name', sorted(cases.rmhmc_cases()))
def test_rmhmc_oracle_reproduces_reference_fixture(name):
    """The RMHMC oracle driven by the stored stream returns the reference's chain (explicit / implicit, both metrics)."""
    from oracle import rmhmc_oracle as R
    torch.set_num_threads(1)
    case = cases.rmhmc_cases()[name]
    d = np.load(os.path.join(GOLD, name + '.npz'))
    explicit = case['integrator'] == 'EXPLICIT'
    kw = dict(num_samples=case['num_samples'], num_steps_per_sample=case['num_steps_per_sample'],
              step_size=case['step_size'], burn=case['burn'], jitter=case['jitter'], softabs_const=case['softabs_const'],
              integrator=R.EXPLICIT if explicit else R.IMPLICIT,
              metric={'SOFTABS': R.SOFTABS, 'HESSIAN': R.HESSIAN, 'JACOBIAN_DIAG': R.JACOBIAN_DIAG}[case['metric']])
    if explicit:
        kw['explicit_binding_const'] = case['explicit_binding_const']
    else:
        kw.update(fixed_point_threshold=case['fixed_point_threshold'],
                  fixed_point_max_iterations=case['fixed_point_max_iterations'])
    ci = 0
    res = R.sample_rmhmc(case['target'], torch.tensor(case['init']), normals=torch.from_numpy(d['z_%d' % ci]),
                         log_uniforms=torch.from_numpy(d['logu_%d' % ci]),
                         uniforms=torch.from_numpy(d['uniforms_%d' % ci]) if case['jitter'] is not None else None, **kw)
    assert list(np.array(res['accepted'], dtype=np.uint8)) == list(d['accepted_%d' % ci])
    np.testing.assert_allclose(torch.stack(res['samples']).numpy(), d['samples_%d' % ci], rtol=1e-5, atol=1e-5)


def test_cfg3_pin_fixture_rejects_logprob_errors_and_nan_retries():
    """tests/golden/cfg3_rmhmc_pin.npz: BASELINE config 3 chains of the UNMODIFIED reference (torch global RNG) that
    reject, raise LogProbError and run the NaN-retry loop of samplers.py:402-410; the oracle under the same seed must
    return the same chain -- this is what pins those paths (and what caught the oracle's off-by-one in the retry
    loop).  Exact on this torch build; decisions + 1e-5 elsewhere."""
    from oracle import gen_cfg3 as G, rmhmc_oracle as R
    torch.set_num_threads(1)
    d = np.load(os.path.join(GOLD, 'cfg3_rmhmc_pin.npz'))
    assert sum(int(d['diverged_%d' % c].sum()) for c in range(len(d['seeds']))) > 0
    assert sum(int(d['nan_retries_%d' % c].sum()) for c in range(len(d['seeds']))) > 0
    from hamiltorch_b200 import targets as T
    import contextlib
    import io
    ci = 0
    with contextlib.redirect_stdout(io.StringIO()):
        torch.manual_seed(int(d['seeds'][ci]))
        res = R.sample_rmhmc(T.Funnel(2), torch.tensor(G.INIT), num_samples=25, burn=3, **G.KW)
    assert list(np.array(res['accepted'], dtype=np.uint8)) == list(d['accepted_%d' % ci])
    assert list(np.array(res['diverged'], dtype=np.uint8)) == list(d['diverged_%d' % ci])
    assert list(res['nan_retries']) == list(d['nan_retries_%d' % ci])
    np.testing.assert_allclose(torch.stack(res['samples']).numpy(), d['samples_%d' % ci], rtol=1e-5, atol=1e-5)


def test_cfg4_oracle_equals_reference_live():
    """BASELINE config 4 exactly (oracle/cfg4.py): hamiltorch.sample_split_model == the oracle, bit for bit, against
    the reference's output stored by oracle/ref_pins.py."""
    torch.set_num_threads(1)
    d = np.load(ref_pins.PINS)
    assert torch.equal(torch.from_numpy(d['cfg4_samples']), torch.stack(ref_pins.oracle_cfg4()['samples']))
