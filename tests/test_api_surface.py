"""CPU: the host-side mirror keeps the reference's names, signatures, defaults and error behaviour
(SURVEY.md section 8b); and refuses -- loudly -- what cannot run in a kernel."""
import inspect
import json

import pytest
import torch

import hamiltorch_b200 as hb
from hamiltorch_b200 import targets as T
from oracle import ref_pins


def test_exports():
    for name in ('sample', 'Sampler', 'Integrator', 'Metric', 'set_random_seed'):
        assert hasattr(hb, name)
    for name in ('flatten', 'unflatten', 'update_model_params_in_place', 'setup_chain', 'multi_chain',
                 'LogProbError', 'has_nan_or_inf'):
        assert hasattr(hb.util, name)
    assert [e.name for e in hb.Sampler] == ['HMC', 'RMHMC', 'HMC_NUTS']
    assert [(e.name, e.value) for e in hb.Integrator] == [('EXPLICIT', 1), ('IMPLICIT', 2), ('S3', 3),
                                                          ('SPLITTING', 4), ('SPLITTING_RAND', 5),
                                                          ('SPLITTING_KMID', 6)]
    assert [e.name for e in hb.Metric] == ['HESSIAN', 'SOFTABS', 'JACOBIAN_DIAG']


def test_signatures_match_reference():
    """Positional parameters and defaults of the reference's sampler entry points, as oracle/ref_pins.py stored them."""
    with open(ref_pins.SIGNATURES) as f:
        ref = json.load(f)
    assert tuple(ref) == ref_pins.SIGNATURE_FUNCTIONS
    for fn, rp in ref.items():
        op = inspect.signature(getattr(hb.samplers, fn)).parameters
        pos = [p for p in op.values() if p.kind != inspect.Parameter.KEYWORD_ONLY]
        assert [p.name for p in pos] == [name for name, _ in rp], fn
        for p, (_, rd) in zip(pos, rp):
            assert ref_pins.encode_default(p.default) == rd, (fn, p.name)


def test_sample_argument_errors_match_reference():
    tgt = T.GaussianIso(4)
    with pytest.raises(RuntimeError, match='params_init must be a 1d tensor'):
        hb.sample(tgt, torch.zeros(2, 4))
    with pytest.raises(RuntimeError, match='burn must be less than num_samples'):
        hb.sample(tgt, torch.zeros(4), num_samples=5, burn=5)
    with pytest.raises(RuntimeError, match='burn must be greater than 0 for NUTS'):
        hb.sample(tgt, torch.zeros(4), sampler=hb.Sampler.HMC_NUTS)
    with pytest.raises(RuntimeError, match='must be list'):
        hb.sample(tgt, torch.zeros(4), integrator=hb.Integrator.SPLITTING, rng='philox')
    with pytest.raises(RuntimeError, match='not implemented for RMHMC'):
        hb.sample(tgt, torch.zeros(4), sampler=hb.Sampler.RMHMC, pass_grad=torch.zeros(4))


def test_opaque_callable_is_refused():
    with pytest.raises(TypeError, match='no CPU fallback'):
        hb.sample(lambda x: -(x * x).sum(), torch.zeros(4))


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU failure mode')
def test_no_gpu_fails_loudly():
    from hamiltorch_b200._native import NativeError
    with pytest.raises(NativeError, match='no CPU fallback'):
        hb.sample(T.GaussianIso(4), torch.zeros(4), verbose=False)


def test_flatten_unflatten_roundtrip():
    """The reference's tests/test_util.py:12-24 on our util."""
    import torch.nn as nn
    model = nn.Linear(4, 4)
    flat = hb.util.flatten(model)
    new_model = nn.Linear(4, 4)
    hb.util.update_model_params_in_place(new_model, hb.util.unflatten(new_model, flat))
    assert torch.all(torch.eq(flat, hb.util.flatten(new_model)))
    assert flat.shape == (20,)
    assert torch.equal(flat[:16].view(4, 4), model.weight)       # weight (o,i) row-major then bias


def test_nuts_table_matches_python_doubles():
    from hamiltorch_b200 import engine
    tab = engine.nuts_table(3)
    for n in range(4):
        t = n + 1
        assert tab[n, 0].item() == 1 - (1 / (t + 10))
        assert tab[n, 1].item() == (1 / (t + 10))
        assert tab[n, 2].item() == (t ** 0.5) / 0.05
        assert tab[n, 3].item() == t ** -0.75
        assert tab[n, 4].item() == 1 - t ** -0.75


def test_sink_and_rmhmc_routing_errors_are_raised_on_the_host():
    """Argument checks that must fire before any CUDA work (so they are testable without a GPU): the sample sink is only
    wired into the element-wise persistent kernel; RMHMC at D > 64 needs a constant metric."""
    import pytest
    import torch
    import hamiltorch_b200 as hb
    from hamiltorch_b200 import targets as T
    D = 80
    full = T.GaussianFull(torch.zeros(D), cov=torch.eye(D, dtype=torch.float64) * 2)
    for kw in (dict(thin=2), dict(moments=True), dict(keep_samples=False), dict(store_on_GPU=False)):
        with pytest.raises(NotImplementedError):
            hb.sample_chains(full, torch.zeros(2, D), num_samples=5, **kw)
    with pytest.raises(NotImplementedError):                       # position-dependent metric at D > 64
        hb.sample_chains(T.Funnel(D), torch.zeros(2, D), num_samples=5, sampler=hb.Sampler.RMHMC,
                         integrator=hb.Integrator.EXPLICIT)
    with pytest.raises(NotImplementedError):                       # jitter makes the metric a per-call random matrix
        hb.sample_chains(full, torch.zeros(2, D), num_samples=5, jitter=1e-3, sampler=hb.Sampler.RMHMC,
                         integrator=hb.Integrator.EXPLICIT)
    with pytest.raises(RuntimeError):                              # burn >= num_samples (samplers.py:928-929)
        hb.sample_chains(T.GaussianIso(8), torch.zeros(2, 8), num_samples=5, burn=5)


def test_bench_clock_sampler_degrades_without_a_gpu():
    """bench.py's clock sampler never raises: without NVML / nvidia-smi it reports that instead of clocks."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(root, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    s = mod.ClockSampler(0)
    s.start()
    out = s.stop()
    assert set(out) >= {'sm_mhz', 'sm_max_mhz', 'reasons'}


def test_full_inv_mass_operands_are_cached_per_tensor_object_and_version():
    """engine.native_mass: a 2-D / block-list inv_mass is inverted and factorised once per tensor OBJECT and version
    (samplers.py:942-952 does it once per sample() call); an in-place update or another tensor builds new operands."""
    import torch
    from hamiltorch_b200 import engine
    A = torch.eye(6) * 2.0
    m1 = engine.native_mass(A, 6, 'cpu')
    assert engine.native_mass(A, 6, 'cpu') is m1
    assert m1.ref() is not None and m1.kind == 2
    A.mul_(2.0)                                              # version bump
    m2 = engine.native_mass(A, 6, 'cpu')
    assert m2 is not m1
    assert torch.allclose(m2._keep['tril'], torch.eye(6) * 0.5)
    assert engine.native_mass(A.clone(), 6, 'cpu') is not m2
    blocks = [torch.eye(2), torch.eye(4) * 4.0]
    b1 = engine.native_mass(blocks, 6, 'cpu')
    assert engine.native_mass(blocks, 6, 'cpu') is b1
    assert engine.native_mass(torch.ones(6), 6, 'cpu') is not engine.native_mass(torch.ones(6), 6, 'cpu')   # 1-D: cheap, uncached
