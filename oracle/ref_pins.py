"""ORACLE -- TEST INFRASTRUCTURE ONLY.  What the UNMODIFIED reference returns on the cases that pin the oracle and the
host-side API to it directly, stored so that the tests compare against it without the reference tree:

  tests/golden/ref_signatures.json  positional parameters and defaults of the reference's sampler entry points
  tests/golden/ref_pins.npz         hamiltorch.sample on a 12-D diagonal Gaussian (HMC and HMC_NUTS, torch.manual_seed)
                                    and hamiltorch.sample_split_model at BASELINE config 4 exactly (oracle/cfg4.py)

    python -m oracle.ref_pins        (needs the reference tree, see oracle/ref_import.py)

Before it writes, it asserts that the oracle, run here through the functions below, is bit-identical to the reference.
"""
import inspect
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import cfg4, hmc_oracle as O           # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
SIGNATURES = os.path.join(GOLD, 'ref_signatures.json')
PINS = os.path.join(GOLD, 'ref_pins.npz')
SIGNATURE_FUNCTIONS = ('sample', 'leapfrog', 'hamiltonian', 'gibbs', 'acceptance', 'adaptation')
GAUSS12_KW = dict(num_samples=25, num_steps_per_sample=4, step_size=0.4, burn=8)
GAUSS12_SEED, CFG4_SEED, CFG4_SAMPLES = 99, 5, 4


def encode_default(d):
    """A parameter default as JSON: {'required': true} for none, {'enum': name} for a Sampler / Integrator / Metric."""
    if d is inspect.Parameter.empty:
        return {'required': True}
    if hasattr(d, 'name'):
        return {'enum': d.name}
    return d


def gauss12_target():
    from hamiltorch_b200 import targets as T
    return T.GaussianDiag(torch.linspace(-1, 1, 12), 0.3 + torch.rand(12, generator=torch.Generator().manual_seed(0)))


def oracle_gauss12(nuts):
    """oracle.sample_hmc under the torch RNG state hamiltorch.sample is given in run_reference()."""
    torch.manual_seed(GAUSS12_SEED)
    return O.sample_hmc(gauss12_target(), torch.zeros(12), nuts=nuts, **GAUSS12_KW)


def _cfg4_loader(X, y):
    import torch.utils.data as tud
    return tud.DataLoader(tud.TensorDataset(X, y), batch_size=cfg4.N_ROWS // cfg4.M, shuffle=False)


def _cfg4_kw(D):
    return dict(num_samples=CFG4_SAMPLES, num_steps_per_sample=cfg4.L, step_size=cfg4.EPS, inv_mass=torch.ones(D))


def oracle_cfg4():
    """The oracle's config-4 chain under the torch RNG state sample_split_model is given in run_reference()."""
    from hamiltorch_b200 import util
    model, X, y = cfg4.problem()
    descs = cfg4.descriptors(model, X, y)
    init = util.flatten(model).detach().clone()
    torch.manual_seed(CFG4_SEED)
    next(iter(_cfg4_loader(X, y)))           # the DataLoader's base-seed draw (see oracle/gen_golden.py)
    return O.sample_hmc(descs, init, split_scheme=O.SPLIT_SYM, **_cfg4_kw(descs[0].dim))


def run_reference(ref):
    out = {}
    for nuts in (False, True):
        tag = 'nuts' if nuts else 'hmc'
        torch.manual_seed(GAUSS12_SEED)
        r = ref.sample(log_prob_func=gauss12_target(), params_init=torch.zeros(12), verbose=False, debug=2,
                       sampler=ref.Sampler.HMC_NUTS if nuts else ref.Sampler.HMC, **GAUSS12_KW)
        o = oracle_gauss12(nuts)
        assert torch.equal(torch.stack(r[0]), torch.stack(o['samples'])), tag
        out['gauss12_%s_samples' % tag] = torch.stack(r[0]).numpy()
        out['gauss12_%s_extra' % tag] = np.float64(r[1])       # acceptance rate (HMC) / adapted step size (NUTS)
        if nuts:
            assert r[1] == o['step_size']
    model, X, y = cfg4.problem()
    init = ref.util.flatten(model).detach().clone()
    torch.manual_seed(CFG4_SEED)
    r = ref.sample_split_model(model, _cfg4_loader(X, y), params_init=init, num_splits=cfg4.M,
                               model_loss='regression', tau_out=cfg4.TAU_OUT, integrator=ref.Integrator.SPLITTING,
                               verbose=False, **_cfg4_kw(init.numel()))
    assert torch.equal(torch.stack(r), torch.stack(oracle_cfg4()['samples'])), 'config 4'
    out['cfg4_samples'] = torch.stack(r).numpy()
    return out


def main():
    from oracle.ref_import import import_reference
    torch.set_num_threads(1)
    ref = import_reference()
    lines = []
    for fn in SIGNATURE_FUNCTIONS:                   # one function per line
        params = inspect.signature(getattr(ref.samplers, fn)).parameters.values()
        lines.append('%s: %s' % (json.dumps(fn), json.dumps([[p.name, encode_default(p.default)] for p in params])))
    with open(SIGNATURES, 'w') as f:
        f.write('{\n%s\n}\n' % ',\n'.join(lines))
    np.savez_compressed(PINS, **run_reference(ref))
    print('wrote', SIGNATURES, PINS)


if __name__ == '__main__':
    main()
