"""ORACLE -- TEST INFRASTRUCTURE ONLY.  BASELINE config 4 (SURVEY 8d) as the oracle sees it: Linear(64,128)-ReLU-
Linear(128,1) Bayesian regression (D=8449), N=1024 rows in M=4 splits of 256, symmetric split HMC (samplers.py:494-547),
eps=5e-4, L=10, inv_mass=ones(D), tau_out=100, tau_list=[1,1,1,1].

The fixture would be 27 MB per 8 x 100 chain block, so the GPU tests run this oracle LIVE on the GPU box's host cores
(one process per chain); the random stream of a chain is a seeded CPU torch.Generator, identical on every machine with
this torch build.  sample_hmc's split branch is pinned bit-identical to the unmodified reference by
oracle/gen_golden.py (tests/golden/mlp_split_*.npz) and, at this exact configuration, by oracle/ref_pins.py
(tests/test_oracle_golden.py::test_cfg4_oracle_equals_reference_live)."""
import torch

M, L, EPS, TAU_OUT, N_ROWS, N_IN, HID = 4, 10, 5e-4, 100., 1024, 64, 128


def problem():
    """(model, X, y): X ~ N(0,I) (1024 x 64), y = sin(X w / 8) + 0.1 N(0,1), torch.manual_seed(0) (SURVEY 8d cfg 4)."""
    import torch.nn as nn
    g = torch.Generator().manual_seed(0)
    X = torch.randn(N_ROWS, N_IN, generator=g)
    w = torch.randn(N_IN, 1, generator=g)
    y = torch.sin(X @ w / 8) + 0.1 * torch.randn(N_ROWS, 1, generator=g)
    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(N_IN, HID), nn.ReLU(), nn.Linear(HID, 1))
    return model, X, y


def descriptors(model, X, y):
    from hamiltorch_b200 import targets as T
    B = N_ROWS // M
    return [T.MLPRegression.from_model(model, X[m * B:(m + 1) * B], y[m * B:(m + 1) * B], None, TAU_OUT, prior_scale=M)
            for m in range(M)]


def stream(seed, S, D, flat):
    """(init, normals (S,D), log_uniforms (S,)) of chain `seed`."""
    g = torch.Generator().manual_seed(4000 + seed)
    init = flat + 0.01 * torch.randn(D, generator=g)
    z = torch.randn(S, D, generator=g)
    logu = torch.log(torch.rand(S, generator=g))
    return init, z, logu


def run_chain(args):
    """One chain through the oracle; returns numpy arrays (samples (S,D), accepted (S,), ham (S,2)).  perturb=1 moves
    params_init by one ulp per element (random sign): how far the REFERENCE itself drifts under fp32 round-off."""
    seed, S, perturb = (tuple(args) + (0,))[:3]
    import numpy as np
    torch.set_num_threads(1)
    from hamiltorch_b200 import util
    from oracle import hmc_oracle as O
    model, X, y = problem()
    descs = descriptors(model, X, y)
    D = descs[0].dim
    init, z, logu = stream(seed, S, D, util.flatten(model).detach().clone())
    if perturb:
        sign = torch.sign(torch.randn(D, generator=torch.Generator().manual_seed(99 + seed)))
        init = init * (1 + 1.1920929e-07 * sign)
    r = O.sample_hmc(descs, init, num_samples=S, num_steps_per_sample=L, step_size=EPS, inv_mass=torch.ones(D),
                     split_scheme=O.SPLIT_SYM, normals=z, log_uniforms=logu)
    return (torch.stack(r['samples']).numpy(), np.array(r['accepted'], np.uint8),
            np.stack([r['ham_old'], r['ham_new']], 1))
