"""ORACLE -- TEST INFRASTRUCTURE ONLY.

Imports the UNMODIFIED reference (AdamCobb/hamiltorch @ 19b627b) from REFERENCE_ROOT.  Only the fixture generators
(oracle/gen_golden.py, oracle/gen_cfg3.py, oracle/ref_pins.py) call this; the tests, smoke() and bench.py compare
against what they stored under tests/golden/ and never need the reference tree.

The reference needs ``termcolor`` (util.py:4, used only by eval_print) which is not installed here; a two-line
shim module is injected into sys.modules (SURVEY.md section 8c).  torch.distributions argument validation is
switched off because modern torch turns the notebook funnel's scale underflow into a ValueError (section 8a).
"""
import os
import sys
import types

REFERENCE_ROOT = '/root/reference'


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'hamiltorch'))


def import_reference():
    if not reference_available():
        raise ImportError('reference tree not present at ' + REFERENCE_ROOT)
    if 'termcolor' not in sys.modules:
        shim = types.ModuleType('termcolor')
        shim.colored = lambda s, *a, **k: s
        sys.modules['termcolor'] = shim
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import torch
    torch.distributions.Distribution.set_default_validate_args(False)
    import hamiltorch  # noqa: E402  (the reference package)
    if not hamiltorch.__file__.startswith(REFERENCE_ROOT):
        raise ImportError('imported a hamiltorch that is not the reference: ' + hamiltorch.__file__)
    return hamiltorch
