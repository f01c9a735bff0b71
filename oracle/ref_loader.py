"""TEST INFRASTRUCTURE ONLY -- loader for the REAL reference closures.

Imports the reference's own ``define_model_log_prob`` factories from a checkout
of the original VI-HMC project so that golden vectors can be produced from
reference code rather than from a restatement.  The checkout is looked for in
``oracle/_ref/`` (ignored by git) or wherever ``VIHMC_REFERENCE_ROOT`` points.
The reference is not part of this repository: ``oracle/make_golden.py`` needs
it, and the tests compare with its stored outputs (tests/golden/) and re-run it
live only when it is present.

Obstacles handled here (SURVEY.md section 8(c) "Gotchas"):
  * ``matplotlib`` and ``hamiltorch`` are absent  -> stubbed in ``sys.modules``;
  * every script does ``import config as cfg`` / ``import util`` by bare name and
    the four script directories each own a different ``config``/``util`` ->
    modules are loaded one directory at a time with a clean ``sys.modules``;
  * ``import util`` reseeds every RNG from the wall clock (util.py:13-25) ->
    callers must seed AFTER loading;
  * closures ``torch.load`` VI artefacts from ``cfg.prior_file`` at construction
    (main_VI_HMC.py:76-79) -> ``cfg.prior_file``/``cfg.prior_uid`` are pointed at
    a temporary directory holding synthetic artefacts.
"""
from __future__ import annotations

import contextlib
import importlib
import io
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("VIHMC_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")

_LOCAL_MODULES = ("config", "config_splitting", "config_sens", "util", "utils", "my_make_func", "model", "metrics", "bayesian_model",
                  "layers", "layers.BBB", "layers.BBB.BBBLinear", "layers.BBB.BBBConv", "layers.BBB_LRT", "layers.BBB_LRT.BBBLinear",
                  "layers.BBB_LRT.BBBConv", "layers.misc")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "Neural_network", "VI_HMC"))


def _install_stubs() -> None:
    """Stub the two absent third-party imports; nothing in them is called by the closures."""
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        mpl.rcParams = {}
        mpl.use = lambda *a, **k: None
        plt = types.ModuleType("matplotlib.pyplot")
        plt.rcParams = {}
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    if "hamiltorch" not in sys.modules:
        ham = types.ModuleType("hamiltorch")
        samplers = types.ModuleType("hamiltorch.samplers")

        class _Enum:  # attribute access only (Sampler.HMC etc. are evaluated at call sites we never run)
            HMC = 1
            RMHMC = 2
            HMC_NUTS = 3
            IMPLICIT = 1
            EXPLICIT = 2
            SPLITTING = 3

        samplers.Sampler = _Enum
        samplers.Integrator = _Enum
        ham.samplers = samplers
        ham.util = types.ModuleType("hamiltorch.util")
        sys.modules["hamiltorch"] = ham
        sys.modules["hamiltorch.samplers"] = samplers
        sys.modules["hamiltorch.util"] = ham.util


def load_script(rel_dir: str, script: str, alias: str):
    """Import ``<REFERENCE_ROOT>/<rel_dir>/<script>.py`` under the module name ``alias``.

    The script's bare-name siblings (config, util, my_make_func, model) are resolved from its own
    directory and then renamed out of the way (``alias.config`` ...) so another script directory
    can be loaded afterwards.  Returns the module; its ``cfg`` attribute is the script's own config.
    """
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}: put a checkout of the original VI-HMC project there "
                           "or point VIHMC_REFERENCE_ROOT at one")
    _install_stubs()
    directory = os.path.join(REFERENCE_ROOT, rel_dir)
    saved = {name: sys.modules.pop(name) for name in _LOCAL_MODULES if name in sys.modules}
    cwd = os.getcwd()
    sys.path.insert(0, directory)
    sys.dont_write_bytecode, old_dwb = True, sys.dont_write_bytecode  # reference tree is read-only
    try:
        os.chdir(directory)  # get_data() uses ../Data relative paths (main_VI_HMC.py:270)
        with contextlib.redirect_stdout(io.StringIO()):  # configs print L at import
            spec = importlib.util.spec_from_file_location(alias, os.path.join(directory, script + ".py"))
            module = importlib.util.module_from_spec(spec)
            sys.modules[alias] = module
            spec.loader.exec_module(module)
    finally:
        os.chdir(cwd)
        sys.path.remove(directory)
        sys.dont_write_bytecode = old_dwb
        for name in _LOCAL_MODULES:
            mod = sys.modules.pop(name, None)
            if mod is not None:
                sys.modules[f"{alias}.{name}"] = mod
        sys.modules.update(saved)
    return module


def load_bnn_vi_hmc():
    """Neural_network/VI_HMC/main_VI_HMC.py (define_model_log_prob :28-153)."""
    return load_script("Neural_network/VI_HMC", "main_VI_HMC", "ref_bnn_vi_hmc")


def load_deeponet_vi_hmc():
    """Operator_network/VI_HMC/main_VI_HMC_burgers.py (define_model_log_prob :27-180)."""
    return load_script("Operator_network/VI_HMC", "main_VI_HMC_burgers", "ref_don_vi_hmc")


def load_deeponet_split_hmc():
    """Operator_network/HMC/main_HMC_splitting.py (define_model_log_prob :79-206, split :209-258)."""
    return load_script("Operator_network/HMC", "main_HMC_splitting", "ref_don_split_hmc")


def load_bnn_data():
    """The bundled 20-point regression set, Neural_network/Data/{x,y}_{train,val}."""
    import torch

    d = os.path.join(REFERENCE_ROOT, "Neural_network", "Data")
    return tuple(torch.load(os.path.join(d, n)) for n in ("x_train", "y_train", "x_val", "y_val"))
