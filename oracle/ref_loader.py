"""Load the reference's real source files (``acq.py``, ``scalers.py``, ``base_model.py``, ...) by path.

TEST INFRASTRUCTURE ONLY: used by ``oracle/make_golden.py`` alone, to record the reference's own outputs as
the fixtures under ``tests/golden/``.  The tests, smoke() and bench.py read those fixtures and never the
reference sources, so the repository runs and tests without a copy of the reference.

``import hebo`` itself fails here (pymoo / gpytorch missing: evolution_optimizer.py:14, gp.py:14);
the files below import only torch/numpy/sklearn and load unmodified under stub parent packages.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

REF_ROOT = "/root/reference/HEBO/hebo"


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "acquisitions", "acq.py"))


def _load(modname: str, relpath: str):
    if modname in sys.modules:
        return sys.modules[modname]
    spec = importlib.util.spec_from_file_location(modname, os.path.join(REF_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[modname] = mod
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    """Returns a namespace with the reference's MACE, Mean, Sigma, BaseModel, scalers."""
    if not available():
        raise RuntimeError("/root/reference is not present")
    for pkg in ("_hebo_ref", "_hebo_ref.models", "_hebo_ref.acquisitions"):
        if pkg not in sys.modules:
            m = types.ModuleType(pkg)
            m.__path__ = []          # mark as package so relative imports resolve
            sys.modules[pkg] = m
    scalers = _load("_hebo_ref.models.scalers", "models/scalers.py")
    base_model = _load("_hebo_ref.models.base_model", "models/base_model.py")
    acq = _load("_hebo_ref.acquisitions.acq", "acquisitions/acq.py")
    ns = types.SimpleNamespace(MACE=acq.MACE, Mean=acq.Mean, Sigma=acq.Sigma, LCB=acq.LCB,
                               Acquisition=acq.Acquisition, BaseModel=base_model.BaseModel,
                               TorchMinMaxScaler=scalers.TorchMinMaxScaler,
                               TorchStandardScaler=scalers.TorchStandardScaler)
    return ns


def load_file(modname: str, relpath: str, stubs=()):
    """Load one reference source file unmodified, with the parent modules it imports but does not use replaced by
    stubs: ``stubs`` lists (module name, names of placeholder classes it must provide)."""
    saved = {}
    for name, attrs in stubs:
        saved[name] = sys.modules.get(name)
        m = types.ModuleType(name)
        m.__path__ = []
        for k in attrs:
            setattr(m, k, type(k, (), {}))
        sys.modules[name] = m
    try:
        return _load(modname, relpath)
    finally:
        for name, old in saved.items():
            if old is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = old


def load_design_space():
    """The reference's DesignSpace class (design_space/*.py, loaded as one package)."""
    pkg = "_hebo_ref_ds"
    if pkg not in sys.modules:
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(REF_ROOT, "design_space")]
        sys.modules[pkg] = m
    for mod in ("param", "numeric_param", "integer_param", "pow_param", "categorical_param", "bool_param",
                "pow_integer_param", "int_exponent_param", "step_int", "design_space"):
        _load(f"{pkg}.{mod}", os.path.join("design_space", mod + ".py"))
    return sys.modules[f"{pkg}.design_space"].DesignSpace
