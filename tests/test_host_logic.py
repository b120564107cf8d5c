"""CPU-only checks of the host layer: config loader, parameter block, C-ABI exports."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_config_defaults_match_reference_dataclass():
    from dart_planner_b200.config import SE3MPCConfig, make_params
    c = SE3MPCConfig()
    # reference tests/test_sitl_unit_tests.py:43-48 pins these
    assert c.prediction_horizon == 6 and c.max_iterations == 15 and c.convergence_tolerance == 5e-2
    p = make_params(c, dt=1 / 400)
    assert p.mass * p.gravity == pytest.approx(14.715)
    assert p.tilt_thrust == pytest.approx(25.0 * math.sin(math.pi / 4))
    assert (p.gtol, p.ftol) == (0.05, 0.5)
    assert p.struct_size == C.sizeof(type(p))


def test_config_accepts_quantity_like():
    from dart_planner_b200.config import SE3MPCConfig

    class Q:
        def __init__(self, m):
            self.magnitude = m

        def to(self, unit):
            return self

    c = SE3MPCConfig(max_velocity=Q(7.5), max_thrust=Q(20.0))
    assert c.max_velocity == 7.5 and c.max_thrust == 20.0


def test_yaml_loader():
    from dart_planner_b200.config import load_airframe, load_planner_config
    cfg, mass = load_planner_config()
    assert cfg.prediction_horizon == 8 and cfg.dt == 0.1 and mass == 1.5   # defaults.yaml / airframes.yaml
    assert cfg.position_weight == 100.0 and cfg.velocity_weight == 10.0
    cfg, mass = load_planner_config(airframe="racing_drone", prediction_horizon=10)
    assert mass == 0.8 and cfg.prediction_horizon == 10
    assert load_airframe("dji_f550")["type"] == "hexacopter"
    assert load_airframe("dji_f450")["type"] == "quadcopter"       # inherited through `extends`
    with pytest.raises(KeyError):
        load_planner_config(airframe="nope")
    with pytest.raises(KeyError):
        load_planner_config(bogus_key=1)


def test_header_symbols_are_exported():
    """Every function include/dart_se3mpc.h declares is exported by the built library.
    Loading does not touch the GPU."""
    lib_path = os.path.join(ROOT, "dart_planner_b200", "lib", "libdart_se3mpc.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    hdr = open(os.path.join(ROOT, "include", "dart_se3mpc.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(dart_[a-z0-9_]+)\s*\(", hdr))
    assert {"dart_se3mpc_solve_batch", "dart_map_trace_ray_batch"} <= declared
    L = C.CDLL(lib_path)
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in the header but not exported"
    L.dart_abi_version.restype = C.c_int
    assert L.dart_abi_version() == 1
    from dart_planner_b200 import _cabi
    assert set(_cabi.EXPORTS) == declared
    # default params from C agree with the Python mirror
    p = _cabi.Params()
    L.dart_se3mpc_default_params(C.byref(p))
    from dart_planner_b200.config import SE3MPCConfig, make_params
    q = make_params(SE3MPCConfig(), dt=1 / 400)
    for f, _ in _cabi.Params._fields_:
        assert getattr(p, f) == pytest.approx(getattr(q, f)), f


def test_bad_arguments_are_rejected_without_a_gpu():
    from dart_planner_b200 import _cabi
    lib_path = _cabi.LIB_PATH
    if not os.path.exists(lib_path):
        pytest.skip("library not built")
    L = _cabi.lib()
    p = _cabi.Params()
    L.dart_se3mpc_default_params(C.byref(p))
    p.horizon = 65
    assert L.dart_se3mpc_solve_batch(C.byref(p), 1, 1, *([None] * 17)) == _cabi.DART_E_UNSUPPORTED
    p.horizon = 8
    p.max_corrections = 11
    assert L.dart_se3mpc_solve_batch(C.byref(p), 1, 1, *([None] * 17)) == _cabi.DART_E_UNSUPPORTED
    p.max_corrections = 10
    # maxls must be positive, as in SciPy.  An empty batch with valid inputs returns after the
    # argument checks, so DART_OK there tells the accepted values from the refused ones
    buf = np.zeros(3)
    empty = lambda: L.dart_se3mpc_solve_batch(C.byref(p), 0, 0, *([buf.ctypes.data] * 3), *([None] * 14))  # noqa: E731
    for maxls, want in ((0, _cabi.DART_E_BADARG), (-1, _cabi.DART_E_BADARG), (1, _cabi.DART_OK), (20, _cabi.DART_OK)):
        p.max_linesearch = maxls
        assert empty() == want, maxls
    p.max_linesearch = 20
    assert L.dart_se3mpc_solve_batch(C.byref(p), 1, 1, *([None] * 17)) == _cabi.DART_E_BADARG  # null inputs
    p.struct_size = 8
    assert L.dart_se3mpc_solve_batch(C.byref(p), 1, 1, *([None] * 17)) == _cabi.DART_E_BADARG


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under dart_planner_b200/ may reference it."""
    pkg = os.path.join(ROOT, "dart_planner_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "oracle/" not in src, f


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import dart_planner_b200 as dp
    with pytest.raises(RuntimeError, match="CUDA"):
        dp.plan_batch(np.zeros((2, 3)), np.zeros((2, 3)), np.ones((2, 3)))


def test_integration_stub_matches_the_header():
    """The ctypes structure printed in INTEGRATION.md (what a maintainer of the reference would
    paste) has exactly the fields of dart_se3mpc_params, in order."""
    from dart_planner_b200 import _cabi
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = doc[doc.index("class _Params(C.Structure)"):doc.index("def _solve_se3_mpc(self, current_state)")]
    names = re.findall(r'"([a-z_0-9]+)"', block)
    assert names == [f for f, _ in _cabi.Params._fields_]
    hdr = open(os.path.join(ROOT, "include", "dart_se3mpc.h")).read()
    struct = hdr[hdr.index("typedef struct dart_se3mpc_params {"):hdr.index("} dart_se3mpc_params;")]
    struct = re.sub(r"/\*.*?\*/", "", struct, flags=re.S)
    declared = []
    for decl in re.findall(r"(?:int32_t|double)\s+([^;]+);", struct):
        declared += [n.strip() for n in decl.split(",")]
    assert declared == names
