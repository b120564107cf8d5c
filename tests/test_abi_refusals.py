"""The argument checks of every solve entry of the C ABI, without a GPU.

With B = 0 every entry returns right after its checks: DART_OK tells an accepted argument set
from a refused one, and no pointer is dereferenced (the non-NULL pointers below point nowhere).
One table of argument combinations runs against every entry; `expected` restates, entry by
entry and in order, the checks the header documents.
"""
import ctypes as C
import math
import os

import pytest

from dart_planner_b200 import _cabi

OK, BAD, UNS = _cabi.DART_OK, _cabi.DART_E_BADARG, _cabi.DART_E_UNSUPPORTED
PTR = 1 << 12                    # non-NULL, 128-byte aligned, never read at B = 0
ROLLOUT = {3, 4, 6, 7, 8}        # thrust-only variables: horizons up to 16, no warm == 2
GRID_PEN = {2, 4}                # the grid penalty
SM_DOUBLES = 495                 # the per-problem shared block (se3mpc_core.cuh, m = 10)
DT = 1.0 / 400.0

ENTRIES = ["solve_batch", "solve_batch_map", "solve_batch_spheres", "solve_batch_track", "solve_batch_rows",
           "closed_loop_step", "closed_loop_step_map", "closed_loop_step_spheres", "closed_loop_step_track",
           "solve_batch_host", "solve_batch_host_spheres", "solve_vjp_batch", "extract_batch", "row_stride"]
FAMILY = {"solve_batch_spheres": "spheres", "closed_loop_step_spheres": "spheres",
          "solve_batch_host_spheres": "spheres", "solve_batch_track": "track", "closed_loop_step_track": "track"}


def need_stride(N, kind):
    """row_stride_doubles: the packed row, padded to 16 doubles; 0 if it does not fit the block."""
    st = -(-((3 if kind == 1 else 9 if kind == 2 else 19) * N + 4) // 16) * 16
    return st if st <= SM_DOUBLES else 0


def base(mode, N):
    grid = dict(nx=4, ny=4, nz=4, resolution=0.5, occ=PTR, cell_bytes=0)
    return dict(mode=mode, N=N, dt=DT, B=0, ld=0, p0=PTR, v0=PTR, goal=PTR, x=PTR, status=PTR, T=PTR, acc=PTR,
                warm=0, plant_dt=DT, ref=dict(len=max(N, 1), start=0, rows=PTR), spheres=dict(n=2, cxyzr=PTR),
                grid=grid, pgrid=dict(grid), first_hit=PTR, rows=PTR, row_kind=0,
                row_stride=need_stride(N, 0) or 16)


def _grid_cases():
    out = []
    for field, v in (("occ", None), ("nx", 0), ("ny", 0), ("nz", -1), ("resolution", 0.0),
                     ("resolution", math.nan), ("cell_bytes", 2), ("cell_bytes", 4), ("cell_bytes", 8),
                     ("cell_bytes", -4), ("cell_bytes", 1)):
        for hit in (PTR, None):
            out.append((f"grid.{field}={v},hit={hit is not None}",
                        lambda a, f=field, v=v, h=hit: (a["grid"].__setitem__(f, v), a.__setitem__("first_hit", h))))
        out.append((f"pgrid.{field}={v}", lambda a, f=field, v=v: a["pgrid"].__setitem__(f, v)))
    return out


def _set(**kw):
    return lambda a: a.update(kw)


CASES = [("base", lambda a: None)]
CASES += [(f"{k}=None", _set(**{k: None})) for k in
          ("p0", "v0", "goal", "x", "status", "T", "acc", "rows", "grid", "pgrid", "first_hit", "ref", "spheres")]
CASES += [("no map check", _set(grid=None, first_hit=None)), ("B=-1", _set(B=-1)), ("ld=-1", _set(ld=-1)),
          ("warm=1", _set(warm=1)), ("warm=2", _set(warm=2)), ("plant_dt=0", _set(plant_dt=0.0)),
          ("plant_dt=nan", _set(plant_dt=math.nan)), ("plant_dt=2dt", _set(plant_dt=2 * DT)),
          ("dt=0", _set(dt=0.0, plant_dt=0.0)), ("dt=2dt", _set(dt=2 * DT, plant_dt=2 * DT)),
          ("rows misaligned", _set(rows=PTR + 8)), ("row_stride=1Mi", _set(row_stride=1 << 20)),
          ("no spheres, no map check", _set(spheres=None, grid=None, first_hit=None)),
          ("no ref, no spheres", _set(ref=None, spheres=None))]
CASES += [(f"ref.{k}={v}", lambda a, k=k, v=v: a["ref"].__setitem__(k, v(a) if callable(v) else v)) for k, v in
          (("rows", None), ("len", 0), ("len", lambda a: a["N"] + 1), ("len", lambda a: a["N"] - 1),
           ("start", -1), ("start", 1))]
CASES += [(f"spheres={n},{p}", lambda a, n=n, p=p: a.__setitem__("spheres", dict(n=n, cxyzr=p)))
          for n, p in ((0, None), (0, PTR), (-1, PTR), (3, None), (3, PTR))]
CASES += [(f"row_kind={k}", _set(row_kind=k)) for k in (-1, 1, 2, 3)]
CASES += [(f"row_kind={k}, no map check", _set(row_kind=k, first_hit=None)) for k in (1, 2)]
CASES += [("row_stride=need-16", lambda a: a.update(row_stride=a["row_stride"] - 16)),
          ("row_stride=need+8", lambda a: a.update(row_stride=a["row_stride"] + 8)),
          ("row_stride=need+16", lambda a: a.update(row_stride=a["row_stride"] + 16))]
CASES += _grid_cases()


# ---- the checks, restated -----------------------------------------------------------------------

def grid_rc(g):
    ok = (g is not None and g["occ"] is not None and g["nx"] > 0 and g["ny"] > 0 and g["nz"] > 0
          and g["resolution"] > 0.0 and g["cell_bytes"] in (0, 4, 8))
    return OK if ok else BAD


def spheres_rc(s):
    return BAD if s["n"] < 0 or (s["n"] > 0 and s["cxyzr"] is None) else OK


def params_rc(a, fam):
    m, N = a["mode"], a["N"]
    if N < 1 or N > 64:
        return UNS
    if fam == "track" and m not in (7, 8) or fam == "spheres" and m not in (5, 6):
        return BAD
    if fam == "plain" and not 0 <= m <= 4:
        return UNS
    if m in ROLLOUT and N > 16:
        return UNS
    return OK if a["dt"] > 0.0 else BAD


def lists_rc(a, fam):
    """The sphere list and the reference of a _spheres or _track entry."""
    s, r = a["spheres"], a["ref"]
    if fam == "track":
        if r is None or r["rows"] is None or r["len"] < 1 or r["start"] < 0:
            return BAD
        if (a["mode"] == 8) != (s is not None):
            return BAD
    return spheres_rc(s) if fam != "plain" and s is not None else OK


def expected(entry, a):
    fam = FAMILY.get(entry, "plain")
    m, N, B, ld = a["mode"], a["N"], a["B"], a["ld"]
    if entry == "solve_vjp_batch":
        if m not in (3, 6, 7, 8):
            return BAD
        track, sph = m in (7, 8), m in (6, 8)
        s, r = a["spheres"], a["ref"]
        if sph != (s is not None) or track != (r is not None) or (s is not None and spheres_rc(s)):
            return BAD
        if r is not None and (r["rows"] is None or r["len"] != N or r["start"] != 0):
            return BAD
        if a["x"] is None or a["status"] is None or a["p0"] is None or a["v0"] is None or \
                (not track and a["goal"] is None) or B < 0 or ld < B or N < 1:
            return BAD
        if N > 16:
            return UNS
        return OK if a["dt"] > 0.0 else BAD
    if fam == "spheres" and a["spheres"] is None:
        return BAD
    rc = params_rc(a, fam) or lists_rc(a, fam)
    if entry == "row_stride":
        return rc or (OK if 0 <= a["row_kind"] <= 2 else BAD)
    if rc:
        return rc
    if entry == "extract_batch":
        return BAD if B < 0 or ld < B or a["T"] is None or a["acc"] is None else OK
    if entry.startswith("solve_batch_host"):
        return BAD if B < 0 or a["p0"] is None or a["v0"] is None or a["goal"] is None else OK
    if B < 0 or ld < B or a["p0"] is None or a["v0"] is None or (a["goal"] is None and fam != "track"):
        return BAD
    if entry == "solve_batch_rows":
        if a["rows"] is None or not 0 <= a["row_kind"] <= 2:
            return BAD
        check = a["first_hit"] is not None
        if a["row_kind"] == 1 and check:
            return UNS
        need = need_stride(N, a["row_kind"])
        if need == 0:
            return UNS
        st = a["row_stride"]
        if st < need or st % 16 or st > SM_DOUBLES or a["rows"] % 128:
            return BAD
        return grid_rc(a["grid"]) if check or m in GRID_PEN else OK
    if entry.startswith("solve_batch"):
        hit = a["first_hit"] if entry != "solve_batch" else None
        return grid_rc(a["grid"] if entry != "solve_batch" else None) if hit is not None or m in GRID_PEN else OK
    # closed-loop steps
    if a["x"] is None or not a["plant_dt"] > 0.0:
        return BAD
    if entry == "closed_loop_step":
        if m in GRID_PEN:
            return UNS
        return BAD if m == 3 and a["warm"] == 2 else OK
    if fam == "track" and a["plant_dt"] != a["dt"]:
        return BAD
    if m in GRID_PEN and grid_rc(a["pgrid"]):
        return BAD
    if (a["grid"] is None) != (a["first_hit"] is None) or (a["grid"] is not None and grid_rc(a["grid"])):
        return BAD
    return BAD if m in ROLLOUT and a["warm"] == 2 else OK


# ---- the calls ----------------------------------------------------------------------------------

def _grid(g):
    if g is None:
        return None
    return C.byref(_cabi.Grid(nx=g["nx"], ny=g["ny"], nz=g["nz"], resolution=g["resolution"], occ=g["occ"],
                              cell_bytes=g["cell_bytes"]))


def _spheres(s):
    return None if s is None else C.byref(_cabi.Spheres(n=s["n"], cxyzr=s["cxyzr"], margin=0.1))


def _ref(r):
    return None if r is None else C.byref(_cabi.TrackRef(len=r["len"], start=r["start"], rows=r["rows"]))


def call(L, entry, a, p):
    p.gradient_mode, p.horizon, p.dt = a["mode"], a["N"], a["dt"]
    P, B, ld = C.byref(p), a["B"], a["ld"]
    p0, v0, goal, x, st = a["p0"], a["v0"], a["goal"], a["x"], a["status"]
    outs = [PTR] * 10                                          # x_out cost nit nfev status task acc att rates thrust
    grid, hit, sph, ref = _grid(a["grid"]), a["first_hit"], _spheres(a["spheres"]), _ref(a["ref"])
    f = getattr(L, "dart_se3mpc_" + entry)
    if entry == "solve_batch":
        return f(P, B, ld, p0, v0, goal, PTR, PTR, PTR, *outs, None)
    if entry == "solve_batch_map":
        return f(P, B, ld, p0, v0, goal, PTR, PTR, PTR, *outs, grid, 0.1, 0.5, hit, None)
    if entry == "solve_batch_spheres":
        return f(P, B, ld, p0, v0, goal, PTR, PTR, PTR, *outs, sph, grid, 0.1, 0.5, hit, None)
    if entry == "solve_batch_track":
        return f(P, B, ld, p0, v0, PTR, PTR, PTR, *outs, ref, sph, grid, 0.1, 0.5, hit, None)
    if entry == "solve_batch_rows":
        return f(P, B, ld, p0, v0, goal, PTR, PTR, PTR, a["rows"], a["row_stride"], a["row_kind"], grid, 0.1, 0.5,
                 int(hit is not None), None)
    if entry == "closed_loop_step":
        return f(P, B, ld, p0, v0, goal, PTR, x, a["warm"], PTR, PTR, PTR, PTR, a["plant_dt"], None)
    head = (P, B, ld, p0, v0) + ((goal,) if entry != "closed_loop_step_track" else ()) + \
        (PTR, x, a["warm"], PTR, PTR, PTR, PTR, a["plant_dt"])
    if entry == "closed_loop_step_map":
        return f(*head, _grid(a["pgrid"]), grid, 0.1, 0.5, 3, hit, None)
    if entry == "closed_loop_step_spheres":
        return f(*head, sph, grid, 0.1, 0.5, 3, hit, None)
    if entry == "closed_loop_step_track":
        return f(*head, ref, sph, grid, 0.1, 0.5, 3, hit, None)
    if entry == "solve_batch_host":
        return f(P, B, p0, v0, goal, PTR, PTR, *outs[:5], *outs[6:])
    if entry == "solve_batch_host_spheres":
        return f(P, B, p0, v0, goal, PTR, PTR, *outs[:5], *outs[6:], sph)
    if entry == "solve_vjp_batch":
        return f(P, B, ld, p0, v0, goal, PTR, x, ref, sph, PTR, PTR, PTR, PTR, PTR, PTR, PTR, st, None)
    if entry == "extract_batch":
        return f(P, B, ld, a["T"], a["acc"], PTR, PTR, PTR, 0, None)
    return f(P, a["row_kind"])                                 # row_stride


@pytest.mark.parametrize("entry", ENTRIES)
def test_every_solve_entry_refuses_what_its_checks_refuse(entry):
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    L = _cabi.lib()
    p = _cabi.Params()
    L.dart_se3mpc_default_params(C.byref(p))
    bad = []
    for mode in range(10):
        for N in (0, 1, 16, 17, 64, 65):
            for name, change in CASES:
                a = base(mode, N)
                change(a)
                got = call(L, entry, a, p)
                want = expected(entry, a)
                if entry == "row_stride":                      # 0 when refused, else the padded row
                    want = 0 if want else need_stride(N, a["row_kind"])
                if got != want:
                    bad.append(f"mode {mode} N {N} {name}: got {got}, want {want}")
    assert not bad, f"{len(bad)} mismatches, first: " + "; ".join(bad[:8])
