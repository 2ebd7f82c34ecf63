"""The bundle-adjustment problems of tests/test_zz_ref_backend_dropin.py, without the reference tree.

tests/golden/ref_backend.npz holds every problem the reference's own Backend::BuildProblem + adapt::Solve (modes 0 and 1),
imu::FullBA (2), Initializer::Initialize (3) and Environment::Optimize (4) handed to the solver through the product shim, as
the C ABI received it (recorded by oracle/ref_record.cpp, written by tests/golden/make_ref_golden.py), with the oracle's solve
of each and, for modes 0 and 1, the cost the reference's own functors assign to the problem.  Each problem is replayed here
through the same C ABI -- the oracle on the CPU, liblvio_b200.so on the device -- against the tolerances of the drop-in tests."""
import ctypes as C
import os

import numpy as np
import pytest

from lvio_fusion_b200 import _capi, backend

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_backend.npz"))
MODES = (0, 1, 2, 3, 4)


def _solves(mode):
    n = int(G["m%d_n_solves" % mode])
    assert n >= 1
    return [{k[len("m%d_s%d_" % (mode, j)):]: G[k] for k in G.files if k.startswith("m%d_s%d_" % (mode, j))} for j in range(n)]


def _replay(ctx, g):
    p = backend.Problem(ctx)
    try:
        p.set_cameras(g["cameras"])
        p.set_poses(g["poses"], g["poses_const"])
        p.set_vec3(g["vec3"], g["vec3_const"])
        p.set_inv_depths(g["rho"], g["rho_const"])
        for k in range(6):
            if "f%d_consts" % k in g:
                p.add_factors(k, g["f%d_consts" % k], g["f%d_idx" % k])
            p.set_loss(k, g["loss"][k])
        p.finalize()
        types = dict(_capi.SolveOptions._fields_)
        opt = backend.default_options(ctx.api, **{f: (int(v) if types[f] is C.c_int else float(v)) for (f, _), v in zip(_capi.SolveOptions._fields_, g["options"])})
        s = p.solve(opt)
        return s, p.poses(), p.vec3(), p.inv_depths()
    finally:
        p.close()


def _quat_to_R(q):
    x, y, z, w = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _relative_motion_gap(a, b):
    """RMS translation and rotation-angle gap between the relative motions T_i^-1 T_(i+1) of two pose sets (gauge-free)."""
    dt, dr = [], []
    for i in range(len(a) - 1):
        rel = []
        for P in (a, b):
            Ri, Rj = _quat_to_R(P[i, :4]), _quat_to_R(P[i + 1, :4])
            rel.append((Ri.T @ Rj, Ri.T @ (P[i + 1, 4:] - P[i, 4:])))
        dt.append(np.linalg.norm(rel[0][1] - rel[1][1]))
        dr.append(np.arccos(np.clip((np.trace(rel[0][0].T @ rel[1][0]) - 1) / 2, -1.0, 1.0)))
    return float(np.sqrt(np.mean(np.square(dt)))), float(np.sqrt(np.mean(np.square(dr))))


def _check(ctx, mode, init_tol):
    for g in _solves(mode):
        s, P, V, R = _replay(ctx, g)
        rc, init0, final0 = g["summary"][:3]
        assert rc == 0 and s.termination_type == int(g["summary"][5]) == 0
        assert abs(s.initial_cost - init0) <= init_tol * init0
        assert s.final_cost < s.initial_cost
        if mode < 2:
            # Backend::BuildProblem's problem: the cost the reference's functors assign to it, and adapt::Solve does its job on it
            ref_cost = float(G["m%d_reference_initial_cost" % mode])
            assert abs(s.initial_cost - ref_cost) <= init_tol * ref_cost
            assert s.final_cost < 0.25 * s.initial_cost
            assert abs(s.final_cost - final0) <= 1e-5 * final0
            got, want = np.concatenate([P.ravel(), V.ravel(), R]), np.concatenate([g["out_poses"].ravel(), g["out_vec3"].ravel(), g["out_rho"]])
            assert np.max(np.abs(got - want)) < 1e-4
        elif mode == 4:
            # one keyframe re-solved against constant blocks: its translation within 1e-7 (bounds the gap in moved_t)
            free = np.flatnonzero(g["poses_const"] == 0)
            assert len(free) == 1 and np.all(P[g["poses_const"] == 1] == g["poses"][g["poses_const"] == 1])
            assert np.max(np.abs(P[free, 4:] - g["out_poses"][free, 4:])) < 1e-7
            assert abs(s.final_cost - final0) <= 1e-6 * final0
        else:
            # FullBA problems have a gauge and are stiff (prior whitening ~1e9): compare the relative motion and the shared
            # biases.  The motion gap bounds the gap between the two runs' relative-motion errors (5 % of the oracle's error).
            rel = G["m%d_rel" % mode]
            gap_t, gap_r = _relative_motion_gap(P, g["out_poses"])
            assert gap_t < 0.05 * rel[2] + 1e-5 and gap_r < 0.05 * rel[3] + 1e-6, (gap_t, gap_r)
            bias = g["f3_idx"][0, 2:4]                    # ImuInitError: idx = pose_i v_i ba bg pose_j v_j -1 -1, one shared ba / bg
            assert np.all(g["f3_idx"][:, 2:4] == bias)
            assert np.max(np.abs(V[bias] - g["out_vec3"][bias])) < (5e-5 if mode == 2 else 2e-3)


@pytest.mark.parametrize("mode", MODES)
def test_oracle_solves_the_reference_backend_problems(orc_ctx, mode):
    _check(orc_ctx, mode, 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_cuda_solves_the_reference_backend_problems(lvb_ctx, mode):
    _check(lvb_ctx, mode, 1e-9)
