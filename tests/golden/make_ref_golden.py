"""Generate tests/golden/ref_factors.npz by running the REFERENCE's own factor functors.

`make -C oracle ref` compiles /root/reference/src/lvio_fusion/include/lvio_fusion/ceres/{visual,lidar,pose}_error.hpp (in
place, never copied) against the stand-in third-party headers in oracle/ref_compat and the oracle's dual numbers; this script
feeds it seeded KITTI-shaped inputs and stores inputs + residuals + Jacobians.  The oracle (tests/test_ref_golden.py, CPU)
and the CUDA path (same file, -m gpu) must reproduce them.  Only runs where /root/reference is mounted.

    python tests/golden/make_ref_golden.py
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lvio_fusion_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
N = 24
N_IMU = 12


def _unit_pose(rng, P, sigma_q=0.01, sigma_t=0.05, scale=1.0):
    q = P[:4] + rng.normal(0, sigma_q, 4)
    return np.concatenate([q / np.linalg.norm(q) * scale, P[4:] + rng.normal(0, sigma_t, 3)])


def build_cases(seed=synth.SEED):
    rng = np.random.default_rng(seed)
    d = synth.make_ba_problem(6, 120, with_imu=False, seed=seed)
    P = d["poses"]
    c0, i0 = d["factors"][0]; c1, i1 = d["factors"][1]; c2, i2 = d["factors"][2]
    cases = {"cameras": np.asarray(d["cameras"], dtype=np.float64)}
    # a1: consts (first_ob, ob, w), params rho, T1, T2 -- one pose pair with a non-unit quaternion (QuaternionRotatePoint normalises)
    sel = rng.choice(len(c0), N, replace=False)
    T1 = np.stack([_unit_pose(rng, P[i0[s, 1]], scale=1.0 + 0.01 * (k % 3)) for k, s in enumerate(sel)])
    T2 = np.stack([_unit_pose(rng, P[i0[s, 2]]) for s in sel])
    cases["tf_c"] = c0[sel]; cases["tf_x"] = np.concatenate([d["rho"][i0[sel, 0]][:, None], T1, T2], axis=1)
    sel = rng.choice(len(c1), N, replace=False)
    cases["po_c"] = c1[sel]; cases["po_x"] = np.stack([_unit_pose(rng, P[i1[s, 0]]) for s in sel])
    sel = rng.choice(len(c2), N, replace=False)
    cases["tc_c"] = c2[sel]; cases["tc_x"] = d["rho"][i2[sel, 0]][:, None] * rng.uniform(0.9, 1.1, (N, 1))
    # a5: mode, p, pa, pb, pc, Twc1, rpyxyz, w
    lid = []
    for k in range(N):
        pa = rng.normal(0, 8, 3); pb = pa + rng.normal(0, 0.4, 3); pc = pa + rng.normal(0, 0.4, 3)
        p = rng.normal(0, 8, 3)
        T = _unit_pose(rng, P[k % len(P)], sigma_q=0.05, sigma_t=1.0)
        e = np.concatenate([rng.normal(0, 0.05, 3), rng.normal(0, 0.3, 3)])
        lid.append(np.concatenate([[k % 2], p, pa, pb, pc, T, e, [rng.uniform(0.01, 1.0)]]))
    cases["lidar"] = np.asarray(lid)
    # a6
    pg, pe, pr = [], [], []
    for k in range(N):
        a, b = _unit_pose(rng, P[k % 5]), _unit_pose(rng, P[k % 5 + 1])
        x1, x2 = _unit_pose(rng, P[k % 5], 0.02, 0.1, 1.0 + 0.005 * (k % 2)), _unit_pose(rng, P[k % 5 + 1], 0.02, 0.1)
        pg.append(np.concatenate([a, b, [rng.uniform(1, 100), rng.uniform(0, 2)], x1, x2]))
        pe.append(np.concatenate([a, [rng.uniform(1, 100), rng.uniform(0, 2)], x1]))
        pr.append(np.concatenate([[k % 2], rng.normal(0, 0.3, 6), [rng.uniform(1, 100)], rng.normal(0, 0.3, 3)]))
    cases["pg"] = np.asarray(pg); cases["pe"] = np.asarray(pe); cases["pr"] = np.asarray(pr)
    # a4: noise4, then per case: ba bg acc0 gyr0 n_samples samples[n][7] | pose_i v_i ba_i bg_i pose_j v_j ba_j bg_j
    cases["imu_noise"] = np.array(synth.IMU_NOISE, dtype=np.float64)
    imu = []
    for k in range(N_IMU):
        ns = 6 + (k % 7)
        ba, bg = rng.normal(0, 0.05, 3), rng.normal(0, 0.01, 3)
        acc = rng.normal(0, 0.8, (ns + 1, 3)) + [0.3, 0.1, 9.81]; gyr = rng.normal(0, 0.15, (ns + 1, 3))
        dt = rng.uniform(0.008, 0.012, ns)
        T = dt.sum()
        pose_i = _unit_pose(rng, P[k % len(P)], 0.05, 0.5)
        v_i = np.array([9.5, 0.3, -0.1]) + rng.normal(0, 0.3, 3)
        pose_j = _unit_pose(rng, np.concatenate([pose_i[:4], pose_i[4:] + v_i * T]), 0.02, 0.03)
        v_j = v_i + rng.normal(0, 0.2, 3)
        x = np.concatenate([pose_i, v_i, ba + rng.normal(0, 0.01, 3), bg + rng.normal(0, 0.002, 3), pose_j, v_j, ba + rng.normal(0, 0.01, 3), bg + rng.normal(0, 0.002, 3)])
        imu.append({"ba": ba, "bg": bg, "acc0": acc[0], "gyr0": gyr[0], "samples": np.concatenate([dt[:, None], acc[1:], gyr[1:]], axis=1), "x": x})
    cases["imu_first"] = np.concatenate([[0], np.cumsum([len(c["samples"]) for c in imu])]).astype(np.int32)
    cases["imu_samples"] = np.concatenate([c["samples"] for c in imu])
    for key in ("ba", "bg", "acc0", "gyr0", "x"):
        cases["imu_" + key] = np.stack([c[key] for c in imu])
    return cases


def run_reference(cases):
    subprocess.check_call(["make", "-s", "-j4", "-C", os.path.join(ROOT, "oracle"), "ref"])
    flat = [cases["cameras"], np.array([N] * 7 + [N_IMU], dtype=np.float64)]
    flat += [np.concatenate([cases["tf_c"], cases["tf_x"]], axis=1).ravel(), np.concatenate([cases["po_c"], cases["po_x"]], axis=1).ravel(),
             np.concatenate([cases["tc_c"], cases["tc_x"]], axis=1).ravel(), cases["lidar"].ravel(), cases["pg"].ravel(), cases["pe"].ravel(), cases["pr"].ravel(), cases["imu_noise"]]
    for k in range(N_IMU):
        lo, hi = cases["imu_first"][k], cases["imu_first"][k + 1]
        flat += [cases["imu_ba"][k], cases["imu_bg"][k], cases["imu_acc0"][k], cases["imu_gyr0"][k], np.array([hi - lo], dtype=np.float64), cases["imu_samples"][lo:hi].ravel(), cases["imu_x"][k]]
    with tempfile.TemporaryDirectory() as td:
        np.concatenate(flat).astype(np.float64).tofile(os.path.join(td, "cases.bin"))
        subprocess.check_call([os.path.join(ROOT, "oracle", "_ref", "ref_factors"), os.path.join(td, "cases.bin"), os.path.join(td, "out.bin")])
        o = np.fromfile(os.path.join(td, "out.bin"), dtype=np.float64)
    out, pos = {}, 0
    for name, R, C in (("tf", 2, 15), ("po", 2, 7), ("tc", 2, 1), ("lidar", 1, 3), ("pg", 6, 14), ("pe", 6, 7), ("pr", 3, 3)):
        blk = o[pos:pos + N * (R + R * C)].reshape(N, R + R * C); pos += N * (R + R * C)
        out[name + "_r"] = blk[:, :R].copy(); out[name + "_J"] = blk[:, R:].reshape(N, R, C).copy()
    per = 17 + 225 + 225 + 15 + 105 + 45 * 3 + 105 + 45 * 3 + 2 * (15 + 105 + 45 * 3 + 105 + 45)
    blk = o[pos:pos + N_IMU * per].reshape(N_IMU, per); pos += N_IMU * per
    out["imu_record"] = blk[:, :467].copy()                      # LVB_IMU layout without the two prior slots
    out["imu_r"] = blk[:, 467:482].copy()
    sizes, q, Js = [7, 3, 3, 3, 7, 3, 3, 3], 482, []
    for w in sizes:
        Js.append(blk[:, q:q + 15 * w].reshape(N_IMU, 15, w)); q += 15 * w
    out["imu_J"] = np.concatenate(Js, axis=2)                      # [n, 15, 32] in the block order of imu_error.hpp:12
    out["imuinit_r"] = blk[:, q:q + 15].copy(); q += 15
    Js = []
    for w in [7, 3, 3, 3, 7, 3]:
        Js.append(blk[:, q:q + 15 * w].reshape(N_IMU, 15, w)); q += 15 * w
    out["imuinit_J"] = np.concatenate(Js, axis=2)                  # [n, 15, 26], ImuInitError with priors 1e8 / 1e8
    out["imuinit2_r"] = blk[:, q:q + 15].copy(); q += 15
    Js = []
    for w in [7, 3, 3, 3, 7, 3]:
        Js.append(blk[:, q:q + 15 * w].reshape(N_IMU, 15, w)); q += 15 * w
    out["imuinit2_J"] = np.concatenate(Js, axis=2)                 # the reference's real priors 1e4 / 1e2 (initializer.cpp:62): indefinite cov^-1
    assert q == per
    assert pos == len(o)
    return out


LIDAR_CFG = dict(num_scans=64, horizon_scan=450, ang_res_y=0.427, ang_bottom=24.9, ground_rows=60, min_range=5.0, max_range=30.0)


def run_reference_lidar(scan):
    """ImageProjection::Process (src/projection.cpp) + filter_points_by_distance (utility.h) of the reference on a raw sweep."""
    c = LIDAR_CFG
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "in.bin"), "wb") as f:
            np.array([c["num_scans"], c["horizon_scan"], c["ang_res_y"], c["ang_bottom"], c["ground_rows"], c["min_range"], c["max_range"]], dtype=np.float64).tofile(f)
            np.array([len(scan)], dtype=np.int32).tofile(f)
            np.ascontiguousarray(scan[:, :3], dtype=np.float32).tofile(f)
        subprocess.check_call([os.path.join(ROOT, "oracle", "_ref", "ref_lidar"), os.path.join(td, "in.bin"), os.path.join(td, "out.bin")])
        raw = open(os.path.join(td, "out.bin"), "rb").read()
    m = int(np.frombuffer(raw[:4], dtype=np.int32)[0]); off = 4
    R = c["num_scans"]
    out = {}
    out["points"] = np.frombuffer(raw[off:off + 16 * m], dtype=np.float32).reshape(m, 4).copy(); off += 16 * m
    out["range"] = np.frombuffer(raw[off:off + 4 * m], dtype=np.float32).copy(); off += 4 * m
    out["ground"] = np.frombuffer(raw[off:off + m], dtype=np.uint8).copy(); off += m
    out["col"] = np.frombuffer(raw[off:off + 4 * m], dtype=np.int32).copy(); off += 4 * m
    out["start_ring"] = np.frombuffer(raw[off:off + 4 * R], dtype=np.int32).copy(); off += 4 * R
    out["end_ring"] = np.frombuffer(raw[off:off + 4 * R], dtype=np.int32).copy(); off += 4 * R
    out["orientation"] = np.frombuffer(raw[off:off + 12], dtype=np.float32).copy(); off += 12
    assert off == len(raw)
    return out


ASSOC_EXT = [0.01, -0.02, 0.005, 1.0, 0.27, 0.0, 0.08]
W_VISUAL, N_FEATURES_LEFT = 71.8856, 120


def _assoc_cfg(horizon, ext):
    return np.array([64, horizon, 0.427, 24.9, 60, 0.1036, 5, 30, 0.2, 0], dtype=np.float64).tobytes() + np.asarray(ext, dtype=np.float64).tobytes()


def _read_cloud(raw, off):
    m = int(np.frombuffer(raw[off:off + 4], dtype=np.int32)[0]); off += 4
    return np.frombuffer(raw[off:off + 16 * m], dtype=np.float32).reshape(m, 4).copy(), off + 16 * m


def run_reference_extract(scan, horizon):
    """FeatureAssociation::Preprocess .. ExtractFeatures (association.cpp:88-268) of the reference on a raw sweep."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_assoc")
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "in.bin"), "wb") as f:
            f.write(_assoc_cfg(horizon, ASSOC_EXT)); np.array([len(scan)], dtype=np.int32).tofile(f); np.ascontiguousarray(scan[:, :3], dtype=np.float32).tofile(f)
        subprocess.check_call([exe, "extract", os.path.join(td, "in.bin"), os.path.join(td, "out.bin")])
        raw = open(os.path.join(td, "out.bin"), "rb").read()
    seg, off = _read_cloud(raw, 0)
    curv = np.frombuffer(raw[off:off + 4 * len(seg)], dtype=np.float32).copy(); off += 4 * len(seg)
    ground, off = _read_cloud(raw, off); surf, off = _read_cloud(raw, off)
    assert off == len(raw)
    return {"seg": seg, "curvature": curv, "ground": ground, "surf": surf}


def run_reference_scan2map(sc, mode, e0):
    """FeatureAssociation::ScanToMapWithGround / ScanToMapWithSegmented (association.cpp:270-384) of the reference."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_assoc")
    scan = np.ascontiguousarray(sc["scan"][:, :4], dtype=np.float32); mp = np.ascontiguousarray(sc["map"][:, :4], dtype=np.float32)
    w = [W_VISUAL, sc["weight"] if mode == 0 else 1.0, sc["weight"] if mode == 1 else 0.01]
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "in.bin"), "wb") as f:
            f.write(_assoc_cfg(1800, [0, 0, 0, 1, 0, 0, 0]))
            np.array([mode], dtype=np.int32).tofile(f)
            for a in (sc["frame_pose"], sc["map_pose"], e0, w):
                np.asarray(a, dtype=np.float64).tofile(f)
            np.array([N_FEATURES_LEFT, 0], dtype=np.int32).tofile(f)
            np.array([len(scan)], dtype=np.int32).tofile(f); scan.tofile(f); np.array([len(mp)], dtype=np.int32).tofile(f); mp.tofile(f)
        subprocess.check_call([exe, "scan2map", os.path.join(td, "in.bin"), os.path.join(td, "out.bin")])
        o = np.fromfile(os.path.join(td, "out.bin"), dtype=np.float64)
    return o[:4].copy(), o[4:].reshape(len(scan), 5).copy()


def assoc_case(kind):
    """Scan / map feature clouds with a share of scan points pushed away from every map surface, so that the gate rejects."""
    sc = synth.make_icp_problem(1200, 9000, seed=synth.SEED + (7 if kind == "ground" else 8), kind=kind)
    rng = np.random.default_rng(99)
    scan = np.array(sc["scan"], dtype=np.float32, copy=True)
    far = rng.choice(len(scan), len(scan) // 6, replace=False)
    scan[far, :3] += rng.normal(0, 1.5, (len(far), 3)).astype(np.float32)
    sc = dict(sc); sc["scan"] = scan
    return sc


BACKEND_MODES = (0, 1, 2, 3, 4)       # tests/cpp/ref_backend_dropin.cpp: window + IMU, visual only, FullBA, Initializer, Environment


def _parse_ba_record(raw):
    """The log of oracle/ref_record.cpp -> one dict per solve: the problem as the C ABI received it, the options (the fields
    of lvb_solve_options in order), and the oracle's summary (rc, initial cost, final cost, iterations, successful steps,
    termination) and solved blocks."""
    from lvio_fusion_b200.backend import CONST_STRIDE, IDX_STRIDE
    off, solves, cur = 0, [], None

    def take(dtype, n):
        nonlocal off
        a = np.frombuffer(raw, dtype=dtype, count=n, offset=off).copy()
        off += a.nbytes
        return a
    while off < len(raw):
        tag = int(take(np.int32, 1)[0])
        if tag == 1:
            cur = {"loss": np.zeros(6)}
        elif tag == 2:
            cur["cameras"] = take(np.float64, 22)
        elif tag in (3, 4, 5):
            name, w = {3: ("poses", 7), 4: ("vec3", 3), 5: ("rho", 1)}[tag]
            n = int(take(np.int32, 1)[0])
            cur[name] = take(np.float64, n * w).reshape(n, w) if w > 1 else take(np.float64, n)
            cur[name + "_const"] = take(np.uint8, n) if take(np.int32, 1)[0] else np.zeros(n, np.uint8)
        elif tag == 6:
            kind, n = (int(v) for v in take(np.int32, 2))
            cur["f%d_consts" % kind] = take(np.float64, n * CONST_STRIDE[kind]).reshape(n, CONST_STRIDE[kind])
            cur["f%d_idx" % kind] = take(np.int32, n * IDX_STRIDE[kind]).reshape(n, IDX_STRIDE[kind])
        elif tag == 7:
            kind = int(take(np.int32, 1)[0])
            cur["loss"][kind] = take(np.float64, 1)[0]
        elif tag == 8:
            cur["options"], cur["summary"] = take(np.float64, 10), take(np.float64, 6)
            for name, w in (("poses", 7), ("vec3", 3), ("rho", 1)):
                cur["out_" + name] = take(np.float64, len(cur[name]) * w).reshape(cur[name].shape)
            solves.append(cur)
        else:
            raise ValueError("bad record tag %d" % tag)
    return solves


def _harness_values(stdout):
    """`tag key value key value ...` lines of the drop-in harness -> {"tag.key": value} for the numeric ones."""
    rec = {}
    for line in stdout.splitlines():
        t = line.split()
        for k, v in zip(t[1::2], t[2::2]):
            try:
                rec[t[0] + "." + k] = float(v)
            except ValueError:
                pass
    return rec


def run_reference_backend():
    """Every bundle-adjustment problem the reference's Backend::BuildProblem / adapt::Solve, imu::FullBA, Initializer and
    Environment::Optimize (tests/cpp/ref_backend_dropin.cpp, compiled in place) hand to the solver through the product shim, as
    the oracle received and solved it; with the cost the reference's own functors assign to the problems of modes 0 and 1
    (ref_backend_truth) and the harness' error summary before and after (ref_backend_orc)."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    out = {}
    for mode in BACKEND_MODES:
        with tempfile.TemporaryDirectory() as td:
            log = os.path.join(td, "ba.log")
            env = dict(os.environ, LVB_RECORD=log, LD_PRELOAD=os.path.join(ref, "ref_record.so"))
            orc = _harness_values(subprocess.run([os.path.join(ref, "ref_backend_orc"), str(mode)], env=env, check=True, capture_output=True, text=True).stdout)
            with open(log, "rb") as f:
                solves = _parse_ba_record(f.read())
        out["m%d_n_solves" % mode] = np.array(len(solves))
        for j, s in enumerate(solves):
            out.update({"m%d_s%d_%s" % (mode, j, k): v for k, v in s.items()})
        out["m%d_rel" % mode] = np.array([orc.get(k, np.nan) for k in ("before.rel_t", "before.rel_r", "after.rel_t", "after.rel_r")])
        if mode < 2:
            truth = _harness_values(subprocess.run([os.path.join(ref, "ref_backend_truth"), str(mode)], check=True, capture_output=True, text=True).stdout)
            out["m%d_reference_initial_cost" % mode] = np.array(truth["reference.initial_cost"])
    return out


def main():
    if not os.path.isdir("/root/reference"):
        raise SystemExit("the reference tree is not mounted here; the committed fixture stays as it is")
    cases = build_cases()
    out = run_reference(cases)
    np.savez_compressed(os.path.join(HERE, "ref_factors.npz"), **cases, **out)
    print("reference golden written:", {k: v.shape for k, v in out.items()})
    scan = synth.make_lidar_scan(seed=synth.SEED + 5, horizon_scan=LIDAR_CFG["horizon_scan"], n_boxes=10)
    lid = run_reference_lidar(scan)
    np.savez_compressed(os.path.join(HERE, "ref_lidar.npz"), scan=scan[:, :3].astype(np.float32), **lid)
    print("reference lidar golden written:", len(lid["points"]), "segmented points of", len(scan))
    ext = run_reference_extract(scan, LIDAR_CFG["horizon_scan"])
    out = {"scan": scan[:, :3].astype(np.float32), "ext_seg": ext["seg"], "ext_curvature": ext["curvature"], "ext_ground": ext["ground"], "ext_surf": ext["surf"]}
    for kind, mode in (("ground", 0), ("surf", 1)):
        sc = assoc_case(kind)
        e0 = synth.relative_rpyxyz(sc["map_pose"], sc["frame_pose"])
        head, tab = run_reference_scan2map(sc, mode, e0)
        out.update({kind + "_head": head, kind + "_table": tab, kind + "_e0": np.asarray(e0)})
        print("reference scan-to-map (%s): %d blocks of %d scan points, prior weight %.3f, huber %.2f" % (kind, int(head[0]), len(tab), head[2], head[3]))
    np.savez_compressed(os.path.join(HERE, "ref_assoc.npz"), **out)
    ba = run_reference_backend()
    np.savez_compressed(os.path.join(HERE, "ref_backend.npz"), **ba)
    print("reference backend problems written:", {m: int(ba["m%d_n_solves" % m]) for m in BACKEND_MODES})


if __name__ == "__main__":
    main()
