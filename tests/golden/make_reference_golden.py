"""Known-answer vectors from the reference's own arithmetic (tests/golden/reference_kat.npz).

oracle/_ref/libvicalib_ref.so is the reference's header-only code (types.h, vicalibrator-utils.h,
interpolation-buffer.h, ceres-cost-functions.h, local-param-se3.h) compiled unmodified against the stand-ins in
oracle/ref_shim (recipe: oracle/Makefile, `make -C oracle _ref REF=<reference checkout>`).  This script evaluates it
on the inputs tests/test_cpu_oracle_ref.py uses and stores inputs and outputs, so that the oracle is pinned to the
reference text wherever the suite runs, with or without a reference checkout.

    make -C oracle _ref REF=<reference checkout> && python tests/golden/make_reference_golden.py
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from vicalib_b200 import synth  # noqa: E402

SO = os.path.join(ROOT, "oracle", "_ref", "libvicalib_ref.so")
MODELS = ["fov", "poly2", "poly3", "kb4", "linear"]


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _imu(p):
    return C.c_int(len(p.imu_t)), _p(_c(p.imu_t)), _p(_c(p.imu_w)), _p(_c(p.imu_a))


def _problem(**kw):
    args = dict(models=("poly3",), n_frames=12, grid=(14, 10), inertial=True, seed=77, ts_truth=0.003)
    args.update(kw)
    return synth.make_problem(**args)


def _imu_inputs(prefix, p):
    out = {f"{prefix}_{k}": _c(getattr(p, k)) for k in ("imu_t", "imu_w", "imu_a", "ftime", "T_wp", "v_w", "g", "b", "sf")}
    out[f"{prefix}_ts"] = np.float64(p.ts)
    return out


def get_range(ref):
    """InterpolationBufferT::GetRange on interval ends before / at / after the samples, several time offsets"""
    p = _problem()
    t0s = [p.ftime[0], p.ftime[3], p.imu_t[0] - 0.01, p.imu_t[0], p.imu_t[5], p.imu_t[-1] - 0.004, p.imu_t[-1] + 0.01]
    q, n, rows = [], [], []
    for ts in (-0.0049, 0.0, 0.00251, 0.0074):
        for t0 in t0s:
            for dt in (1e-4, 1.0 / 30, 0.2):
                out = np.zeros((256, 7))
                m = ref.ref_get_range(*_imu(p), C.c_double(t0), C.c_double(t0 + dt), C.c_double(ts), _p(out), 256)
                q.append((t0, t0 + dt, ts))
                n.append(m)
                rows.append(out)
    w = max(n)
    rows = np.stack([np.where(np.arange(256)[:, None] < m, r, np.nan) for r, m in zip(rows, n)])[:, :w]
    return dict(_imu_inputs("range", p), range_query=np.array(q), range_n=np.array(n, dtype=np.int32), range_rows=rows)


def imu_eval(ref):
    """SwitchedFullImuCostFunction with ceres::Jet<double, 35> + LocalParamSe3: residual, 9 x 33 tangent Jacobian"""
    p = _problem()
    rng = np.random.default_rng(3)
    p.b = 1e-2 * rng.standard_normal(6)
    p.sf = 1 + 1e-2 * rng.standard_normal(6)
    p.ts = 0.0021
    p.v_w = p.truth["v_w"] + 1e-2 * rng.standard_normal(p.v_w.shape)
    W = rng.standard_normal((p.n_frames - 1, 9, 9)) + 30 * np.eye(9)
    W = 0.5 * (W + W.transpose(0, 2, 1))
    r_all, J_all = np.zeros((2, p.n_frames - 1, 9)), np.zeros((2, p.n_frames - 1, 9, 33))
    for rot_only in (0, 1):
        for k in range(p.n_frames - 1):
            r, J = np.zeros(9), np.zeros((9, 33))
            rc = ref.ref_imu_eval(*_imu(p), C.c_double(p.ftime[k]), C.c_double(p.ftime[k + 1]), _p(_c(W[k])), C.c_int(rot_only),
                                  _p(_c(p.T_wp[k + 1])), _p(_c(p.T_wp[k])), _p(_c(p.v_w[k + 1])), _p(_c(p.v_w[k])),
                                  _p(_c(p.g)), _p(_c(p.b)), _p(_c(p.sf)), C.c_double(p.ts), _p(r), _p(J))
            assert rc == 0
            r_all[rot_only, k], J_all[rot_only, k] = r, J
    return dict(_imu_inputs("imu", p), imu_W=W, imu_r=r_all, imu_J=J_all)


def update_weights(ref):
    """the loop body of ViCalibrator::UpdateImuWeights: the 9 x 9 weight_sqrt_ of every interval"""
    p = _problem(n_frames=16)
    rng = np.random.default_rng(5)
    p.b = 1e-2 * rng.standard_normal(6)
    p.sf = 1 + 1e-2 * rng.standard_normal(6)
    p.ts = 0.0013
    p.v_w = p.truth["v_w"].copy()
    Ws = np.zeros((p.n_frames - 1, 9, 9))
    for k in range(p.n_frames - 1):
        m = C.c_double()
        rc = ref.ref_update_weight(*_imu(p), C.c_double(p.ftime[k]), C.c_double(p.ftime[k + 1]), _p(_c(p.T_wp[k])),
                                   _p(_c(p.v_w[k])), _p(_c(p.T_wp[k + 1])), _p(_c(p.v_w[k + 1])), _p(_c(p.g)), _p(_c(p.b)),
                                   _p(_c(p.sf)), C.c_double(p.ts), C.c_double(synth.GYRO_SIGMA), C.c_double(synth.ACCEL_SIGMA),
                                   _p(Ws[k]), C.byref(m))
        assert rc == 1
    return dict(_imu_inputs("weights", p), weights_W=Ws, weights_sigma=np.array([synth.GYRO_SIGMA, synth.ACCEL_SIGMA]))


def local_parameterisations(ref):
    """LocalParamSe3 / LocalParamSo3 Plus at three step scales, ComputeJacobian, and Plus at +-h along each tangent axis"""
    rng = np.random.default_rng(9)
    h = 1e-6
    X, D, P7, P4, J, A, B = [], [], [], [], [], [], []
    for _ in range(50):
        q = rng.standard_normal(4)
        q /= np.linalg.norm(q)
        x = np.concatenate([q, rng.standard_normal(3)])
        ds, p7, p4 = [], [], []
        for scale in (1e-12, 1e-3, 0.7):
            d = scale * rng.standard_normal(6)
            out, out4 = np.zeros(7), np.zeros(4)
            ref.ref_se3_plus(_p(x), _p(d), _p(out))
            ref.ref_so3_plus(_p(_c(q)), _p(_c(d[3:])), _p(out4))
            ds.append(d)
            p7.append(out)
            p4.append(out4)
        Jx = np.zeros((7, 6))
        ref.ref_se3_jacobian(_p(x), _p(Jx))
        a, b = np.zeros((6, 7)), np.zeros((6, 7))
        for c in range(6):
            e = np.zeros(6)
            e[c] = h
            ref.ref_se3_plus(_p(x), _p(e), _p(a[c]))
            ref.ref_se3_plus(_p(x), _p(-e), _p(b[c]))
        X.append(x)
        D.append(ds)
        P7.append(p7)
        P4.append(p4)
        J.append(Jx)
        A.append(a)
        B.append(b)
    return dict(lp_x=np.array(X), lp_d=np.array(D), lp_se3_plus=np.array(P7), lp_so3_plus=np.array(P4), lp_J=np.array(J),
                lp_h=np.array(h), lp_plus_fwd=np.array(A), lp_plus_bwd=np.array(B))


def reprojection(ref):
    """ImuReprojectionCostFunctor with Jet<double, 22>: residual and 2 x 22 tangent Jacobian of every 17th observation of
    camera 0, for every camera model (camera 1 is poly3)"""
    out = {}
    for model in MODELS:
        p = synth.make_problem(models=(model, "poly3"), n_frames=4, seed=12, inertial=True)
        sel = np.where(p.obs_cam == 0)[0][::17]
        rs, Js = np.zeros((len(sel), 2)), np.zeros((len(sel), 2, 22))
        for j, i in enumerate(sel):
            f = p.obs_frame[i]
            rc = ref.ref_reproj(C.c_int(int(p.models[0])), _p(_c(p.T_wp[f])), _p(_c(p.q_ck[0])), _p(_c(p.p_ck[0])),
                                _p(_c(p.intr[0])), _p(_c(p.p_w[i])), _p(_c(p.p_c[i])), _p(rs[j]), _p(Js[j]))
            assert rc == 0
        pre = f"reproj_{model}"
        out.update({f"{pre}_T_wp": _c(p.T_wp), f"{pre}_intr": _c(p.intr), f"{pre}_q_ck": _c(p.q_ck), f"{pre}_p_ck": _c(p.p_ck),
                    f"{pre}_obs_frame": p.obs_frame[sel].astype(np.int32), f"{pre}_p_w": _c(p.p_w[sel]),
                    f"{pre}_p_c": _c(p.p_c[sel]), f"{pre}_r": rs, f"{pre}_J": Js})
    return out


def main():
    if not os.path.exists(SO):
        sys.exit(f"{SO} is missing: build it with `make -C oracle _ref REF=<reference checkout>`")
    ref = C.CDLL(SO)
    for f in ("ref_get_range", "ref_imu_eval", "ref_update_weight", "ref_integrate", "ref_reproj"):
        getattr(ref, f).restype = C.c_int
    out = {}
    for part in (get_range, imu_eval, update_weights, local_parameterisations, reprojection):
        out.update(part(ref))
    path = os.path.join(HERE, "reference_kat.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {len(out)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
