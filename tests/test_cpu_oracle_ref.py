"""CPU: the oracle restatement against the reference's OWN arithmetic — types.h, vicalibrator-utils.h,
interpolation-buffer.h, ceres-cost-functions.h, local-param-se3.h, compiled unmodified against stand-ins for
Eigen / Sophus / ceres::Jet / glog (oracle/ref_shim, recipe: `make -C oracle _ref`).  Its inputs and outputs are stored
in tests/golden/reference_kat.npz (tests/golden/make_reference_golden.py), so the comparison needs no reference checkout.

This pins to reference TEXT: the IMU cost functor incl. its RK4 integrator and the interpolation buffer (SURVEY §8 a5-a8),
UpdateImuWeights' double integrator with covariance and the hand-derived derivative tables (a9), the SE3 / SO3 local
parameterisations (a4) and the pose chain of the reprojection functor (a1).  Still recalled, not pinned: Sophus'
exp / log (stand-in written from the published formulas), Calibu's Project bodies (a2) and the Ceres loop (a12)."""
import os

import numpy as np
import pytest

from vicalib_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kat.npz")


@pytest.fixture(scope="module")
def gold():
    with np.load(GOLD) as z:
        return {k: z[k] for k in z.files}


def _problem(gold, prefix, **kw):
    """the synthetic problem of the stored inputs, with the stored IMU samples, frames and IMU parameters"""
    args = dict(models=("poly3",), n_frames=len(gold[f"{prefix}_ftime"]), grid=(14, 10), inertial=True, seed=77, ts_truth=0.003)
    args.update(kw)
    p = synth.make_problem(**args)
    for k in ("imu_t", "imu_w", "imu_a", "ftime", "T_wp", "v_w", "g", "b", "sf"):
        setattr(p, k, gold[f"{prefix}_{k}"].copy())
    p.ts = float(gold[f"{prefix}_ts"])
    return p


def test_interpolation_buffer_get_range(gold):
    """InterpolationBufferT::GetRange (interpolation-buffer.h:208-226) incl. the edges: intervals that start before the
    first sample / end after the last one, time offsets that move interval ends across samples."""
    from oracle.binding import Oracle

    p = _problem(gold, "range")
    o = Oracle(p, inertial=1)
    for (t0, t1, ts), n, rows in zip(gold["range_query"], gold["range_n"], gold["range_rows"]):
        mine = o.imu_get_range(t0, t1, ts)
        assert n == mine.shape[0]
        assert np.allclose(rows[:n], mine, rtol=1e-14, atol=1e-15), (ts, t0, t1)  # same samples; FMA contraction differs


@pytest.mark.parametrize("rot_only", [0, 1])
def test_imu_cost_functor_and_jacobian(gold, rot_only):
    """SwitchedFullImuCostFunction (ceres-cost-functions.h:379-490) with ceres::Jet<double, 35> + LocalParamSe3's Jacobian,
    as AutoDiffCostFunction evaluates it, vs the oracle's EvalImu: residual and 9 x 33 tangent Jacobian."""
    from oracle.binding import Oracle

    p = _problem(gold, "imu")
    o = Oracle(p, inertial=1, rotation_only=rot_only, bias_active=1, scale_active=1, optimize_ts=1)
    o.set_imu_weights(gold["imu_W"])
    r_o, J_o = o.eval_imu()
    for k in range(p.n_frames - 1):
        r, J = gold["imu_r"][rot_only, k], gold["imu_J"][rot_only, k]
        assert np.abs(r - r_o[k]).max() <= 1e-11 * max(1.0, np.abs(r_o[k]).max()), k
        assert np.abs(J - J_o[k]).max() <= 1e-11 * np.abs(J_o[k]).max(), k


def test_update_imu_weights(gold):
    """The loop body of ViCalibrator::UpdateImuWeights (vicalibrator.h:726-796) on the reference's double integrator with
    Jacobians + covariance (types.h:330-687) and derivative tables (vicalibrator-utils.h:106-434) vs the oracle's
    restatement: the 9 x 9 weight_sqrt_ of every interval."""
    from oracle.binding import Oracle

    assert tuple(gold["weights_sigma"]) == (synth.GYRO_SIGMA, synth.ACCEL_SIGMA)
    p = _problem(gold, "weights")
    o = Oracle(p, inertial=1, bias_active=1, scale_active=1, optimize_ts=1)
    o.update_imu_weights()
    W_o = o.imu_weights()
    for k in range(p.n_frames - 1):
        W = gold["weights_W"][k]
        assert np.abs(W - W_o[k]).max() <= 1e-8 * np.abs(W_o[k]).max(), (k, np.abs(W - W_o[k]).max() / np.abs(W_o[k]).max())


def test_local_parameterisations(gold):
    """LocalParamSe3 / LocalParamSo3 Plus and ComputeJacobian (local-param-se3.h:14-91, 107-157) vs the oracle's."""
    from oracle import binding

    h = float(gold["lp_h"])
    for x, ds, p7, p4, J, fwd, bwd in zip(gold["lp_x"], gold["lp_d"], gold["lp_se3_plus"], gold["lp_so3_plus"], gold["lp_J"],
                                          gold["lp_plus_fwd"], gold["lp_plus_bwd"]):
        for d, out, out4 in zip(ds, p7, p4):
            assert np.abs(out - binding.se3_plus(x, d)).max() <= 1e-14
            assert np.abs(out4 - binding.so3_plus(x[:4], d[3:])).max() <= 1e-14
        # the Jacobians are the derivative of Plus at delta = 0 (central differences of the REFERENCE's Plus)
        for c in range(6):
            e = np.zeros(6)
            e[c] = h
            assert np.abs(fwd[c] - binding.se3_plus(x, e)).max() <= 1e-14
            assert np.abs(bwd[c] - binding.se3_plus(x, -e)).max() <= 1e-14
            assert np.abs((fwd[c] - bwd[c]) / (2 * h) - J[:, c]).max() <= 1e-8


@pytest.mark.parametrize("model", ["fov", "poly2", "poly3", "kb4", "linear"])
def test_reprojection_functor_pose_chain(gold, model):
    """ImuReprojectionCostFunctor (ceres-cost-functions.h:342-377) with Jet<double, 22> and the reference's local
    parameterisations vs the oracle's EvalReprojection: residual and 2 x (6 + 3 + 3 + K) tangent Jacobian.  (Project itself
    is the oracle's restatement of Calibu on both sides: this pins the pose chain and the tangent-space algebra.)"""
    from oracle.binding import Oracle

    pre = f"reproj_{model}"
    p = synth.make_problem(models=(model, "poly3"), n_frames=4, seed=12, inertial=True)
    for k in ("T_wp", "intr", "q_ck", "p_ck", "obs_frame", "p_w", "p_c"):
        setattr(p, k, gold[f"{pre}_{k}"].copy())
    p.obs_cam = np.zeros(p.obs_frame.shape[0], dtype=np.int32)  # every stored observation is one of camera 0's
    o = Oracle(p, inertial=1)
    r_o, J_o = o.eval_reproj()
    assert r_o.shape[0] == gold[f"{pre}_r"].shape[0] > 0
    for r, J, ro, Jo in zip(gold[f"{pre}_r"], gold[f"{pre}_J"], r_o, J_o):
        assert np.abs(r - ro).max() <= 1e-10
        assert np.abs(J - Jo).max() <= 1e-11 * np.abs(Jo).max()
