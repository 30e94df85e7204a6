"""Problem descriptions ("wire format") and synthetic workload generators.

A ProblemSpec is the array form of what a user builds with
``ProblemCUDA::AddParameterBlock / AddResidualBlock<F, kRes, Ns...> / SetManifold /
SetParameterBlockConstant`` (reference: include/ceres/problem_cuda.h:85-486).  The
test driver (tests/driver/driver.cu) replays it through the real templated C++
API; the oracle consumes the same arrays.

Generators follow SURVEY.md section 8(d): BAL-shaped bundle adjustment problems
(examples/bal_problem.cc:81-108 layout: observations grouped by point, camera
ascending; points are elimination group 0, cameras group 1,
examples/bundle_adjuster.cu.cc:253-268) and pose-graph problems built on
internal/ceres/autodiff_benchmarks/relative_pose_error.h:46-92.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

# ---- cost type ids (shared with tests/driver/cost_types.h and oracle/oracle_eval.cc)
SNAVELY = 0             # <2, 9, 3>   examples/snavely_reprojection_error.h:52-101
SNAVELY_QUAT = 1        # <2, 10, 3>  evaluator_cuda_test.cu.cc:171-230
SNAVELY_NO_RADIAL = 2   # <2, 7, 3>   evaluator_cuda_test.cu.cc:115-164
POINT_DISPLACEMENT = 3  # <3, 3>      evaluator_cuda_test.cu.cc:83-109
RELATIVE_POSE = 4       # <6, 7, 7>   autodiff_benchmarks/relative_pose_error.h
BINARY_SCALAR = 5       # <1, 2, 2>   autodiff_cost_function_cuda_test.cu.cc:42-54
TEN_PARAMETER = 6       # <1, 1 x 10>
ONLY_FILLS_ONE = 7      # <2, 1>
AFFINE_1_3_234 = 8      # ParameterIgnoringCostFunction<1, 3, 2, 3, 4> (evaluator_test.cc:59-100)
AFFINE_1_3_432 = 9
AFFINE_1_2_23 = 10
AFFINE_2_3_24 = 11
AFFINE_3_4_34 = 12
AFFINE_FAIL = 13        # <20, 3, 2, 3, 4>(succeeds=false)
PARAMETER_SENSITIVE = 14
POSE_GRAPH_3D = 15      # <6, 3, 4, 3, 4> examples/slam/pose_graph_3d/pose_graph_3d_error_term.h
JET_BATTERY = 16        # <40, 2> every Jet operation (jet_cuda_test.cu.cc)
SQRT_OF_CONSTANT = 17   # <1, 1>  x + sqrt(T(c)): derivative of a constant sub-expression

# (num_residuals, block sizes, functor data length)
COST_TYPES = {
    SNAVELY: (2, (9, 3), 2),
    SNAVELY_QUAT: (2, (10, 3), 2),
    SNAVELY_NO_RADIAL: (2, (7, 3), 2),
    POINT_DISPLACEMENT: (3, (3,), 3),
    RELATIVE_POSE: (6, (7, 7), 7),
    BINARY_SCALAR: (1, (2, 2), 1),
    TEN_PARAMETER: (1, (1,) * 10, 0),
    ONLY_FILLS_ONE: (2, (1,), 0),
    AFFINE_1_3_234: (3, (2, 3, 4), 0),
    AFFINE_1_3_432: (3, (4, 3, 2), 0),
    AFFINE_1_2_23: (2, (2, 3), 0),
    AFFINE_2_3_24: (3, (2, 4), 0),
    AFFINE_3_4_34: (4, (3, 4), 0),
    AFFINE_FAIL: (3, (2, 3, 4), 0),
    PARAMETER_SENSITIVE: (2, (2,), 0),
    POSE_GRAPH_3D: (6, (3, 4, 3, 4), 43),
    JET_BATTERY: (40, (2,), 0),
    SQRT_OF_CONSTANT: (1, (1,), 1),
}

# ---- loss kinds (include/ceres/loss_function_cuda.h:62-149)
LOSS_NONE, LOSS_TRIVIAL, LOSS_HUBER, LOSS_CAUCHY = 0, 1, 2, 3
LOSS_SCALED_HUBER, LOSS_SCALED_CAUCHY, LOSS_SCALED_TRIVIAL = 4, 5, 6
LOSS_CONVEX_TEST = 7  # test-only user loss rho(s) = s + a s^2 (rho'' > 0)
# (tests/driver/driver_losses.cu: SnavelyReprojectionError; SoftLOne also on RelativePoseError)
LOSS_SOFT_L1, LOSS_ARCTAN, LOSS_TOLERANT, LOSS_TUKEY = 8, 9, 10, 11  # (a); Tolerant (a, b)
LOSS_SCALED_SOFT_L1, LOSS_SCALED_TUKEY = 12, 13  # ScaledLossCUDA<...>(L(a), b)
LOSS_COMPOSED = 14  # ComposedLossCUDA(ScaledLossCUDA<SoftLOneLossCUDA>(SoftLOne(a), b), Cauchy(a))

# bal_problem(loss=...) names: kind, a, b
LOSS_BY_NAME = {
    "none": (LOSS_NONE, 1.0, 0.0), "huber": (LOSS_HUBER, 1.0, 0.0),
    "cauchy": (LOSS_CAUCHY, 1.0, 0.0), "soft_l1": (LOSS_SOFT_L1, 1.0, 0.0),
    "arctan": (LOSS_ARCTAN, 1.0, 0.0), "tolerant": (LOSS_TOLERANT, 1.0, 1.0),
    "tukey": (LOSS_TUKEY, 1.0, 0.0),
}

# ---- manifold kinds (internal/ceres/manifold.cc, include/ceres/product_manifold.h)
MANIFOLD_NONE, MANIFOLD_SUBSET, MANIFOLD_QUATERNION, MANIFOLD_EIGEN_QUATERNION = 0, 1, 2, 3
MANIFOLD_QUATERNION_X_EUCLIDEAN, MANIFOLD_EIGEN_QUATERNION_X_EUCLIDEAN = 4, 5
MANIFOLD_OPAQUE_SUBSET = 6  # a SubsetManifold the kernel is not told about (generic path)

JACOBIAN_BLOCK_SPARSE, JACOBIAN_COMPRESSED_ROW = 0, 1


@dataclass
class ProblemSpec:
    pb_size: np.ndarray            # int32 [num_pb], in AddParameterBlock order
    pb_values: np.ndarray          # float64 [sum(pb_size)]
    rb_type: np.ndarray            # int32 [num_rb]
    rb_pb: np.ndarray              # int32 [sum blocks], parameter block ids per argument
    fdata: np.ndarray              # float64, functor constants concatenated in rb order
    pb_constant: np.ndarray = None        # uint8 [num_pb]
    pb_manifold_kind: np.ndarray = None   # int32 [num_pb]
    pb_manifold_param: np.ndarray = None  # int32 [num_pb]
    rb_loss_kind: np.ndarray = None       # int32 [num_rb]
    rb_loss_a: np.ndarray = None          # float64 [num_rb]
    rb_loss_b: np.ndarray = None          # float64 [num_rb]
    num_eliminate_blocks: int = 0
    meta: dict = field(default_factory=dict)

    def __post_init__(self):
        self.pb_size = np.ascontiguousarray(self.pb_size, dtype=np.int32)
        self.pb_values = np.ascontiguousarray(self.pb_values, dtype=np.float64)
        self.rb_type = np.ascontiguousarray(self.rb_type, dtype=np.int32)
        self.rb_pb = np.ascontiguousarray(self.rb_pb, dtype=np.int32)
        self.fdata = np.ascontiguousarray(self.fdata, dtype=np.float64)
        npb, nrb = self.pb_size.size, self.rb_type.size

        def _d(x, dtype, n):
            if x is None:
                return np.zeros(n, dtype=dtype)
            return np.ascontiguousarray(x, dtype=dtype)

        self.pb_constant = _d(self.pb_constant, np.uint8, npb)
        self.pb_manifold_kind = _d(self.pb_manifold_kind, np.int32, npb)
        self.pb_manifold_param = _d(self.pb_manifold_param, np.int32, npb)
        self.rb_loss_kind = _d(self.rb_loss_kind, np.int32, nrb)
        self.rb_loss_a = _d(self.rb_loss_a, np.float64, nrb)
        self.rb_loss_b = _d(self.rb_loss_b, np.float64, nrb)
        assert self.pb_values.size == int(self.pb_size.sum())

    @property
    def num_pb(self) -> int:
        return int(self.pb_size.size)

    @property
    def num_rb(self) -> int:
        return int(self.rb_type.size)


class ProblemBuilder:
    """Small-problem convenience used by the fixtures (mirrors the Problem API)."""

    def __init__(self):
        self.sizes, self.values, self.constant = [], [], []
        self.mkind, self.mparam = [], []
        self.rb_type, self.rb_pb, self.loss, self.fdata = [], [], [], []

    def add_parameter_block(self, values, manifold=(MANIFOLD_NONE, 0), constant=False) -> int:
        values = np.asarray(values, dtype=np.float64)
        self.sizes.append(values.size)
        self.values.append(values)
        self.constant.append(1 if constant else 0)
        self.mkind.append(manifold[0])
        self.mparam.append(manifold[1])
        return len(self.sizes) - 1

    def set_constant(self, pb):
        self.constant[pb] = 1

    def set_manifold(self, pb, kind, param=0):
        self.mkind[pb], self.mparam[pb] = kind, param

    def add_residual_block(self, cost_type, pbs, fdata=(), loss=(LOSS_NONE, 0.0, 0.0)):
        nres, sizes, flen = COST_TYPES[cost_type]
        assert len(pbs) == len(sizes) and len(fdata) == flen
        for pb, s in zip(pbs, sizes):
            assert self.sizes[pb] == s, "parameter block size mismatch"
        self.rb_type.append(cost_type)
        self.rb_pb.extend(pbs)
        self.fdata.extend(fdata)
        loss = tuple(loss) + (0.0,) * (3 - len(loss))
        self.loss.append(loss)

    def build(self, num_eliminate_blocks=0) -> ProblemSpec:
        loss = np.array(self.loss, dtype=np.float64).reshape(-1, 3)
        return ProblemSpec(
            pb_size=self.sizes,
            pb_values=np.concatenate(self.values) if self.values else np.zeros(0),
            rb_type=self.rb_type, rb_pb=self.rb_pb, fdata=self.fdata,
            pb_constant=self.constant, pb_manifold_kind=self.mkind,
            pb_manifold_param=self.mparam,
            rb_loss_kind=loss[:, 0].astype(np.int32), rb_loss_a=loss[:, 1],
            rb_loss_b=loss[:, 2], num_eliminate_blocks=num_eliminate_blocks)


# ------------------------------------------------------------------ BAL
BAL_SHAPES = {
    # name: (num_cameras, num_points, num_observations, seed)   SURVEY.md section 8(d)
    "S": (16, 22106, 83718, 1),
    "M": (1778, 993923, 5001946, 2),
    "L": (13682, 4456117, 28987644, 3),
}


def _rodrigues_project(cam, pt):
    """numpy restatement of SnavelyReprojectionError's projection, used only to
    synthesise observations (data generation, not a checker)."""
    aa, t = cam[:, 0:3], cam[:, 3:6]
    f, l1, l2 = cam[:, 6], cam[:, 7], cam[:, 8]
    theta = np.sqrt((aa * aa).sum(1))
    safe = np.where(theta > 0, theta, 1.0)
    w = aa / safe[:, None]
    c, s = np.cos(theta)[:, None], np.sin(theta)[:, None]
    wxp = np.cross(w, pt)
    wdp = (w * pt).sum(1)[:, None]
    p = pt * c + wxp * s + w * wdp * (1 - c)
    small = (theta == 0)[:, None]
    p = np.where(small, pt + np.cross(aa, pt), p) + t
    xp, yp = -p[:, 0] / p[:, 2], -p[:, 1] / p[:, 2]
    r2 = xp * xp + yp * yp
    d = 1.0 + r2 * (l1 + l2 * r2)
    return np.stack([f * d * xp, f * d * yp], axis=1)


def bal_problem(num_cameras, num_points, num_observations, seed=1, loss="huber",
                subset_manifold=False, constant_cameras=0) -> ProblemSpec:
    """Synthetic BAL-shaped problem (SURVEY.md section 8(d)).

    Parameter blocks: points first (elimination group 0), then cameras.  Residual
    blocks grouped by point, camera ascending.  Observation = exact projection +
    N(0, 0.5^2) px noise, 2% outliers with N(0, 20^2) so the Huber outlier branch runs.
    """
    assert num_observations >= 2 * num_points and num_cameras >= 2
    # a point is seen at most once by a camera
    assert num_observations <= num_points * num_cameras, "more observations than camera-point pairs"
    rng = np.random.default_rng(seed)
    nc, npts, nobs = num_cameras, num_points, num_observations
    # degrees: every point seen by >= 2 cameras
    extra = nobs - 2 * npts
    deg = np.full(npts, 2, dtype=np.int64)
    if extra > 0:
        deg += rng.multinomial(extra, np.full(npts, 1.0 / npts)) if npts < 200000 else \
            np.bincount(rng.integers(0, npts, size=extra), minlength=npts)
    over = deg > nc
    if over.any():  # clamp and push the excess to other points
        excess = int((deg[over] - nc).sum())
        deg[over] = nc
        room = np.flatnonzero(deg < nc)
        while excess > 0:
            take = rng.choice(room, size=min(excess, room.size), replace=False)
            deg[take] += 1
            excess -= take.size
            room = np.flatnonzero(deg < nc)
    assert int(deg.sum()) == nobs
    point_of_obs = np.repeat(np.arange(npts, dtype=np.int64), deg)
    # distinct cameras per point: skewed start + positive gaps with sum < nc
    start = np.floor(nc * rng.random(npts) ** 2).astype(np.int64)
    gmax = np.maximum(1, (nc - 1) // deg)
    gaps = 1 + np.floor(rng.random(nobs) * gmax[point_of_obs]).astype(np.int64)
    csum = np.cumsum(gaps)
    first = np.concatenate([[0], np.cumsum(deg)[:-1]])
    base = np.repeat(csum[first] - gaps[first], deg)
    cam_of_obs = (start[point_of_obs] + (csum - base)) % nc
    order = np.lexsort((cam_of_obs, point_of_obs))
    cam_of_obs = cam_of_obs[order]

    cameras = np.empty((nc, 9))
    cameras[:, 0:3] = rng.normal(0, 0.1, (nc, 3))
    cameras[:, 3:5] = rng.normal(0, 0.5, (nc, 2))
    cameras[:, 5] = -8.0 + rng.normal(0, 0.5, nc)
    cameras[:, 6] = rng.uniform(400, 1200, nc)
    cameras[:, 7] = rng.normal(0, 1e-7, nc)
    cameras[:, 8] = rng.normal(0, 1e-13, nc)
    points = rng.normal(0, 1.0, (npts, 3))

    obs = np.empty((nobs, 2))
    chunk = 4_000_000
    for lo in range(0, nobs, chunk):
        hi = min(nobs, lo + chunk)
        obs[lo:hi] = _rodrigues_project(cameras[cam_of_obs[lo:hi]], points[point_of_obs[lo:hi]])
    obs += rng.normal(0, 0.5, (nobs, 2))
    outl = rng.random(nobs) < 0.02
    obs[outl] += rng.normal(0, 20.0, (int(outl.sum()), 2))
    # the problem is evaluated at a perturbed state so residuals are not just noise
    points = points + rng.normal(0, 0.01, points.shape)

    pb_size = np.concatenate([np.full(npts, 3, np.int32), np.full(nc, 9, np.int32)])
    pb_values = np.concatenate([points.ravel(), cameras.ravel()])
    rb_pb = np.empty((nobs, 2), dtype=np.int32)
    rb_pb[:, 0] = npts + cam_of_obs  # argument 0 = camera
    rb_pb[:, 1] = point_of_obs       # argument 1 = point
    kind, loss_a, loss_b = LOSS_BY_NAME[loss]
    mk = np.zeros(npts + nc, np.int32)
    mp = np.zeros(npts + nc, np.int32)
    if subset_manifold:  # SubsetManifold(9, {0}) on every camera (BASELINE.json config 4)
        mk[npts:] = MANIFOLD_SUBSET
        mp[npts:] = 1
    const = np.zeros(npts + nc, np.uint8)
    if constant_cameras:
        const[npts:npts + constant_cameras] = 1
    return ProblemSpec(
        pb_size=pb_size, pb_values=pb_values,
        rb_type=np.full(nobs, SNAVELY, np.int32), rb_pb=rb_pb.ravel(), fdata=obs.ravel(),
        pb_constant=const, pb_manifold_kind=mk, pb_manifold_param=mp,
        rb_loss_kind=np.full(nobs, kind, np.int32), rb_loss_a=np.full(nobs, loss_a),
        rb_loss_b=np.full(nobs, loss_b), num_eliminate_blocks=npts,
        meta={"workload": f"bal-{nc}x{npts}", "num_cameras": nc, "num_points": npts,
              "num_observations": nobs, "seed": seed})


def bal_shape(name, scale=1.0, **kw) -> ProblemSpec:
    nc, npts, nobs, seed = BAL_SHAPES[name]
    if scale != 1.0:
        nc = max(2, int(nc * scale))
        npts = max(4, int(npts * scale))
        nobs = max(2 * npts, int(nobs * scale))
    return bal_problem(nc, npts, nobs, seed=seed, **kw)


# ------------------------------------------------------------ pose graph
def _quat_mul_xyzw(a, b):
    ax, ay, az, aw = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bx, by, bz, bw = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([
        aw * bx + ax * bw + ay * bz - az * by,
        aw * by + ay * bw + az * bx - ax * bz,
        aw * bz + az * bw + ax * by - ay * bx,
        aw * bw - ax * bx - ay * by - az * bz], axis=-1)


def _quat_conj_xyzw(a):
    return a * np.array([-1.0, -1.0, -1.0, 1.0])


def _quat_rot_xyzw(q, v):
    u = q[..., :3]
    uv = 2.0 * np.cross(u, v)
    return v + q[..., 3:4] * uv + np.cross(u, uv)


def _small_quat(rng, n, sigma):
    w = rng.normal(0, sigma, (n, 3))
    th = np.linalg.norm(w, axis=1, keepdims=True)
    safe = np.where(th > 0, th, 1.0)
    q = np.concatenate([np.sin(th / 2) * w / safe, np.cos(th / 2)], axis=1)
    return q


def pose_graph_problem(num_poses, num_edges, seed=5, loss="none", order="temporal") -> ProblemSpec:
    """Pose-graph SLAM, RelativePoseError<6,7,7>, pose = [q(x,y,z,w), t],
    ProductManifold<EigenQuaternionManifold, EuclideanManifold<3>> (7 -> 6),
    pose 0 constant (SURVEY.md section 8(d), config 5).

    order="temporal" (default): edges in the order a SLAM front end emits them and g2o files
    list them - an edge appears when its later pose is created, so the list is sorted by
    max(i, j).  order="random": odometry edges first, then the loop closures in random order
    (the same edges; worst case for locality: every edge touches two random poses)."""
    assert num_edges >= num_poses - 1
    rng = np.random.default_rng(seed)
    n = num_poses
    # random-walk trajectory (ground truth)
    dq = _small_quat(rng, n, 0.2)
    dt = rng.normal(0, 0.5, (n, 3)) + np.array([1.0, 0, 0])
    q = np.empty((n, 4)); t = np.empty((n, 3))
    q[0] = [0, 0, 0, 1]; t[0] = 0
    # sequential composition is inherently serial; do it in blocks of python loops
    # only for small n, vectorised "independent pose" placement for big n.
    if n <= 200000:
        for i in range(1, n):
            q[i] = _quat_mul_xyzw(q[i - 1], dq[i]); q[i] /= np.linalg.norm(q[i])
            t[i] = t[i - 1] + _quat_rot_xyzw(q[i - 1], dt[i])
    else:
        q = _small_quat(rng, n, 1.0)
        t = np.cumsum(dt, axis=0)
    # edges: odometry + random loop closures
    i_idx = np.concatenate([np.arange(n - 1), rng.integers(0, n, num_edges - (n - 1))])
    off = rng.integers(2, max(3, min(n, 50)), num_edges - (n - 1))
    j_idx = np.concatenate([np.arange(1, n), (i_idx[n - 1:] + off) % n])
    same = i_idx == j_idx
    j_idx[same] = (j_idx[same] + 1) % n
    # measurement: true relative pose j<-i perturbed; functor computes
    # res = meas * (q_j^-1 q_i), so meas ~ (q_j^-1 q_i)^-1 = q_i^-1 q_j
    qi, qj, ti, tj = q[i_idx], q[j_idx], t[i_idx], t[j_idx]
    est_q = _quat_mul_xyzw(_quat_conj_xyzw(qj), qi)
    est_t = _quat_rot_xyzw(_quat_conj_xyzw(qj), ti - tj)
    meas_q = _quat_mul_xyzw(_small_quat(rng, num_edges, 0.01), _quat_conj_xyzw(est_q))
    meas_q /= np.linalg.norm(meas_q, axis=1, keepdims=True)
    meas_t = -_quat_rot_xyzw(meas_q, est_t) + rng.normal(0, 0.01, (num_edges, 3))
    fdata = np.concatenate([meas_q, meas_t], axis=1)
    if order == "temporal":
        perm = np.argsort(np.maximum(i_idx, j_idx), kind="stable")
        i_idx, j_idx, fdata = i_idx[perm], j_idx[perm], fdata[perm]
    else:
        assert order == "random"
    # evaluate at a perturbed state
    qn = _quat_mul_xyzw(q, _small_quat(rng, n, 0.02))
    qn /= np.linalg.norm(qn, axis=1, keepdims=True)
    poses = np.concatenate([qn, t + rng.normal(0, 0.02, (n, 3))], axis=1)
    const = np.zeros(n, np.uint8); const[0] = 1
    kind = {"none": LOSS_NONE, "cauchy": LOSS_CAUCHY, "huber": LOSS_HUBER}[loss]
    rb_pb = np.stack([i_idx, j_idx], axis=1).astype(np.int32)
    return ProblemSpec(
        pb_size=np.full(n, 7, np.int32), pb_values=poses.ravel(),
        rb_type=np.full(num_edges, RELATIVE_POSE, np.int32), rb_pb=rb_pb.ravel(),
        fdata=fdata.ravel(), pb_constant=const,
        pb_manifold_kind=np.full(n, MANIFOLD_EIGEN_QUATERNION_X_EUCLIDEAN, np.int32),
        pb_manifold_param=np.zeros(n, np.int32),
        rb_loss_kind=np.full(num_edges, kind, np.int32), rb_loss_a=np.full(num_edges, 1.0),
        rb_loss_b=np.zeros(num_edges), num_eliminate_blocks=0,
        meta={"workload": f"pose-graph-{n}x{num_edges}", "seed": seed, "edge_order": order})


# ------------------------------------------------------ reference fixtures
def evaluator_cuda_test_problem() -> ProblemSpec:
    """The 6-residual-block problem of internal/ceres/evaluator_cuda_test.cu.cc:232-316."""
    camera1 = [9.99946154126841180165e-01, 7.87061670168454075025e-03,
               -6.39535329165887445751e-03, -2.20038540935716883662e-03,
               -3.4093839577186584e-02, -1.0751387104921525e-01, 1.1202240291236032e+00,
               3.9975152639358436e+02, -3.1770643852803579e-07, 5.8820490534594022e-13]
    camera2 = [9.99877513605250900497e-01, 7.98833588996764563939e-03,
               -1.26117173449355086945e-02, -4.69987892415464365153e-03,
               -8.5667661408224093e-03, -1.2188049069425422e-01, 7.1901330750094605e-01,
               4.0201753385955931e+02, -3.7804765613385677e-07, 9.3074311683844792e-13]
    camera3 = [1.4846251175275622e-02, -2.1062899405576294e-02, -1.1669480098224182e-03,
               -2.4950970734443037e-02, -1.1398470545726247e-01, 9.2166020737027976e-01,
               4.0040175368358570e+02]
    point1 = [-6.1200015717226364e-01, 5.7175904776028286e-01, -1.8470812764548823e+00]
    point2 = [1.7074972220818254e+00, 9.5386921723786655e-01, -6.8771685779735616e+00]
    b = ProblemBuilder()
    # parameter blocks enter the program in first-use order
    c1 = b.add_parameter_block(camera1)
    p1 = b.add_parameter_block(point1)
    c2 = b.add_parameter_block(camera2)
    p2 = b.add_parameter_block(point2)
    c3 = b.add_parameter_block(camera3)
    cauchy, huber = (LOSS_CAUCHY, 1.0), (LOSS_HUBER, 1.0)
    b.add_residual_block(SNAVELY_QUAT, [c1, p1], [-3.326500e+02, 2.620900e+02], cauchy)
    b.add_residual_block(SNAVELY_QUAT, [c2, p1], [-1.997600e+02, 1.667000e+02], cauchy)
    b.add_residual_block(SNAVELY_QUAT, [c1, p2], [1.224100e+02, 6.554999e+01], cauchy)
    b.add_residual_block(SNAVELY_NO_RADIAL, [c3, p1], [-2.530600e+02, 2.022700e+02], huber)
    b.add_residual_block(POINT_DISPLACEMENT, [p1], point1)
    b.add_residual_block(POINT_DISPLACEMENT, [p2], point2)
    b.set_constant(c2)
    b.set_constant(p2)
    b.set_manifold(c1, MANIFOLD_QUATERNION_X_EUCLIDEAN)
    return b.build(num_eliminate_blocks=0)
