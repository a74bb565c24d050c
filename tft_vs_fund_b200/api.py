"""Host-side mirror of the reference's function interface, over the C ABI.

Same names, argument meaning and error behaviour as the MATLAB functions they
stand in for (file:line into the reference in every docstring), so the parity
tests read like calls of the reference.  Arrays use the MATLAB shapes:
``Corresp`` 6xN, ``CalM`` 9x3, poses 3x4, ``T`` 3x3x3 with ``T[:, :, i]`` the
i-th slice, ``Reconst`` 3xN.  Every function also takes a leading batch axis
(``Corresp`` (B,6,N), ``CalM`` (9,3) or (B,9,3)) and then returns batched
arrays ((B,3,4), (B,3,N), (B,3,3,3), ...).

All arithmetic happens in libtvf.so on the GPU; this module only reshapes
between NumPy (row-major) and the library's MATLAB column-major layout.
"""
import ctypes as C

import numpy as np

from . import _lib

_dp = _lib.c_double_p
_ip = _lib.c_int32_p


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


# ---- layout helpers ---------------------------------------------------------------------------
def _cm(a, nd):
    """MATLAB array (optionally with a leading batch axis) -> flat column-major buffer.
    `nd` = number of MATLAB dimensions.  Returns (buffer, batched, B)."""
    a = np.asarray(a, dtype=np.float64)
    batched = a.ndim == nd + 1
    if not batched:
        if a.ndim != nd:
            raise ValueError("expected %d-D array (or %d-D with a leading batch axis), got shape %s"
                             % (nd, nd + 1, a.shape))
        a = a[None]
    axes = (0,) + tuple(range(nd, 0, -1))            # (B, d1..dn) -> (B, dn..d1): column-major per item
    return np.ascontiguousarray(a.transpose(axes)), batched, a.shape[0]


def _from_cm(buf, B, dims, batched):
    """flat column-major buffer -> (B, *dims) (or dims when not batched)."""
    nd = len(dims)
    a = buf.reshape((B,) + tuple(reversed(dims))).transpose((0,) + tuple(range(nd, 0, -1)))
    return a if batched else a[0]


def _calm(CalM, B):
    CalM = np.asarray(CalM, dtype=np.float64)
    if CalM.ndim == 2:
        if CalM.shape != (9, 3):
            raise ValueError("CalM must be 9x3")
        return np.ascontiguousarray(CalM.T), 0
    if CalM.shape != (B, 9, 3):
        raise ValueError("batched CalM must be (B,9,3)")
    return np.ascontiguousarray(CalM.transpose(0, 2, 1)), 1


class PoseResult(tuple):
    """(R_t_2, R_t_3, Reconst, T, iter) like the reference, plus .repr_err, .status, .votes (and .F21/.F31).
    votes: (B,10) int32 -- the cheirality votes of recover_R_t (R_t_from_TFT.m:91-104): 4 for pair (1,2), 4 for pair
    (1,3) in the reference's candidate order, then the two NaN bit masks."""
    repr_err = None
    status = None
    votes = None
    F21 = None
    F31 = None


def _vp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _pose(method, Corresp, CalM, device):
    h = _lib.handle(device)
    c, batched, B = _cm(Corresp, 2)
    if c.shape[2] != 6:
        raise ValueError("Corresp must be 6xN")
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    Rt2 = np.empty((B, 12)); Rt3 = np.empty((B, 12)); Rec = np.empty((B, 3 * n)); T = np.empty((B, 27))
    rep = np.empty(B); st = np.zeros(B, dtype=np.int32); votes = np.zeros((B, 10), dtype=np.int32)
    F21 = F31 = its = None
    if method != "tft":
        F21 = np.empty((B, 9)); F31 = np.empty((B, 9))
    if method == "optf":
        its = np.zeros(B, dtype=np.int32)
    out = _lib.PoseOut(_vp(Rt2), _vp(Rt3), _vp(Rec), _vp(T), _vp(rep), _vp(F21), _vp(F31), _vp(its), _vp(votes), _vp(st))
    h.call("tvf_pose", _lib.METHOD_IDS[method], _p(c), _p(calm), cb, n, B, C.byref(out))
    it = np.zeros(B) if batched else 0                      # iter=0  (LinearTFTPoseEstimation.m:62)
    if method == "optf":
        it = its.astype(np.float64) if batched else int(its[0])      # iter=it1+it2 (OptimFPoseEstimation.m:49)
    out = PoseResult((_from_cm(Rt2, B, (3, 4), batched), _from_cm(Rt3, B, (3, 4), batched),
                      _from_cm(Rec, B, (3, n), batched), _from_cm(T, B, (3, 3, 3), batched), it))
    out.repr_err = rep if batched else float(rep[0])
    out.status = st if batched else int(st[0])
    out.votes = votes if batched else votes[0]
    if F21 is not None:
        out.F21 = _from_cm(F21, B, (3, 3), batched); out.F31 = _from_cm(F31, B, (3, 3), batched)
    if not batched and (out.status & (_lib.ST_NO_POSE_2 | _lib.ST_NO_POSE_3)):
        # the reference fails here with "Undefined function or variable 'R_f'" (R_t_from_TFT.m:91-104)
        raise _lib.TvfError("recover_R_t: no candidate pose received a non-negative vote (R_f undefined)")
    return out


def LinearTFTPoseEstimation(Corresp, CalM, device=None):
    """[R_t_2,R_t_3,Reconst,T,iter]=LinearTFTPoseEstimation(Corresp,CalM)
    (TFT_methods/LinearTFTPoseEstimation.m:1,45-62)."""
    return _pose("tft", Corresp, CalM, device)


def LinearFPoseEstimation(Corresp, CalM, device=None):
    """[R_t_2,R_t_3,Reconst,T,iter]=LinearFPoseEstimation(Corresp,CalM)
    (F_methods/LinearFPoseEstimation.m:1,42-78).  Raises ValueError with linearF's message for N<8."""
    return _pose("f", Corresp, CalM, device)


def OptimFPoseEstimation(Corresp, CalM, device=None):
    """[R_t_2,R_t_3,Reconst,T,iter]=OptimFPoseEstimation(Corresp,CalM)
    (F_methods/OptimFPoseEstimation.m:1,43-72): both F refined by optimF's Gauss-Helmert iteration."""
    c = np.asarray(Corresp)
    if c.shape[-1] < 8:
        raise ValueError(_lib.LINEARF_ERRMSG)                          # optimF.m:36-38
    return _pose("optf", Corresp, CalM, device)


def optimF(p1, p2, device=None):
    """[F,iter]=optimF(p1,p2) (F_methods/optimF.m:1,34-78).  ValueError (optimF.m:37 text) if N<8 or N differs."""
    a, batched, B = _cm(p1, 2); b, _, _ = _cm(p2, 2)
    if a.shape[1] != b.shape[1] or a.shape[1] < 8:                    # optimF.m:36-38
        raise ValueError(_lib.LINEARF_ERRMSG)
    h = _lib.handle(device)
    rows, n = a.shape[2], a.shape[1]
    if b.shape != a.shape or rows not in (2, 3):
        raise ValueError("p1,p2 must both be 2xN or 3xN")
    F = np.empty((B, 9)); its = np.zeros(B, dtype=np.int32)
    h.call("tvf_optim_f", _p(a), _p(b), rows, n, B, _p(F), its.ctypes.data_as(_ip), None)
    return _from_cm(F, B, (3, 3), batched), (its.astype(np.float64) if batched else int(its[0]))


def linearTFT(p1, p2, p3, device=None):
    """[T,P1,P2,P3]=linearTFT(p1,p2,p3) (TFT_methods/linearTFT.m:1,36-91); p* are 2xN or 3xN."""
    h = _lib.handle(device)
    a, batched, B = _cm(p1, 2); b, _, _ = _cm(p2, 2); c, _, _ = _cm(p3, 2)
    rows, n = a.shape[2], a.shape[1]
    if b.shape != a.shape or c.shape != a.shape or rows not in (2, 3):
        raise ValueError("p1,p2,p3 must all be 2xN or 3xN")
    T = np.empty((B, 27)); P2 = np.empty((B, 12)); P3 = np.empty((B, 12))
    h.call("tvf_linear_tft", _p(a), _p(b), _p(c), rows, n, B, _p(T), _p(P2), _p(P3), None)
    P1 = np.eye(3, 4) if not batched else np.broadcast_to(np.eye(3, 4), (B, 3, 4)).copy()   # linearTFT.m:88
    return (_from_cm(T, B, (3, 3, 3), batched), P1, _from_cm(P2, B, (3, 4), batched),
            _from_cm(P3, B, (3, 4), batched))


def linearF(p1, p2, device=None):
    """F=linearF(p1,p2) (F_methods/linearF.m:1,32-62).  ValueError (linearF.m:36 text) if N<8 or N differs."""
    a, batched, B = _cm(p1, 2); b, _, _ = _cm(p2, 2)
    if a.shape[1] != b.shape[1] or a.shape[1] < 8:                    # linearF.m:35-37
        raise ValueError(_lib.LINEARF_ERRMSG)
    h = _lib.handle(device)
    rows, n = a.shape[2], a.shape[1]
    if b.shape != a.shape or rows not in (2, 3):
        raise ValueError("p1,p2 must both be 2xN or 3xN")
    F = np.empty((B, 9))
    h.call("tvf_linear_f", _p(a), _p(b), rows, n, B, _p(F), None)
    return _from_cm(F, B, (3, 3), batched)


def Normalize2Ddata(points, device=None):
    """[new_points,N_matrix]=Normalize2Ddata(points) (auxiliar_functions/Normalize2Ddata.m:1,33-39)."""
    h = _lib.handle(device)
    a, batched, B = _cm(points, 2)
    n = a.shape[1]
    out = np.empty((B, 2 * n)); N = np.empty((B, 9))
    h.call("tvf_normalize2d", _p(a), n, B, _p(out), _p(N))
    return _from_cm(out, B, (2, n), batched), _from_cm(N, B, (3, 3), batched)


def transform_TFT(T_old, M1, M2, M3, inverse=0, device=None):
    """T_new=transform_TFT(T_old,M1,M2,M3,inverse) (TFT_methods/transform_TFT.m:1,32-49)."""
    h = _lib.handle(device)
    t, batched, B = _cm(T_old, 3)
    m1, mb, _ = _cm(M1, 2); m2, _, _ = _cm(M2, 2); m3, _, _ = _cm(M3, 2)
    out = np.empty((B, 27))
    h.call("tvf_transform_tft", _p(t), _p(m1), _p(m2), _p(m3), int(mb), int(inverse), B, _p(out))
    return _from_cm(out, B, (3, 3, 3), batched)


def R_t_from_TFT(T, CalM, Corresp, device=None, return_votes=False):
    """[R_t_2,R_t_3]=R_t_from_TFT(T,CalM,Corresp) (TFT_methods/R_t_from_TFT.m:1,40-106).  return_votes=True appends
    the (B,10) / (10,) int32 cheirality votes of the local recover_R_t (:91-104; layout: see PoseResult)."""
    h = _lib.handle(device)
    t, batched, B = _cm(T, 3)
    c, _, _ = _cm(Corresp, 2)
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    Rt2 = np.empty((B, 12)); Rt3 = np.empty((B, 12)); st = np.zeros(B, dtype=np.int32)
    votes = np.zeros((B, 10), dtype=np.int32)
    h.call("tvf_rt_from_tft", _p(t), _p(calm), cb, _p(c), n, B, _p(Rt2), _p(Rt3), votes.ctypes.data_as(_ip),
           st.ctypes.data_as(_ip))
    out = (_from_cm(Rt2, B, (3, 4), batched), _from_cm(Rt3, B, (3, 4), batched))
    return out + ((votes if batched else votes[0]),) if return_votes else out


def TFT_from_P(P1, P2, P3, device=None):
    """T=TFT_from_P(P1,P2,P3) (TFT_methods/TFT_from_P.m:1,25-33)."""
    h = _lib.handle(device)
    a, batched, B = _cm(P1, 2); b, _, _ = _cm(P2, 2); c, _, _ = _cm(P3, 2)
    out = np.empty((B, 27))
    h.call("tvf_tft_from_p", _p(a), _p(b), _p(c), B, _p(out))
    return _from_cm(out, B, (3, 3, 3), batched)


def _cams(Pcam, B, batched):
    """cell array of M 3x4 matrices -> (buffer 3x4xM[xB], M, cams_batched)."""
    Ps = [np.asarray(P, dtype=np.float64) for P in Pcam]
    M = len(Ps)
    cb = int(Ps[0].ndim == 3)
    if cb:
        arr = np.stack(Ps, axis=1)                       # (B, M, 3, 4)
        buf = np.ascontiguousarray(arr.transpose(0, 1, 3, 2))
    else:
        arr = np.stack(Ps, axis=0)                       # (M, 3, 4)
        buf = np.ascontiguousarray(arr.transpose(0, 2, 1))
    return buf, M, cb


def triangulation3D(Pcam, image_points, device=None):
    """space_points=triangulation3D(Pcam,image_points) (auxiliar_functions/triangulation3D.m:1,32-64).
    Returns 4xN unit vectors; None where the reference returns without assigning (:33-35,:46-47)."""
    M = len(Pcam)
    if M < 2:
        return None
    pts, batched, B = _cm(image_points, 2)
    n, r = pts.shape[1], pts.shape[2]
    if r == 2 * M:
        rows = 2
    elif r == 3 * M:
        rows = 3
    else:
        return None
    h = _lib.handle(device)
    buf, M, cb = _cams(Pcam, B, batched)
    X = np.empty((B, 4 * n))
    h.call("tvf_triangulate", _p(buf), M, cb, _p(pts), rows, n, B, _p(X))
    return _from_cm(X, B, (4, n), batched)


def ReprError(ProjM, Corresp, Points3D=None, device=None):
    """error=ReprError(ProjM,Corresp,Points3D) (auxiliar_functions/ReprError.m:1,39-65)."""
    h = _lib.handle(device)
    M = len(ProjM)
    c, batched, B = _cm(Corresp, 2)
    n, r = c.shape[1], c.shape[2]
    rows = 3 if r == 3 * M else 2
    buf, M, cb = _cams(ProjM, B, batched)
    x = None; pr = 0
    if Points3D is not None:
        x, _, _ = _cm(Points3D, 2); pr = x.shape[2]
    err = np.empty(B)
    h.call("tvf_repr_error", _p(buf), M, cb, _p(c), rows, n, B, _p(x), pr, _p(err))
    return err if batched else float(err[0])


def project3Dpoints(Points3D, Pcam, device=None):
    """Corresp=project3Dpoints(Points3D,Pcam) (auxiliar_functions/project3Dpoints.m:1,28-35): 3xN -> 2MxN."""
    h = _lib.handle(device)
    x, batched, B = _cm(Points3D, 2)
    n = x.shape[1]
    buf, M, cb = _cams(Pcam, B, batched)
    out = np.empty((B, 2 * M * n))
    h.call("tvf_project3d", _p(x), _p(buf), M, cb, n, B, _p(out))
    return _from_cm(out, B, (2 * M, n), batched)


def AngError(R_t_true, R_t_est, device=None):
    """[rot_err,t_err]=AngError(R_t_true,R_t_est) (auxiliar_functions/AngError.m:1,21-28), degrees."""
    h = _lib.handle(device)
    e, batched, B = _cm(R_t_est, 2)
    t, tb, _ = _cm(R_t_true, 2)
    rot = np.empty(B); tr = np.empty(B)
    h.call("tvf_ang_error", _p(t), int(tb), _p(e), B, _p(rot), _p(tr))
    return (rot, tr) if batched else (float(rot[0]), float(tr[0]))


class BundleAdjustResult(tuple):
    """(R_t_2, R_t_3, Reconst, iter) of bundle_adjust, plus .repr_err and .status.  epfl.run_real(covariance=True) also
    sets .sigma2 and the predicted RMS errors .pred_rot_err, .pred_t_err (degrees, mean of views 2 and 3)."""
    repr_err = None
    status = None
    sigma2 = None
    pred_rot_err = None
    pred_t_err = None


def bundle_adjust(Corresp, CalM, R_t_2, R_t_3, Reconst=None, device=None):
    """Three-view bundle adjustment of a pose (tvf_bundle_adjust, include/tvf.h): minimises the pixel reprojection error
    over R2, t2 (|t2| = 1), R3, t3 and the points, camera 1 fixed at K1[I|0], from the start (R_t_2, R_t_3, Reconst).
    Reconst None: the start points are triangulated from the start poses.  Not the reference's BundleAdjustment.m (which
    normalises the image data first; DESIGN.md section 8).  Returns (R_t_2, R_t_3, Reconst, iter) with .repr_err (the
    result's ReprError) and .status (TVF_ST_* bits: NONFINITE, BA_NOCONV)."""
    c, batched, B = _cm(Corresp, 2)
    if c.shape[2] != 6:
        raise ValueError("Corresp must be 6xN")
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    r2, _, _ = _cm(np.broadcast_to(R_t_2, (B, 3, 4)) if batched else R_t_2, 2)
    r3, _, _ = _cm(np.broadcast_to(R_t_3, (B, 3, 4)) if batched else R_t_3, 2)
    x0 = None
    if Reconst is not None:
        x0, _, _ = _cm(Reconst, 2)
        if x0.shape != (B, n, 3):
            raise ValueError("Reconst must be 3xN (with the batch axis of Corresp)")
    if r2.shape != (B, 4, 3) or r3.shape != (B, 4, 3):
        raise ValueError("R_t_2, R_t_3 must be 3x4 (with the batch axis of Corresp)")
    h = _lib.handle(device)
    Rt2 = np.empty((B, 12)); Rt3 = np.empty((B, 12)); Rec = np.empty((B, 3 * n)); rep = np.empty(B)
    its = np.zeros(B, dtype=np.int32); st = np.zeros(B, dtype=np.int32)
    h.call("tvf_bundle_adjust", _p(c), _p(calm), cb, n, B, _p(r2), _p(r3), _p(x0), _p(Rt2), _p(Rt3), _p(Rec), _p(rep),
           its.ctypes.data_as(_ip), st.ctypes.data_as(_ip))
    out = BundleAdjustResult((_from_cm(Rt2, B, (3, 4), batched), _from_cm(Rt3, B, (3, 4), batched),
                              _from_cm(Rec, B, (3, n), batched), its if batched else int(its[0])))
    out.repr_err = rep if batched else float(rep[0])
    out.status = st if batched else int(st[0])
    return out


class CovarianceResult(tuple):
    """(cov_cam, sigma2) of ba_covariance, plus .cov_pts (None unless points=True) and .status."""
    cov_pts = None
    status = None


def ba_covariance(Corresp, CalM, R_t_2, R_t_3, Reconst, points=False, device=None):
    """First-order covariance of the bundle adjustment at the state (R_t_2, R_t_3, Reconst), usually bundle_adjust's
    result (tvf_ba_covariance, include/tvf.h).  The state is first scaled to |t2| = 1 as bundle_adjust does.  Returns
    (cov_cam, sigma2): cov_cam 12x12 over [w2, dt2, w3, dt3] (rotation vectors R <- exp([w]x) R and translation
    perturbations, rank 11, null direction (0, t2, 0, 0)), for UNIT pixel noise -- multiply by sigma2, the a-posteriori
    noise variance sum r^2 / (3N - 11), or by any other sigma^2.  points=True also fills .cov_pts, 3x3xN (the marginal
    covariance of each point in the gauge-normalised frame, unit noise).  .status: TVF_ST_* bits (NONFINITE,
    COV_SINGULAR); a flagged problem's outputs are NaN.  Batched like bundle_adjust: cov_cam (B,12,12), sigma2 (B,),
    cov_pts (B,3,3,N)."""
    c, batched, B = _cm(Corresp, 2)
    if c.shape[2] != 6:
        raise ValueError("Corresp must be 6xN")
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    r2, _, _ = _cm(np.broadcast_to(R_t_2, (B, 3, 4)) if batched else R_t_2, 2)
    r3, _, _ = _cm(np.broadcast_to(R_t_3, (B, 3, 4)) if batched else R_t_3, 2)
    x, _, _ = _cm(Reconst, 2)
    if r2.shape != (B, 4, 3) or r3.shape != (B, 4, 3):
        raise ValueError("R_t_2, R_t_3 must be 3x4 (with the batch axis of Corresp)")
    if x.shape != (B, n, 3):
        raise ValueError("Reconst must be 3xN (with the batch axis of Corresp)")
    h = _lib.handle(device)
    cc = np.empty((B, 144)); s2 = np.empty(B); st = np.zeros(B, dtype=np.int32)
    cp = np.empty((B, 9 * n)) if points else None
    h.call("tvf_ba_covariance", _p(c), _p(calm), cb, n, B, _p(r2), _p(r3), _p(x), _p(cc), _p(cp), _p(s2),
           st.ctypes.data_as(_ip))
    out = CovarianceResult((_from_cm(cc, B, (12, 12), batched), s2 if batched else float(s2[0])))
    if points:
        out.cov_pts = _from_cm(cp, B, (3, 3, n), batched)
    out.status = st if batched else int(st[0])
    return out


def _pose_pair(R_t_2, R_t_3, B, batched):
    r2, _, _ = _cm(np.broadcast_to(R_t_2, (B, 3, 4)) if batched else R_t_2, 2)
    r3, _, _ = _cm(np.broadcast_to(R_t_3, (B, 3, 4)) if batched else R_t_3, 2)
    if r2.shape != (B, 4, 3) or r3.shape != (B, 4, 3):
        raise ValueError("R_t_2, R_t_3 must be 3x4 (with the batch axis of Corresp)")
    return r2, r3


def consensus(Corresp, CalM, R_t_2, R_t_3, threshold=1.0, device=None):
    """Which matches of Corresp (6xN) the pose (R_t_2, R_t_3) explains (tvf_consensus, include/tvf.h): each match is
    triangulated with K1[I|0], K2*R_t_2, K3*R_t_3, re-projected, and kept iff its six residuals are finite and
    <= threshold pixels -- the inlier rule of experiments_real.m:94-98 (epfl.inlier_filter), except that a NaN
    residual makes the match an outlier.  Returns (mask, count): bool (N) and int, or (B,N) and (B,) when batched."""
    c, batched, B = _cm(Corresp, 2)
    if c.shape[2] != 6:
        raise ValueError("Corresp must be 6xN")
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    r2, r3 = _pose_pair(R_t_2, R_t_3, B, batched)
    h = _lib.handle(device)
    mask = np.zeros((B, n), dtype=np.uint8); cnt = np.zeros(B, dtype=np.int32)
    h.call("tvf_consensus", _p(c), _p(calm), cb, n, B, _p(r2), _p(r3), float(threshold), _vp(mask), cnt.ctypes.data_as(_ip))
    mask = mask.astype(bool)
    return (mask, cnt) if batched else (mask[0], int(cnt[0]))


class RansacResult(tuple):
    """(R_t_2, R_t_3, inliers, n_inliers, sample) of ransac_pose, plus .status (0, or TVF_ST_RANSAC_FAILED)."""
    status = None


RANSAC_SAMPLE_SIZE = {1: 7, 7: 8}


def ransac_pose(Corresp, CalM, method=1, hypotheses=1024, threshold=1.0, seed=0, device=None):
    """Pose from raw matches with outliers (tvf_ransac_pose, include/tvf.h): `hypotheses` minimal solves of method 1
    (LinearTFTPoseEstimation on 7 matches) or 7 (LinearFPoseEstimation on 8), each scored by its consensus (see
    `consensus`, `threshold` pixels); the method is then run again on the consensus of the best one and that refit is
    kept if it explains at least as many matches.  seed: int (problem b gets the key seed + b) or an array (B,) of keys.
    Returns (R_t_2, R_t_3, inliers, n_inliers, sample) -- inliers bool (N), the sample the best hypothesis drew -- with
    .status; batched inputs give (B,3,4), (B,3,4), (B,N), (B,), (B,s)."""
    if method not in RANSAC_SAMPLE_SIZE:
        raise ValueError("ransac_pose: method must be 1 (linear TFT) or 7 (linear F)")
    s = RANSAC_SAMPLE_SIZE[method]
    c, batched, B = _cm(Corresp, 2)
    if c.shape[2] != 6:
        raise ValueError("Corresp must be 6xN")
    n = c.shape[1]
    calm, cb = _calm(CalM, B)
    if np.ndim(seed) == 0:
        seeds = (np.uint64(int(seed) % 2 ** 64) + np.arange(B, dtype=np.uint64)).astype(np.uint64)
    else:
        seeds = np.ascontiguousarray(seed, dtype=np.uint64)
        if seeds.shape != (B,):
            raise ValueError("seed must be an int or an array of B keys")
    h = _lib.handle(device)
    Rt2 = np.empty((B, 12)); Rt3 = np.empty((B, 12)); mask = np.zeros((B, n), dtype=np.uint8)
    cnt = np.zeros(B, dtype=np.int32); smp = np.zeros((B, s), dtype=np.int32); st = np.zeros(B, dtype=np.int32)
    h.call("tvf_ransac_pose", int(method), _p(c), _p(calm), cb, n, B, int(hypotheses), float(threshold), _vp(seeds),
           _p(Rt2), _p(Rt3), _vp(mask), cnt.ctypes.data_as(_ip), smp.ctypes.data_as(_ip), st.ctypes.data_as(_ip))
    mask = mask.astype(bool)
    out = RansacResult((_from_cm(Rt2, B, (3, 4), batched), _from_cm(Rt3, B, (3, 4), batched),
                        mask if batched else mask[0], cnt if batched else int(cnt[0]), smp if batched else smp[0]))
    out.status = st if batched else int(st[0])
    return out


def pose_rms_errors(cov_cam, R_t_2, R_t_3, sigma2=1.0):
    """First-order RMS of the errors AngError measures (auxiliar_functions/AngError.m), in degrees, from a 12x12
    cov_cam of ba_covariance (unit noise) scaled by sigma2: returns (rot_err, t_err), each [view 2, view 3] (shape (2,),
    or (B,2) for batched inputs).  Rotation: sqrt(trace Sigma_w); t2 direction: sqrt(trace Sigma_t2) (|t2| = 1 in the
    covariance's gauge); t3 direction: the t3 block projected on the tangent plane of t3/|t3|, over |t3|^2.  R_t_2 and
    R_t_3 are the state the covariance was taken at (any scale: t3 is taken relative to |t2|)."""
    cov = np.asarray(cov_cam, dtype=np.float64)
    batched = cov.ndim == 3
    cov = cov if batched else cov[None]
    s2 = np.broadcast_to(np.asarray(sigma2, dtype=np.float64), cov.shape[:1])
    t2 = np.asarray(R_t_2, dtype=np.float64).reshape(-1, 3, 4)[:, :, 3]
    t3 = np.asarray(R_t_3, dtype=np.float64).reshape(-1, 3, 4)[:, :, 3] / np.linalg.norm(t2, axis=1)[:, None]
    d3 = t3 / np.linalg.norm(t3, axis=1)[:, None]
    P = np.eye(3) - d3[:, :, None] * d3[:, None, :]
    tr = lambda k: np.trace(cov[:, k:k + 3, k:k + 3], axis1=1, axis2=2)
    t3v = np.trace(P @ cov[:, 9:12, 9:12] @ P, axis1=1, axis2=2) / np.sum(t3 * t3, axis=1)
    deg = 180.0 / np.pi
    rot = np.sqrt(s2[:, None] * np.stack([tr(0), tr(6)], 1)) * deg
    tdir = np.sqrt(s2[:, None] * np.stack([tr(3), t3v], 1)) * deg
    return (rot, tdir) if batched else (rot[0], tdir[0])


def crossM(v):
    """M=crossM(v) (auxiliar_functions/crossM.m:22) -- pure data placement, no arithmetic."""
    v = np.asarray(v, dtype=np.float64).ravel()
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])
