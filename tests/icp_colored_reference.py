"""A plain numpy/scipy reference of cwipc_cuda_estimate_color_gradients and cwipc_cuda_icp_colored (no library calls): the
rules include/cwipc_util_cuda.h states, step by step.  Neighbourhoods, normals, the solve and the Euler matrix are
tests/icp_plane_reference.py's; the moving, matching and looping are tests/icp_reference.py's.

- Intensity: (r + g + b) / 765 in float64, the integer sum exact.
- Gradients: per point, the rows A_j = d_j - (d_j . n) n (d_j = v_j - v_i) and b_j = I_j - I_i of its neighbourhood plus the
  row (nn - 1) n with b = 0, in float64; the minimum-norm solution of (A^T A) g = A^T b from eigh, eigenvalues <= 1e-12
  times the largest dropped; rounded to float32.  (0, 0, 0) for fewer than 4 neighbours or a zero normal.
- Step: the geometric row sg [p' x n, n], sg (p' - q) . n and the photometric row sp [p' x d, d], sp (I_s - I_0) of every
  pair, relative to the target's box centre; the minimum-norm solution of (J^T J) x = -J^T r as in point-to-plane.
"""
import numpy as np
from scipy.spatial.transform import Rotation

from cwipc_util_b200 import synthetic
from icp_plane_reference import box_centre, estimate_normals, euler_matrix, min_norm_solve, neighbourhoods
from icp_reference import Matcher, Result, evaluate, move, xyz32

CHUNK = 100000        # points solved at a time
GRADIENT_MAX_NN = 30  # the neighbourhood size open3d's RegistrationColoredICP takes for the gradients (radius 2 d)


def intensity(pts):
    """float64 (n,) intensities of a cwipc point record array."""
    return (pts["r"].astype(np.int64) + pts["g"].astype(np.int64) + pts["b"].astype(np.int64)).astype(np.float64) / 765.0


def color_gradients(p32, inten, normals, radius, max_nn, tree=None):
    """(n, 3) float32 colour gradients of the points p32 with intensities `inten` and normals `normals`."""
    p32 = np.ascontiguousarray(p32, np.float32)
    n = len(p32)
    out = np.zeros((n, 3), np.float32)
    if n == 0:
        return out
    nb = neighbourhoods(p32, radius, max_nn, tree)
    v = p32.astype(np.float64)
    for lo in range(0, n, CHUNK):
        sl = slice(lo, lo + CHUNK)
        k = nb[sl]
        have = k >= 0
        nn = have.sum(1)
        nv = np.asarray(normals[sl], np.float64)
        d = np.where(have[..., None], v[np.maximum(k, 0)] - v[sl, None, :], 0.0)
        dn = (d[..., 0] * nv[:, None, 0] + d[..., 1] * nv[:, None, 1]) + d[..., 2] * nv[:, None, 2]
        A = d - dn[..., None] * nv[:, None, :]
        b = np.where(have, inten[np.maximum(k, 0)] - inten[sl, None], 0.0)
        c = (nn - 1)[:, None] * nv
        AtA = np.einsum("nka,nkb->nab", A, A) + c[:, :, None] * c[:, None, :]
        Atb = np.einsum("nka,nk->na", A, b)
        # min_norm_solve, one system per point
        w, V = np.linalg.eigh(AtA)
        keep = w > 1e-12 * w[:, -1:]
        coef = np.where(keep, np.einsum("nak,na->nk", V, Atb) / np.where(keep, w, 1.0), 0.0)
        g = np.einsum("nak,nk->na", V, coef)
        ok = (nn >= 4) & np.any(np.asarray(normals[sl]) != 0, axis=1)
        out[sl] = np.where(ok[:, None], g, 0.0).astype(np.float32)
    return out


def colored_step(p, q, nrm, grad, Is, It, origin, lambda_geometric):
    """dT (4x4) of one colored step over the pairs (p, q) with target normals nrm, target gradients grad, source
    intensities Is and target intensities It, about `origin`."""
    o = np.asarray(origin, np.float64)
    p, q, nrm, grad = np.asarray(p, np.float64) - o, np.asarray(q, np.float64) - o, np.asarray(nrm, np.float64), np.asarray(grad, np.float64)
    sg, sp = np.sqrt(lambda_geometric), np.sqrt(1.0 - lambda_geometric)
    r = np.einsum("na,na->n", p - q, nrm)
    JG = sg * np.concatenate([np.cross(p, nrm), nrm], 1)
    JtJ, Jtr = JG.T @ JG, JG.T @ (sg * r)
    if sp != 0.0:
        proj = (p - q) - r[:, None] * nrm
        i0 = np.einsum("na,na->n", grad, proj) + It
        d = -(grad - np.einsum("na,na->n", grad, nrm)[:, None] * nrm)
        JI = sp * np.concatenate([np.cross(p, d), d], 1)
        JtJ, Jtr = JtJ + JI.T @ JI, Jtr + JI.T @ (sp * (Is - i0))
    x = min_norm_solve(JtJ, -Jtr)
    dT = euler_matrix(x)
    shift, back = np.eye(4), np.eye(4)
    shift[:3, 3], back[:3, 3] = -o, o
    return back @ dT @ shift


def icp_colored(source, target, max_distance, normal_radius, init=None, max_iterations=30, relative_fitness=1e-6, relative_rmse=1e-6, normal_max_nn=30,
                lambda_geometric=0.968, origin=None, normals=None, gradients=None):
    """source, target: cwipc point record arrays (the colours are needed).  origin: the centre of the box the library takes
    for the target (by default the target's own bounding box).  normals, gradients: the target's, (n, 3) float32, when the
    caller has them (by default estimated here)."""
    s32, t32 = xyz32(source), xyz32(target)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    if len(s32) == 0 or len(t32) == 0:
        return Result(T, 0.0, 0.0, 0, 0)
    o = box_centre(t32) if origin is None else np.asarray(origin, np.float64)
    Is, It = intensity(source), intensity(target)
    matcher = Matcher(t32)
    nrm = estimate_normals(t32, normal_radius, normal_max_nn, matcher.tree).normals if normals is None else normals
    grad = color_gradients(t32, It, nrm, 2.0 * max_distance, GRADIENT_MAX_NN, matcher.tree) if gradients is None else gradients
    e = evaluate(s32, matcher, T, max_distance)
    it = 0
    while it < max_iterations and e.correspondences >= 3:
        hit = e.index >= 0
        j = e.index[hit]
        T = colored_step(e.src, e.dst, nrm[j], grad[j], Is[hit], It[j], o, lambda_geometric) @ T
        prev, e = e, evaluate(s32, matcher, T, max_distance)
        it += 1
        if abs(prev.fitness - e.fitness) < relative_fitness and abs(prev.inlier_rmse - e.inlier_rmse) < relative_rmse:
            break
    return Result(T, e.fitness, e.inlier_rmse, it, e.correspondences)


# ---- inputs the tests share -------------------------------------------------------------------------------------------------
RAMP_SPACING = 2.0 ** -6
# the true gradients of these ramps lie at least 0.16 float32 ulps away from a float32 rounding boundary, and both of their
# in-plane components are non-zero (a zero one comes out of the solve as a rounding-sized value, not as 0)
RAMP_COLOURS = ((1, 4), (5, 1), (1, 1))


def ramp(n=40, colour=(1, 4)):
    """An n x n lattice in the plane z = 0 (coordinates exact in float32) whose colour sum grows by colour[0] per step in x
    and colour[1] per step in y: the intensity is linear, with gradient (colour[0], colour[1], 0) / 765 / spacing."""
    g = np.stack(np.meshgrid(np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 2)
    g = g[np.random.default_rng(1).permutation(len(g))]
    pts = np.zeros(len(g), synthetic.cwipc_point_numpy_dtype)
    pts["x"], pts["y"] = (g[:, 0] * RAMP_SPACING).astype(np.float32), (g[:, 1] * RAMP_SPACING).astype(np.float32)
    s = colour[0] * g[:, 0] + colour[1] * g[:, 1]
    pts["r"] = np.minimum(s, 255)
    pts["g"] = np.clip(s - 255, 0, 255)
    pts["b"] = np.clip(s - 510, 0, 255)
    assert np.array_equal(pts["r"].astype(int) + pts["g"] + pts["b"], s)
    return pts, np.array([colour[0], colour[1], 0.0]) / 765.0 / RAMP_SPACING


def revolution_pair(y_degrees):
    """The recovery setup of DESIGN.md §4: the target is synthetic_cloud(40000) with 2 mm of noise; the source is the
    z > 0.05 half of a second noisy sampling, turned by y_degrees about the axis of revolution (y), 1 degree about x and
    shifted by about 1.5 cm.  Returns (source, target, the motion applied to the source)."""
    base = synthetic.synthetic_cloud(40000)
    target = synthetic.add_noise(base, 0.002, seed=1)
    second = synthetic.add_noise(base, 0.002, seed=2)
    half = second[second["z"] > 0.05].copy()
    P = np.eye(4)
    P[:3, :3] = Rotation.from_euler("yx", [y_degrees, 1.0], degrees=True).as_matrix()
    P[:3, 3] = [0.01, -0.005, 0.01]
    moved = move(xyz32(half), P)
    for i, a in enumerate("xyz"):
        half[a] = moved[:, i]
    return half, target, P
