// icp.cpp -- cwipc_cuda_icp, cwipc_cuda_icp_point_to_plane and cwipc_cuda_icp_colored: ICP of one device-resident cloud
// against another, the fine step of multi-camera registration (python/cwipc/registration/: open3d's registration_icp with
// TransformationEstimationPointToPoint or PointToPlane, and registration_colored_icp), with cwipc_cuda_estimate_normals and
// cwipc_cuda_estimate_color_gradients.  The correspondences and their sums come from the target's search index in
// outliers.cu (IcpMatcher); the host solves the motion from those 18 or 30 numbers per iteration and runs the loop.
#include <cmath>
#include <cstring>

#include "kernels.hpp"
#include "pointcloud.hpp"

using namespace cwcu;

namespace {

[[noreturn]] void bad(const std::string &what) { throw CudaError{cudaErrorInvalidValue, what}; }

// Horn's closed-form absolute orientation with unit quaternions (J. Opt. Soc. Am. A 4(4):629-642, 1987): of all rotations,
// the one that maximises sum (R a_i) . b_i over centred pairs (a_i, b_i) is given by the eigenvector of the largest
// eigenvalue of a symmetric 4x4 matrix built from S = sum a_i b_i^T.  The eigenvector is found by cyclic Jacobi rotations
// in double.  The result is always a proper rotation (det +1), also for degenerate (collinear, coincident) pairs.
void horn_rotation(const double S[3][3], double R[3][3]) {
    const double xx = S[0][0], xy = S[0][1], xz = S[0][2], yx = S[1][0], yy = S[1][1], yz = S[1][2], zx = S[2][0], zy = S[2][1], zz = S[2][2];
    double N[4][4] = {{xx + yy + zz, yz - zy, zx - xz, xy - yx},
                      {yz - zy, xx - yy - zz, xy + yx, zx + xz},
                      {zx - xz, xy + yx, -xx + yy - zz, yz + zy},
                      {xy - yx, zx + xz, yz + zy, -xx - yy + zz}};
    double V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
    for (int sweep = 0; sweep < 50; sweep++) {
        double off = 0.0;
        for (int p = 0; p < 4; p++)
            for (int q = p + 1; q < 4; q++) off += N[p][q] * N[p][q];
        if (off == 0.0) break;
        for (int p = 0; p < 4; p++) {
            for (int q = p + 1; q < 4; q++) {
                const double g = 100.0 * std::fabs(N[p][q]);
                if (sweep > 3 && std::fabs(N[p][p]) + g == std::fabs(N[p][p]) && std::fabs(N[q][q]) + g == std::fabs(N[q][q])) {
                    N[p][q] = N[q][p] = 0.0; // below the rounding of both diagonal entries
                    continue;
                }
                if (N[p][q] == 0.0) continue;
                const double theta = (N[q][q] - N[p][p]) / (2.0 * N[p][q]);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 4; k++) { // N <- N P, then P^T N, V <- V P
                    const double a = N[k][p], b = N[k][q];
                    N[k][p] = c * a - s * b;
                    N[k][q] = s * a + c * b;
                }
                for (int k = 0; k < 4; k++) {
                    const double a = N[p][k], b = N[q][k];
                    N[p][k] = c * a - s * b;
                    N[q][k] = s * a + c * b;
                }
                for (int k = 0; k < 4; k++) {
                    const double a = V[k][p], b = V[k][q];
                    V[k][p] = c * a - s * b;
                    V[k][q] = s * a + c * b;
                }
            }
        }
    }
    int best = 0;
    for (int k = 1; k < 4; k++)
        if (N[k][k] > N[best][best]) best = k;
    double w = V[0][best], x = V[1][best], y = V[2][best], z = V[3][best];
    const double norm = std::sqrt(w * w + x * x + y * y + z * z);
    w /= norm, x /= norm, y /= norm, z /= norm;
    R[0][0] = w * w + x * x - y * y - z * z, R[0][1] = 2.0 * (x * y - w * z), R[0][2] = 2.0 * (x * z + w * y);
    R[1][0] = 2.0 * (y * x + w * z), R[1][1] = w * w - x * x + y * y - z * z, R[1][2] = 2.0 * (y * z - w * x);
    R[2][0] = 2.0 * (z * x - w * y), R[2][1] = 2.0 * (z * y + w * x), R[2][2] = w * w - x * x - y * y + z * z;
}

// The rigid motion (row-major 4x4) that minimises sum |R p' + t - q|^2 over the correspondences whose sums (relative to
// `origin`, layout of IcpMatcher::evaluate) are given.  sums[0] >= 3.
void rigid_motion(const double sums[ICP_NSUMS], const double origin[3], double dT[16]) {
    const double n = sums[0];
    const double *sp = sums + 2, *sq = sums + 5;
    double S[3][3], R[3][3];
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) S[a][b] = sums[8 + 3 * a + b] - sp[a] * sq[b] / n; // the cross-covariance of the centred pairs
    horn_rotation(S, R);
    // t = mean q - R mean p', both back in the cloud's own coordinates
    double mp[3], mq[3];
    for (int a = 0; a < 3; a++) {
        mp[a] = sp[a] / n + origin[a];
        mq[a] = sq[a] / n + origin[a];
    }
    memset(dT, 0, 16 * sizeof(double));
    for (int r = 0; r < 3; r++) {
        for (int c = 0; c < 3; c++) dT[4 * r + c] = R[r][c];
        dT[4 * r + 3] = mq[r] - (R[r][0] * mp[0] + R[r][1] * mp[1] + R[r][2] * mp[2]);
    }
    dT[15] = 1.0;
}

// The motion (row-major 4x4) of one point-to-plane step from the sums of IcpMatcher::evaluate (point-to-plane layout,
// relative to `origin`): x = (alpha, beta, gamma, tx, ty, tz) is the minimum-norm least-squares solution of
// (sum J J^T) x = -sum J r, from a cyclic Jacobi eigen-decomposition in double that drops the eigenvalues <= 1e-12 times the
// largest (all of them when the system is zero: x = 0).  dT = [Rz(gamma) Ry(beta) Rx(alpha), t] (open3d's
// TransformVector6dToMatrix4d) about origin, shifted back to the cloud's own coordinates.
void plane_motion(const double sums[ICP_PLANE_NSUMS], const double origin[3], double dT[16]) {
    double A[6][6], V[6][6] = {};
    for (int a = 0, t = 2; a < 6; a++) {
        V[a][a] = 1.0;
        for (int b = a; b < 6; b++, t++) A[a][b] = A[b][a] = sums[t];
    }
    for (int sweep = 0; sweep < 50; sweep++) {
        double off = 0.0;
        for (int p = 0; p < 6; p++)
            for (int q = p + 1; q < 6; q++) off += A[p][q] * A[p][q];
        if (off == 0.0) break;
        for (int p = 0; p < 6; p++) {
            for (int q = p + 1; q < 6; q++) {
                const double g = 100.0 * std::fabs(A[p][q]);
                if (sweep > 3 && std::fabs(A[p][p]) + g == std::fabs(A[p][p]) && std::fabs(A[q][q]) + g == std::fabs(A[q][q])) {
                    A[p][q] = A[q][p] = 0.0; // below the rounding of both diagonal entries
                    continue;
                }
                if (A[p][q] == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 6; k++) { // A <- A P, then P^T A, V <- V P
                    const double a = A[k][p], b = A[k][q];
                    A[k][p] = c * a - s * b;
                    A[k][q] = s * a + c * b;
                }
                for (int k = 0; k < 6; k++) {
                    const double a = A[p][k], b = A[q][k];
                    A[p][k] = c * a - s * b;
                    A[q][k] = s * a + c * b;
                }
                for (int k = 0; k < 6; k++) {
                    const double a = V[k][p], b = V[k][q];
                    V[k][p] = c * a - s * b;
                    V[k][q] = s * a + c * b;
                }
            }
        }
    }
    double top = 0.0;
    for (int i = 0; i < 6; i++) top = std::max(top, A[i][i]);
    double x[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 6; i++) {
        if (!(A[i][i] > 1e-12 * top)) continue;
        double vb = 0.0; // v_i . (-sum J r)
        for (int k = 0; k < 6; k++) vb -= V[k][i] * sums[23 + k];
        for (int k = 0; k < 6; k++) x[k] += V[k][i] * (vb / A[i][i]);
    }
    const double ca = std::cos(x[0]), sa = std::sin(x[0]), cb = std::cos(x[1]), sb = std::sin(x[1]), cg = std::cos(x[2]), sg = std::sin(x[2]);
    const double R[3][3] = {{cg * cb, cg * sb * sa - sg * ca, cg * sb * ca + sg * sa},
                            {sg * cb, sg * sb * sa + cg * ca, sg * sb * ca - cg * sa},
                            {-sb, cb * sa, cb * ca}};
    memset(dT, 0, 16 * sizeof(double));
    for (int r = 0; r < 3; r++) { // p -> R (p - o) + t + o
        for (int c = 0; c < 3; c++) dT[4 * r + c] = R[r][c];
        dT[4 * r + 3] = x[3 + r] + origin[r] - (R[r][0] * origin[0] + R[r][1] * origin[1] + R[r][2] * origin[2]);
    }
    dT[15] = 1.0;
}

void compose(const double a[16], const double b[16], double out[16]) { // out = a * b (row-major 4x4)
    double r[16];
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) r[4 * i + j] = a[4 * i] * b[j] + a[4 * i + 1] * b[4 + j] + a[4 * i + 2] * b[8 + j] + a[4 * i + 3] * b[12 + j];
    memcpy(out, r, sizeof(r));
}

struct Evaluation {
    int32_t correspondences = 0;
    double fitness = 0.0, rmse = 0.0;
};

Evaluation summarize(const double *sums, size_t nsource) {
    Evaluation e;
    e.correspondences = (int32_t)sums[0];
    if (e.correspondences > 0) {
        e.fitness = sums[0] / (double)nsource;
        e.rmse = std::sqrt(sums[1] / sums[0]);
    }
    return e;
}

void check_normal_args(double radius, int max_nn) {
    if (!(std::isfinite(radius) && radius > 0.0)) bad("the normal radius must be finite and > 0");
    if (max_nn < 3 || max_nn > ICP_MAX_NN) bad("the normal max_nn must be in [3, " + std::to_string(ICP_MAX_NN) + "]");
}

void check_gradient_args(double radius, int max_nn) {
    if (!(std::isfinite(radius) && radius > 0.0)) bad("the gradient radius must be finite and > 0");
    if (max_nn < 4 || max_nn > ICP_MAX_NN) bad("the gradient max_nn must be in [4, " + std::to_string(ICP_MAX_NN) + "]");
}

struct PlaneOptions {
    double normal_radius;
    int normal_max_nn;
    bool colored;            // colored ICP: also the target's colour gradients and the photometric rows
    double lambda_geometric; // colored only
};

// The loop of open3d's RegistrationICP, shared by the three entry points: point-to-point when plane is null, else
// point-to-plane with the target's normals, or colored ICP with its normals and colour gradients.  The estimation's solve
// is the one difference between point-to-point and the other two, which share plane_motion.
int icp_entry(const char *who, cwipc_pointcloud *source, cwipc_pointcloud *target, const double init[16], double max_correspondence_distance, int max_iterations,
              double relative_fitness, double relative_rmse, const PlaneOptions *plane, struct cwipc_cuda_icp_result *result) {
    if (target == nullptr) return -1;
    return read_entry<int>(who, source, -1, [&](const StoragePtr &src, int dev, cudaStream_t s) -> int {
        if (!(std::isfinite(max_correspondence_distance) && max_correspondence_distance > 0.0)) bad("max_correspondence_distance must be finite and > 0");
        if (max_iterations < 0) bad("max_iterations must be >= 0");
        if (!(std::isfinite(relative_fitness) && relative_fitness >= 0.0 && std::isfinite(relative_rmse) && relative_rmse >= 0.0))
            bad("relative_fitness and relative_rmse must be finite and >= 0");
        if (plane) check_normal_args(plane->normal_radius, plane->normal_max_nn);
        if (plane && plane->colored && !(std::isfinite(plane->lambda_geometric) && plane->lambda_geometric >= 0.0 && plane->lambda_geometric <= 1.0))
            bad("lambda_geometric must be finite and in [0, 1]");
        double T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
        if (init) {
            for (int k = 0; k < 16; k++)
                if (!std::isfinite(init[k])) bad("init has a non-finite entry");
            if (!(init[12] == 0.0 && init[13] == 0.0 && init[14] == 0.0 && init[15] == 1.0)) bad("the last row of init is not (0, 0, 0, 1)");
            memcpy(T, init, sizeof(T));
        }
        if (result == nullptr) bad("result must not be NULL");
        StoragePtr tgt = storage_of(target, who);
        if (!tgt) return -1;
        if (tgt->dev != dev) bad("source and target live on different devices (" + std::to_string(dev) + " and " + std::to_string(tgt->dev) + ")");
        ReadLease lease_t(*tgt, s);

        Evaluation e;
        int iterations = 0;
        const size_t ns = src->count;
        if (ns > 0 && tgt->count > 0) {
            float box[6];
            if (tgt->has_bounds) {
                memcpy(box, tgt->bounds_min, 3 * sizeof(float));
                memcpy(box + 3, tgt->bounds_max, 3 * sizeof(float));
            }
            const float *bounds = tgt->has_bounds ? box : nullptr;
            // colored: open3d's RegistrationColoredICP takes the gradients of the 30 nearest points within 2 d
            IcpMatcher matcher = !plane ? IcpMatcher(tgt->d_pts, tgt->count, target->cellsize(), bounds, dev, s)
                                 : !plane->colored ? IcpMatcher(tgt->d_pts, tgt->count, target->cellsize(), bounds, dev, s, plane->normal_radius, plane->normal_max_nn)
                                                   : IcpMatcher(tgt->d_pts, tgt->count, target->cellsize(), bounds, dev, s, plane->normal_radius, plane->normal_max_nn,
                                                                2.0 * max_correspondence_distance, 30, plane->lambda_geometric);
            const float limit = (float)(max_correspondence_distance * max_correspondence_distance);
            double sums[ICP_PLANE_NSUMS];
            matcher.evaluate(src->d_pts, ns, T, limit, true, sums);
            if (sums[matcher.nsums() - 1] != 0.0) bad("the source or the target contains non-finite coordinates");
            e = summarize(sums, ns);
            while (iterations < max_iterations && e.correspondences >= 3) {
                double dT[16];
                if (plane) plane_motion(sums, matcher.origin(), dT);
                else rigid_motion(sums, matcher.origin(), dT);
                compose(dT, T, T);
                // the composed motion is applied to the original points (open3d moves its moved copy again: its rounding adds up)
                matcher.evaluate(src->d_pts, ns, T, limit, false, sums);
                const Evaluation prev = e;
                e = summarize(sums, ns);
                iterations++;
                if (std::fabs(prev.fitness - e.fitness) < relative_fitness && std::fabs(prev.rmse - e.rmse) < relative_rmse) break;
            }
        }
        memcpy(result->matrix, T, sizeof(T));
        result->fitness = e.fitness;
        result->inlier_rmse = e.rmse;
        result->iterations = iterations;
        result->correspondences = e.correspondences;
        return 0;
    });
}

} // namespace

extern "C" {

// The loop of open3d's RegistrationICP with point-to-point estimation (see include/cwipc_util_cuda.h for every rule).
int cwipc_cuda_icp(cwipc_pointcloud *source, cwipc_pointcloud *target, const double init[16], double max_correspondence_distance, int max_iterations,
                   double relative_fitness, double relative_rmse, struct cwipc_cuda_icp_result *result) {
    return icp_entry("cwipc_cuda_icp", source, target, init, max_correspondence_distance, max_iterations, relative_fitness, relative_rmse, nullptr, result);
}

// The same loop with point-to-plane estimation against the target's normals (see include/cwipc_util_cuda.h).
int cwipc_cuda_icp_point_to_plane(cwipc_pointcloud *source, cwipc_pointcloud *target, const double init[16], double max_correspondence_distance, int max_iterations,
                                  double relative_fitness, double relative_rmse, double normal_radius, int normal_max_nn, struct cwipc_cuda_icp_result *result) {
    const PlaneOptions plane{normal_radius, normal_max_nn, false, 1.0};
    return icp_entry("cwipc_cuda_icp_point_to_plane", source, target, init, max_correspondence_distance, max_iterations, relative_fitness, relative_rmse, &plane, result);
}

// The same loop with colored ICP's estimation against the target's normals and colour gradients (see include/cwipc_util_cuda.h).
int cwipc_cuda_icp_colored(cwipc_pointcloud *source, cwipc_pointcloud *target, const double init[16], double max_correspondence_distance, int max_iterations,
                           double relative_fitness, double relative_rmse, double normal_radius, int normal_max_nn, double lambda_geometric,
                           struct cwipc_cuda_icp_result *result) {
    const PlaneOptions colored{normal_radius, normal_max_nn, true, lambda_geometric};
    return icp_entry("cwipc_cuda_icp_colored", source, target, init, max_correspondence_distance, max_iterations, relative_fitness, relative_rmse, &colored, result);
}

int cwipc_cuda_estimate_color_gradients(cwipc_pointcloud *pc, double normal_radius, int normal_max_nn, double radius, int max_nn, float *gradients, size_t nfloats) {
    return read_entry<int>("cwipc_cuda_estimate_color_gradients", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        check_normal_args(normal_radius, normal_max_nn);
        check_gradient_args(radius, max_nn);
        if (gradients == nullptr) bad("gradients must not be NULL");
        if (nfloats < 3 * in->count) bad("gradients holds " + std::to_string(nfloats) + " floats, " + std::to_string(3 * in->count) + " are needed");
        if (in->count == 0) return 0;
        float box[6];
        if (in->has_bounds) {
            memcpy(box, in->bounds_min, 3 * sizeof(float));
            memcpy(box + 3, in->bounds_max, 3 * sizeof(float));
        }
        // (the weight only matters to evaluate, which the hook does not call)
        IcpMatcher matcher(in->d_pts, in->count, pc->cellsize(), in->has_bounds ? box : nullptr, dev, s, normal_radius, normal_max_nn, radius, max_nn, 1.0);
        if (!matcher.gradients_to_host(gradients)) bad("the cloud contains non-finite coordinates");
        return (int)in->count;
    });
}

int cwipc_cuda_estimate_normals(cwipc_pointcloud *pc, double radius, int max_nn, float *normals, size_t nfloats) {
    return read_entry<int>("cwipc_cuda_estimate_normals", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        check_normal_args(radius, max_nn);
        if (normals == nullptr) bad("normals must not be NULL");
        if (nfloats < 3 * in->count) bad("normals holds " + std::to_string(nfloats) + " floats, " + std::to_string(3 * in->count) + " are needed");
        if (in->count == 0) return 0;
        float box[6];
        if (in->has_bounds) {
            memcpy(box, in->bounds_min, 3 * sizeof(float));
            memcpy(box + 3, in->bounds_max, 3 * sizeof(float));
        }
        IcpMatcher matcher(in->d_pts, in->count, pc->cellsize(), in->has_bounds ? box : nullptr, dev, s, radius, max_nn);
        if (!matcher.normals_to_host(normals)) bad("the cloud contains non-finite coordinates");
        return (int)in->count;
    });
}

} // extern "C"
