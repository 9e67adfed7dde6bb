// backward.cuh — gradient of rtgs_render with respect to the stored Gaussian parameters (sm_100a).
//
// The image is differentiated with the per-pixel layer list held fixed: membership, order and the q = 3
// silhouette are piecewise constant and have no gradient.  One thread per pixel, one warp per 4x8-pixel tile
// (the rays of a warp stay coherent), three phases per thread:
//   1. the `depth` nearest hits: LBVH walk over `nodes` with the inflated float32 slabs of k_trace_closest, a sorted
//      k-buffer of (float64 t1, sorted position), boxes beyond the current K-th t1 pruned once it is full; every
//      hit / miss and t1 is the float64 exact_intersect from `raw` (t1 > 0), exact ties broken by sorted position
//      (exact_less) - the oracle's decisions;
//   2. the forward again: q, alpha in float64 from `raw`, colour + SH from the packed records, the t_cut rule of
//      the forward (composite layer k while the float32 transmittance T_k >= t_cut); T_k kept per layer;
//   3. back to front, with B_n = dL/dT and B_k = alpha_k (c_k.g) + (1 - alpha_k) B_{k+1} (no division):
//        dL/dalpha_k = T_k (c_k.g - B_{k+1}),  dL/dc_k = T_k alpha_k g,
//        alpha = opacity exp(-q):  dL/dopacity = exp(-q) dL/dalpha,  dL/dq = -alpha dL/dalpha,
//        c = colour + sum_j Y_j sh_j (the direction's gradient only with CAM, below),
//        u = W (o - p), v = W d, sigma = u.v / |v|^2, e = u - sigma v = W (x - p), x = o - sigma d:
//        dq/dp = -2 W^T e,  dq/dW = 2 e (x - p)^T,
//        W = S^-1 Rm^T / c^2 (local_frame as written, Rm = quat_to_mat(q), c = |q|^2): differentiated through
//        s, Rm(q) and c, so stored quaternions of any norm get their exact gradient.
//      Gradients are scattered with float32 atomics to the ORIGINAL index (raw[s*3+2].z).
// k_render_backward<true> also differentiates with respect to the camera (rtgs_render_backward_camera).  The camera
// enters only through the ray: o, d = Rm(q_cam) dc, dc = n / |n|, n = (px, py, -1), px = (i + 0.5 - W/2) / fx.
// Per layer dq/do = 2 W^T e, dq/dd = -2 sigma W^T e; the SH colour adds dL/dY_j = sum_k T_k alpha_k (sh_kj . g),
// summed over the layers and taken through dY/d(d/|d|) once per pixel.  Per pixel, from dL/dd:
// dL/dRm = dL/dd dc^T, dL/dn = (I - dc dc^T) Rm^T dL/dd / |n|, dL/dfx = -dL/dpx px / fx (fy alike).  The 14 per-pixel
// values (o 3, Rm 9, fx, fy) are summed in float64 in a fixed order: warp shuffles, the CTA's warps in shared
// memory, one partial record per CTA, and k_camera_grad_finalize (one CTA) over the partials, which also takes
// dL/dRm to dL/dq_cam and adds the float32-rounded results to the caller's buffers.
//
// The three phases take the ray (o, d) as a parameter (walk_layers, replay_layers, back_to_front), so they also serve
// arbitrary rays (rtgs_render_rays / _backward): k_render_rays runs phases 1-2, k_render_rays_backward 1-3, one thread
// per ray.  A ray is the (n,8) float32 record of rtgs_generate_rays: o, d (used as given, not normalised; the SH
// colour uses d / |d|), start, end.  Its layer list is the Gaussians with start < t1 < end (float64 exact_intersect),
// ascending t1, ties by sorted position, truncated to `depth`, composited under the t_cut rule; start = 0, end = +inf
// is the pixel rule.  Its gradient is dL/do = sum_k 2 dq_k W^T e, dL/dd = sum_k -2 sigma dq_k W^T e plus the SH term
// (I - dn dn^T)(dY/ddn)^T dL/dY / |d|: the gO / gD of the CAM path.  A ray with a non-finite o or d component, d = 0
// or !(start < end) composites nothing (rgb 0, T 1) and gets no gradient.
#pragma once
#include "render_common.cuh"

namespace rtgs_dev {
namespace backward {

constexpr int BWD_WARPS = 4;   // warps (tiles) per CTA
constexpr int CAM_TERMS = 14;  // per-pixel camera gradient: dL/do (3), dL/dRm (9, row-major), dL/dfx, dL/dfy
constexpr int FIN_THREADS = 256;

struct BackwardParams {
    const float4* __restrict__ nodes;
    const float4* __restrict__ geo;
    const float4* __restrict__ shp;
    const float4* __restrict__ raw;
    CamD cam;
    int x0, y0, w, h;
    int tiles_j;                 // tiles per region column (ceil(h / TILE_J))
    int ntiles;
    int depth;
    float t_cut;
    int has_sh;
    const float* dL_drgb;        // (w,h,3) i-major region buffer
    const float* dL_dT;          // (w,h) or null
    float* g_pos;                // (n,3), original order, any may be null
    float* g_rot;                // (n,4)
    float* g_scale;              // (n,3)
    float* g_color;              // (n,3)
    float* g_opacity;            // (n)
    float* g_sh;                 // (n,15,3)
    float* replay_rgb;           // (w,h,3) or null
    float* replay_T;             // (w,h) or null
    double* cam_part;            // k_render_backward<true>: (CAM_TERMS, gridDim.x) per-CTA partial sums
    // the ray kernels: dL_drgb, dL_dT, replay_rgb and replay_T are then indexed by ray
    const float* rays;           // (nrays, 8): o xyz, d xyz, start, end; 16-byte aligned
    int64_t nrays;
    float* g_rays;               // k_render_rays_backward<true>: (nrays, 8), columns 0-5 accumulated
    // DEPTH instantiations (DESIGN.md §12): D = sum_k T_k alpha_k t*_k, t*_k = -sigma_k; indexed like dL_dT / replay_T
    const float* dL_dD;          // or null (no depth gradient)
    float* replay_depth;         // or null
};

// sh_basis (render_common.cuh) in float64: gaussian.py:149-163, incl. the `5z^2 - 3z` term at :160 as coded
__device__ __forceinline__ void sh_basis_d(double x, double y, double z, double (&Y)[15]) {
    const double c0 = 0.9772050238058398, c1 = 2.1850968611841584, c2 = 1.2615662610100802,
                 c3 = 2.360174359706574, c4 = 5.781222885281108, c5 = 1.828183197857863, c6 = 1.4927053303604616;
    const double xx = x * x, yy = y * y, zz = z * z;
    Y[0] = 0.5 * c0 * y;
    Y[1] = 0.5 * c0 * z;
    Y[2] = 0.5 * c0 * x;
    Y[3] = 0.5 * c1 * x * y;
    Y[4] = 0.5 * c1 * y * z;
    Y[5] = 0.25 * c2 * (3.0 * zz - 1.0);
    Y[6] = 0.5 * c1 * x * z;
    Y[7] = 0.25 * c1 * (xx - yy);
    Y[8] = 0.25 * c3 * y * (3.0 * xx - yy);
    Y[9] = 0.5 * c4 * x * y * z;
    Y[10] = 0.25 * c5 * y * (5.0 * zz - 1.0);
    Y[11] = 0.25 * c6 * (5.0 * zz - 3.0 * z);
    Y[12] = 0.25 * c5 * x * (5.0 * zz - 1.0);
    Y[13] = 0.25 * c4 * (xx - yy) * z;
    Y[14] = 0.25 * c3 * x * (xx - 3.0 * yy);
}

// g = sum_j gY[j] dY_j/d(x, y, z): the derivative of sh_basis_d at (x, y, z), contracted with gY
__device__ __forceinline__ void sh_basis_vjp_d(double x, double y, double z, const double (&gY)[15], double (&g)[3]) {
    const double c0 = 0.9772050238058398, c1 = 2.1850968611841584, c2 = 1.2615662610100802,
                 c3 = 2.360174359706574, c4 = 5.781222885281108, c5 = 1.828183197857863, c6 = 1.4927053303604616;
    const double xx = x * x, yy = y * y, zz = z * z;
    g[0] = 0.5 * c0 * gY[2] + 0.5 * c1 * (y * gY[3] + z * gY[6] + x * gY[7]) + 1.5 * c3 * x * y * gY[8] +
           0.5 * c4 * y * z * gY[9] + 0.25 * c5 * (5.0 * zz - 1.0) * gY[12] + 0.5 * c4 * x * z * gY[13] +
           0.75 * c3 * (xx - yy) * gY[14];
    g[1] = 0.5 * c0 * gY[0] + 0.5 * c1 * (x * gY[3] + z * gY[4] - y * gY[7]) + 0.75 * c3 * (xx - yy) * gY[8] +
           0.5 * c4 * x * z * gY[9] + 0.25 * c5 * (5.0 * zz - 1.0) * gY[10] - 0.5 * c4 * y * z * gY[13] -
           1.5 * c3 * x * y * gY[14];
    g[2] = 0.5 * c0 * gY[1] + 0.5 * c1 * (y * gY[4] + x * gY[6]) + 1.5 * c2 * z * gY[5] + 0.5 * c4 * x * y * gY[9] +
           2.5 * c5 * y * z * gY[10] + 0.25 * c6 * (10.0 * z - 3.0) * gY[11] + 2.5 * c5 * x * z * gY[12] +
           0.25 * c4 * (xx - yy) * gY[13];
}

// The part of dL/dq that goes through Rm = quat_to_mat(q) = (w^2 - |u|^2) I + 2 u u^T + 2 w [u]x (quat_rot on the
// basis vectors), given M = dL/dRm.  Shared by the Gaussian rotations and the camera rotation.
__device__ __forceinline__ void rot_mat_vjp(const double (&q)[4], const double (&M)[3][3], double (&g)[4]) {
    const double ux = q[0], uy = q[1], uz = q[2], w = q[3];
    const double tr = M[0][0] + M[1][1] + M[2][2];
    const double Kx = M[2][1] - M[1][2], Ky = M[0][2] - M[2][0], Kz = M[1][0] - M[0][1];
    const double u3[3] = {ux, uy, uz}, K3[3] = {Kx, Ky, Kz};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double Mu = M[i][0] * ux + M[i][1] * uy + M[i][2] * uz;
        const double MTu = M[0][i] * ux + M[1][i] * uy + M[2][i] * uz;
        g[i] = -2.0 * u3[i] * tr + 2.0 * (Mu + MTu) + 2.0 * w * K3[i];
    }
    g[3] = 2.0 * w * tr + 2.0 * (ux * Kx + uy * Ky + uz * Kz);
}

// One layer of one ray, float64 from the raw parameters: everything phases 2 and 3 need.
struct Layer {
    double p[3], q[4], sc[3];
    double Wm[3][3];
    double e[3];      // W (x - p)
    double xp[3];     // x - p, x = o - sigma d: the max-response point
    double sig;       // sigma = u.v / |v|^2
    double v[3];      // W d
    double A;         // |v|^2
    double qm;        // |e|^2 = min Mahalanobis^2 along the ray
    double alpha;
    double ex;        // exp(-q)
    int g;            // original index
};

__device__ __forceinline__ void eval_layer(const BackwardParams& P, int s, const double (&o)[3], const d3& d,
                                           Layer& L) {
    const float4 ra = __ldg(P.raw + (int64_t)s * 3 + 0), rb = __ldg(P.raw + (int64_t)s * 3 + 1),
                 rc = __ldg(P.raw + (int64_t)s * 3 + 2);
    L.p[0] = ra.x; L.p[1] = ra.y; L.p[2] = ra.z;
    L.q[0] = ra.w; L.q[1] = rb.x; L.q[2] = rb.y; L.q[3] = rb.z;
    L.sc[0] = rb.w; L.sc[1] = rc.x; L.sc[2] = rc.y;
    L.g = __float_as_int(rc.z);
    local_frame(L.q, L.sc, L.Wm);
    const double op[3] = {o[0] - L.p[0], o[1] - L.p[1], o[2] - L.p[2]};
    double u[3], v[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        u[k] = L.Wm[k][0] * op[0] + L.Wm[k][1] * op[1] + L.Wm[k][2] * op[2];
        v[k] = L.Wm[k][0] * d.x + L.Wm[k][1] * d.y + L.Wm[k][2] * d.z;
    }
    const double A = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    const double sig = (u[0] * v[0] + u[1] * v[1] + u[2] * v[2]) / A;
    const d3 m = d3cross(d3make(u[0], u[1], u[2]), d3make(v[0], v[1], v[2]));
    L.qm = d3dot(m, m) / A;   // as exact_intersect computes it
#pragma unroll
    for (int k = 0; k < 3; ++k) L.e[k] = u[k] - sig * v[k];
    L.sig = sig;
#pragma unroll
    for (int k = 0; k < 3; ++k) L.v[k] = v[k];
    L.A = A;
    L.xp[0] = op[0] - sig * d.x;
    L.xp[1] = op[1] - sig * d.y;
    L.xp[2] = op[2] - sig * d.z;
    L.ex = exp(-L.qm);
    L.alpha = (double)__ldg(P.geo + (int64_t)s * 4).w * L.ex;
}

// rgb = colour + sum_j Y_j sh_j from the packed record of sorted position s (eval_colour's data, float64 sum)
__device__ __forceinline__ void eval_colour_d(const BackwardParams& P, int s, const double (&Y)[15], double (&c)[3]) {
    if (P.has_sh) {
        const float4* sp = P.shp + (int64_t)s * 12;
        float v[48];
#pragma unroll
        for (int f = 0; f < 12; ++f) {
            const float4 x = __ldg(sp + f);
            v[4 * f] = x.x; v[4 * f + 1] = x.y; v[4 * f + 2] = x.z; v[4 * f + 3] = x.w;
        }
        c[0] = v[45]; c[1] = v[46]; c[2] = v[47];
#pragma unroll
        for (int j = 0; j < 15; ++j) {
            c[0] += Y[j] * v[3 * j + 0];
            c[1] += Y[j] * v[3 * j + 1];
            c[2] += Y[j] * v[3 * j + 2];
        }
    } else {
        const float4 g3 = __ldg(P.geo + (int64_t)s * 4 + 3);
        c[0] = g3.y; c[1] = g3.z; c[2] = g3.w;
    }
}

// gY[j] += wgt * (sh_j . gr) for the SH coefficients of sorted position s (the colour's dependence on Y)
__device__ __forceinline__ void sh_dot_d(const BackwardParams& P, int s, double wgt, const double (&gr)[3],
                                         double (&gY)[15]) {
    const float4* sp = P.shp + (int64_t)s * 12;
    float v[48];
#pragma unroll
    for (int f = 0; f < 12; ++f) {
        const float4 x = __ldg(sp + f);
        v[4 * f] = x.x; v[4 * f + 1] = x.y; v[4 * f + 2] = x.z; v[4 * f + 3] = x.w;
    }
#pragma unroll
    for (int j = 0; j < 15; ++j) gY[j] += wgt * (v[3 * j + 0] * gr[0] + v[3 * j + 1] * gr[1] + v[3 * j + 2] * gr[2]);
}

__device__ __forceinline__ void red_add(float* base, int64_t i, double v) {
    if (base != nullptr) atomicAdd(base + i, (float)v);
}

// ---- the three phases of one ray (o, d): shared by the pixel kernels and the ray kernels -----------------------

// Phase 1: the K nearest hits, ascending float64 t1, ties by sorted position, into kt / ks; returns their count.
// INTERVAL = false is the pixel rule t1 > 0; INTERVAL = true keeps t_start < t1 < t_end and also prunes boxes entered
// beyond t_end (the box holds its Gaussians' ellipsoids, so none of them has a t1 before the box's entry).
template <bool INTERVAL>
__device__ __forceinline__ int walk_layers(const BackwardParams& P, const double (&o)[3], const d3& d, double t_start,
                                           double t_end, double (&kt)[RTGS_MAX_DEPTH], int (&ks)[RTGS_MAX_DEPTH]) {
    const int K = P.depth;
    int cnt = 0;
    const float of[3] = {(float)o[0], (float)o[1], (float)o[2]};
    const float idf[3] = {1.0f / (float)d.x, 1.0f / (float)d.y, 1.0f / (float)d.z};
    auto slab = [&](float mnx, float mny, float mnz, float mxx, float mxy, float mxz) -> float {
        return slab_entry(of, idf, {mnx, mny, mnz}, {mxx, mxy, mxz});
    };
    int stack[RTGS_MAX_TREE_DEPTH + 2];
    int sp = 0;
    stack[sp++] = 0;
    while (sp > 0) {
        const int node = stack[--sp];
        const float4 a = __ldg(P.nodes + (int64_t)node * 4 + 0), b = __ldg(P.nodes + (int64_t)node * 4 + 1),
                     c = __ldg(P.nodes + (int64_t)node * 4 + 2), dd = __ldg(P.nodes + (int64_t)node * 4 + 3);
        const int ch[2] = {__float_as_int(dd.x), __float_as_int(dd.y)};
        // The root of a single-Gaussian tree has an empty right child (half extent -inf, reference ~0 = leaf 0
        // again): the slabs of an inverted box span every t, so it is skipped here, or leaf 0 would enter the
        // k-buffer twice.  (A closest-hit walk can afford the duplicate; a list of layers cannot.)
        const float te[2] = {a.w >= 0.0f ? slab(a.x - a.w, a.y - b.x, a.z - b.y, a.x + a.w, a.y + b.x, a.z + b.y)
                                         : INFINITY,
                             c.y >= 0.0f ? slab(b.z - c.y, b.w - c.z, c.x - c.w, b.z + c.y, b.w + c.z, c.x + c.w)
                                         : INFINITY};
        const int first = te[0] <= te[1] ? 0 : 1;
        for (int k = 1; k >= 0; --k) {
            const int w = k == 0 ? first : 1 - first;
            if (!(te[w] < INFINITY) || (cnt == K && (double)te[w] > kt[K - 1])) continue;
            if (INTERVAL && (double)te[w] > t_end) continue;
            if (ch[w] >= 0) {
                stack[sp++] = ch[w];
                continue;
            }
            const int s = ~ch[w];
            const float4 ra = __ldg(P.raw + (int64_t)s * 3 + 0), rb = __ldg(P.raw + (int64_t)s * 3 + 1),
                         rc = __ldg(P.raw + (int64_t)s * 3 + 2);
            const double p[3] = {ra.x, ra.y, ra.z}, q[4] = {ra.w, rb.x, rb.y, rb.z}, sc[3] = {rb.w, rc.x, rc.y};
            const ExactHit e = exact_intersect(p, q, sc, o, d);
            if (!(e.hit && (INTERVAL ? (e.t1 > t_start && e.t1 < t_end) : e.t1 > 0.0))) continue;
            const double t = e.t1;
            if (cnt == K && !(t < kt[K - 1] || (t == kt[K - 1] && s < ks[K - 1]))) continue;
            int at = cnt < K ? cnt++ : K - 1;
            while (at > 0 && (t < kt[at - 1] || (t == kt[at - 1] && s < ks[at - 1]))) {
                kt[at] = kt[at - 1];
                ks[at] = ks[at - 1];
                --at;
            }
            kt[at] = t;
            ks[at] = s;
        }
    }
    return cnt;
}

// Phase 2: the forward again over the cnt layers; kt[k] becomes T_k, Y the SH basis of d / |d|.  The image goes to
// replay_rgb / replay_T[out] (each may be null), with DEPTH the composited t* = -sigma to replay_depth[out]; returns
// the number of layers composited under the t_cut rule.
template <bool DEPTH = false>
__device__ __forceinline__ int replay_layers(const BackwardParams& P, const double (&o)[3], const d3& d, int cnt,
                                             double (&kt)[RTGS_MAX_DEPTH], const int (&ks)[RTGS_MAX_DEPTH],
                                             int64_t out, double (&Y)[15]) {
    {
        const double il = 1.0 / sqrt(d.x * d.x + d.y * d.y + d.z * d.z);
        sh_basis_d(d.x * il, d.y * il, d.z * il, Y);
    }
    double T = 1.0, rgb[3] = {0.0, 0.0, 0.0}, D = 0.0;
    float Tf = 1.0f;   // the forward's float32 transmittance decides the t_cut rule
    int L = 0;
    for (int k = 0; k < cnt; ++k) {
        if (!(Tf >= P.t_cut)) break;
        Layer ly;
        eval_layer(P, ks[k], o, d, ly);
        double c[3];
        eval_colour_d(P, ks[k], Y, c);
        kt[k] = T;
        const double wgt = T * ly.alpha;
        rgb[0] += wgt * c[0];
        rgb[1] += wgt * c[1];
        rgb[2] += wgt * c[2];
        if constexpr (DEPTH) D -= wgt * ly.sig;
        T *= 1.0 - ly.alpha;
        Tf *= 1.0f - (float)ly.alpha;
        L = k + 1;
    }
    if (P.replay_rgb != nullptr) {
        P.replay_rgb[out * 3 + 0] = (float)rgb[0];
        P.replay_rgb[out * 3 + 1] = (float)rgb[1];
        P.replay_rgb[out * 3 + 2] = (float)rgb[2];
    }
    if (P.replay_T != nullptr) P.replay_T[out] = (float)T;
    if (DEPTH && P.replay_depth != nullptr) P.replay_depth[out] = (float)D;
    return L;
}

// Phase 3: back to front over the L composited layers (T_k in kt) from dL/drgb = gr and B = dL/dT, scattering the
// Gaussian gradients.  RAY_GRAD also returns the ray's own gradient: gO = dL/do, gD = dL/dd including the SH colour's
// dependence on d / |d| (gO, gD enter as zeros).  DEPTH adds dL/dD = gDep: t*_k enters like one more colour channel,
// and through t* = -sigma, dL/dsigma_k = -T_k alpha_k gDep with dsigma/du = v / A, dsigma/dv = (e - sigma v) / A.
template <bool RAY_GRAD, bool DEPTH = false>
__device__ __forceinline__ void back_to_front(const BackwardParams& P, const double (&o)[3], const d3& d, int L,
                                              const double (&kt)[RTGS_MAX_DEPTH], const int (&ks)[RTGS_MAX_DEPTH],
                                              const double (&Y)[15], const double (&gr)[3], double B,
                                              double (&gO)[3], double (&gD)[3], double gDep = 0.0) {
    double gY[15];   // RAY_GRAD: dL/dY_j
    if constexpr (RAY_GRAD) {
#pragma unroll
        for (int j = 0; j < 15; ++j) gY[j] = 0.0;
    }
    for (int k = L - 1; k >= 0; --k) {
        const int s = ks[k];
        Layer ly;
        eval_layer(P, s, o, d, ly);
        double c[3];
        eval_colour_d(P, s, Y, c);
        const double Tk = kt[k], a = ly.alpha;
        double cg = c[0] * gr[0] + c[1] * gr[1] + c[2] * gr[2];
        if constexpr (DEPTH) cg -= ly.sig * gDep;
        const double dA = Tk * (cg - B);
        B = a * cg + (1.0 - a) * B;
        const double wgt = Tk * a;
        const int64_t g = ly.g;
        // colour and SH
        if (P.g_color != nullptr || P.g_sh != nullptr) {
            const double dc[3] = {wgt * gr[0], wgt * gr[1], wgt * gr[2]};
            red_add(P.g_color, g * 3 + 0, dc[0]);
            red_add(P.g_color, g * 3 + 1, dc[1]);
            red_add(P.g_color, g * 3 + 2, dc[2]);
            if (P.g_sh != nullptr) {
#pragma unroll
                for (int j = 0; j < 15; ++j) {
                    red_add(P.g_sh, g * 45 + j * 3 + 0, Y[j] * dc[0]);
                    red_add(P.g_sh, g * 45 + j * 3 + 1, Y[j] * dc[1]);
                    red_add(P.g_sh, g * 45 + j * 3 + 2, Y[j] * dc[2]);
                }
            }
        }
        red_add(P.g_opacity, g, ly.ex * dA);
        const double dq = -a * dA;
        // DEPTH: hu = dL/du = dL/dsigma v / A, hv = dL/dv = dL/dsigma (e - sigma v) / A
        double hu[3], hv[3];
        if constexpr (DEPTH) {
            const double ds = -wgt * gDep / ly.A;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                hu[i] = ds * ly.v[i];
                hv[i] = ds * (ly.e[i] - ly.sig * ly.v[i]);
            }
        }
        if (P.g_pos != nullptr) {
            // dq/dp = -2 W^T e;  du/dp = -W
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                double gp = -2.0 * dq * (ly.Wm[0][j] * ly.e[0] + ly.Wm[1][j] * ly.e[1] + ly.Wm[2][j] * ly.e[2]);
                if constexpr (DEPTH) gp -= ly.Wm[0][j] * hu[0] + ly.Wm[1][j] * hu[1] + ly.Wm[2][j] * hu[2];
                red_add(P.g_pos, g * 3 + j, gp);
            }
        }
        if constexpr (RAY_GRAD) {
            // dq/do = 2 W^T e, dq/dd = -2 sigma W^T e;  du/do = W, dv/dd = W
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double wte = 2.0 * dq * (ly.Wm[0][j] * ly.e[0] + ly.Wm[1][j] * ly.e[1] + ly.Wm[2][j] * ly.e[2]);
                gO[j] += wte;
                gD[j] -= ly.sig * wte;
                if constexpr (DEPTH) {
                    gO[j] += ly.Wm[0][j] * hu[0] + ly.Wm[1][j] * hu[1] + ly.Wm[2][j] * hu[2];
                    gD[j] += ly.Wm[0][j] * hv[0] + ly.Wm[1][j] * hv[1] + ly.Wm[2][j] * hv[2];
                }
            }
            if (P.has_sh) sh_dot_d(P, s, wgt, gr, gY);
        }
        if (P.g_scale == nullptr && P.g_rot == nullptr) continue;
        // G = dL/dW = 2 dq e (x - p)^T (DEPTH: + hu (o - p)^T + hv d^T); W_kj = Rm[j][k] f_k with f_k = 1 / (s_k c^2)
        double GW[3];   // sum_j G_kj W_kj per row k
        double M[3][3]; // dL/dRm
        const double c2 = ly.q[0] * ly.q[0] + ly.q[1] * ly.q[1] + ly.q[2] * ly.q[2] + ly.q[3] * ly.q[3];
#pragma unroll
        for (int k2 = 0; k2 < 3; ++k2) {
            const double f = 1.0 / (ly.sc[k2] * c2 * c2);
            GW[k2] = 0.0;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                double G = 2.0 * dq * ly.e[k2] * ly.xp[j];
                if constexpr (DEPTH) G += hu[k2] * (o[j] - ly.p[j]) + hv[k2] * (j == 0 ? d.x : j == 1 ? d.y : d.z);
                GW[k2] += G * ly.Wm[k2][j];
                M[j][k2] = G * f;
            }
        }
        if (P.g_scale != nullptr) {
#pragma unroll
            for (int k2 = 0; k2 < 3; ++k2) red_add(P.g_scale, g * 3 + k2, -GW[k2] / ly.sc[k2]);
        }
        if (P.g_rot != nullptr) {
            // through Rm(q) (rot_mat_vjp) and through c = |q|^2
            double gq[4];
            rot_mat_vjp(ly.q, M, gq);
            const double dLdc = -2.0 / c2 * (GW[0] + GW[1] + GW[2]);
#pragma unroll
            for (int i = 0; i < 4; ++i) red_add(P.g_rot, g * 4 + i, gq[i] + 2.0 * ly.q[i] * dLdc);
        }
    }
    if constexpr (RAY_GRAD) {
        // the SH direction d / |d|: dL/dd += (I - dn dn^T) dL/ddn / |d|
        if (P.has_sh) {
            const double il = 1.0 / sqrt(d.x * d.x + d.y * d.y + d.z * d.z);
            const double dn[3] = {d.x * il, d.y * il, d.z * il};
            double gn[3];
            sh_basis_vjp_d(dn[0], dn[1], dn[2], gY, gn);
            const double pr = dn[0] * gn[0] + dn[1] * gn[1] + dn[2] * gn[2];
#pragma unroll
            for (int j = 0; j < 3; ++j) gD[j] += (gn[j] - dn[j] * pr) * il;
        }
    }
}

// One pixel of k_render_backward; a pixel that contributes nothing returns early.  With CAM, its camera terms are
// written to cam_g[CAM_TERMS] (left untouched, i.e. zero, on an early return).  DEPTH: dL_dD and replay_depth.
template <bool CAM, bool DEPTH>
__device__ __forceinline__ void backward_pixel(const BackwardParams& P, int tile, int lane, double* cam_g) {
    const int ti = tile / P.tiles_j, tj = tile - ti * P.tiles_j;
    const int li = ti * TILE_I + lane / TILE_J, lj = tj * TILE_J + lane % TILE_J;   // region-relative pixel
    if (li >= P.w || lj >= P.h) return;
    const int pi = P.x0 + li, pj = P.y0 + lj;
    const int64_t pix = (int64_t)li * P.h + lj;
    const CamD& cam = P.cam;
    const double o[3] = {cam.o[0], cam.o[1], cam.o[2]};
    const d3 d = cam_dir(cam, (double)pi + 0.5, (double)pj + 0.5);

    double kt[RTGS_MAX_DEPTH];
    int ks[RTGS_MAX_DEPTH];
    const int cnt = walk_layers<false>(P, o, d, 0.0, INFINITY, kt, ks);
    double Y[15];
    const int L = replay_layers<DEPTH>(P, o, d, cnt, kt, ks, pix, Y);
    const double gr[3] = {P.dL_drgb[pix * 3 + 0], P.dL_drgb[pix * 3 + 1], P.dL_drgb[pix * 3 + 2]};
    const double B = P.dL_dT != nullptr ? (double)P.dL_dT[pix] : 0.0;
    const double gDep = DEPTH && P.dL_dD != nullptr ? (double)P.dL_dD[pix] : 0.0;
    if (gr[0] == 0.0 && gr[1] == 0.0 && gr[2] == 0.0 && B == 0.0 && gDep == 0.0) return;
    double gO[3] = {0.0, 0.0, 0.0}, gD[3] = {0.0, 0.0, 0.0};   // CAM: dL/do, dL/dd
    back_to_front<CAM, DEPTH>(P, o, d, L, kt, ks, Y, gr, B, gO, gD, gDep);
    if constexpr (CAM) {
        // d = Rm dc, dc = n / |n| as cam_dir computes them
        const double px = ((double)pi + 0.5 - 0.5 * (double)cam.W) * cam.ifx;
        const double py = ((double)pj + 0.5 - 0.5 * (double)cam.H) * cam.ify;
        const double inv = rsqrt(px * px + py * py + 1.0);
        const double dc[3] = {px * inv, py * inv, -inv};
        double gdc[3];   // Rm^T dL/dd
#pragma unroll
        for (int j = 0; j < 3; ++j) gdc[j] = cam.R[j] * gD[0] + cam.R[3 + j] * gD[1] + cam.R[6 + j] * gD[2];
        const double pr = dc[0] * gdc[0] + dc[1] * gdc[1] + dc[2] * gdc[2];
        cam_g[0] = gO[0]; cam_g[1] = gO[1]; cam_g[2] = gO[2];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int k = 0; k < 3; ++k) cam_g[3 + r * 3 + k] = gD[r] * dc[k];
        cam_g[12] = -(gdc[0] - dc[0] * pr) * inv * px * cam.ifx;
        cam_g[13] = -(gdc[1] - dc[1] * pr) * inv * py * cam.ify;
    }
}

// The CTA's camera terms, summed in a fixed order: lanes by shuffles, then the warps in order.  Every thread of the
// CTA must arrive.
__device__ __forceinline__ void cam_block_reduce(const BackwardParams& P, double (&cg)[CAM_TERMS]) {
    __shared__ double red[BWD_WARPS][CAM_TERMS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < CAM_TERMS; ++i) {
        double v = cg[i];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < CAM_TERMS) {
        double v = red[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < BWD_WARPS; ++w) v += red[w][threadIdx.x];
        P.cam_part[(int64_t)threadIdx.x * gridDim.x + blockIdx.x] = v;
    }
}

// CAM = false: the Gaussian gradients.  CAM = true: also the camera's, as per-CTA partials in P.cam_part (finished
// by k_camera_grad_finalize).  DEPTH: the depth terms as well (rtgs_render_backward_depth), at the occupancy of the
// plain instantiation with the same CAM.
// The minimum CTA counts hold both instantiations at their occupancy (128 registers: 4 CTAs per SM, 168: 3); left to
// itself ptxas gives the CAM path 178 registers without spills, which fits only 2.
template <bool CAM, bool DEPTH = false>
__global__ void __launch_bounds__(BWD_WARPS * 32, CAM ? 3 : 4)
    k_render_backward(const __grid_constant__ BackwardParams P) {
    const int lane = threadIdx.x & 31;
    const int tile = blockIdx.x * BWD_WARPS + (threadIdx.x >> 5);
    if constexpr (!CAM) {
        if (tile >= P.ntiles) return;
        backward_pixel<false, DEPTH>(P, tile, lane, nullptr);
    } else {
        // absent pixels and tiles contribute zeros: every lane reaches the shuffles and the barrier
        double cg[CAM_TERMS];
#pragma unroll
        for (int i = 0; i < CAM_TERMS; ++i) cg[i] = 0.0;
        if (tile < P.ntiles) backward_pixel<true, DEPTH>(P, tile, lane, cg);
        cam_block_reduce(P, cg);
    }
}

// One CTA: sums the (CAM_TERMS, nparts) partials in a fixed order, takes dL/dRm to dL/dq_cam, and adds the three
// float32-rounded results to the caller's buffers (any may be null).
__global__ void __launch_bounds__(FIN_THREADS) k_camera_grad_finalize(const double* __restrict__ part, int nparts,
                                                                      const __grid_constant__ CamD cam, float* g_pos,
                                                                      float* g_rot, float* g_focal) {
    __shared__ double red[CAM_TERMS][FIN_THREADS];
    const int t = threadIdx.x;
    for (int i = 0; i < CAM_TERMS; ++i) {
        double v = 0.0;
        for (int b = t; b < nparts; b += FIN_THREADS) v += part[(int64_t)i * nparts + b];
        red[i][t] = v;
    }
    __syncthreads();
    for (int s = FIN_THREADS / 2; s > 0; s >>= 1) {
        if (t < s)
            for (int i = 0; i < CAM_TERMS; ++i) red[i][t] += red[i][t + s];
        __syncthreads();
    }
    if (t != 0) return;
    if (g_pos != nullptr)
        for (int j = 0; j < 3; ++j) g_pos[j] += (float)red[j][0];
    if (g_rot != nullptr) {
        // the camera uses Rm(q) unscaled: no |q| factor besides the one inside Rm
        const double q[4] = {cam.q[0], cam.q[1], cam.q[2], cam.q[3]};
        double M[3][3], gq[4];
        for (int r = 0; r < 3; ++r)
            for (int k = 0; k < 3; ++k) M[r][k] = red[3 + r * 3 + k][0];
        rot_mat_vjp(q, M, gq);
        for (int j = 0; j < 4; ++j) g_rot[j] += (float)gq[j];
    }
    if (g_focal != nullptr) {
        g_focal[0] += (float)red[12][0];
        g_focal[1] += (float)red[13][0];
    }
}

// ---- arbitrary rays (rtgs_render_rays / rtgs_render_rays_backward): one thread per ray ----------------------------

constexpr int RAY_THREADS = 128;

// Ray r of the (nrays, 8) record (o xyz, d xyz, start, end; 16-byte aligned, two float4 loads).  False for a ray that
// composites nothing: a non-finite o or d component, d = 0, or !(start < end) (NaN included).
__device__ __forceinline__ bool load_ray(const BackwardParams& P, int64_t r, double (&o)[3], d3& d, double& t_start,
                                         double& t_end) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(P.rays) + r * 2 + 0),
                 b = __ldg(reinterpret_cast<const float4*>(P.rays) + r * 2 + 1);
    o[0] = a.x; o[1] = a.y; o[2] = a.z;
    d = d3make(a.w, b.x, b.y);
    t_start = b.z;
    t_end = b.w;
    const bool finite = isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w) && isfinite(b.x) &&
                        isfinite(b.y);
    return finite && (a.w != 0.0f || b.x != 0.0f || b.y != 0.0f) && b.z < b.w;
}

// Phases 1-2 per ray: float32 rgb to replay_rgb (n,3), T to replay_T (n) if not null, with DEPTH the depth to
// replay_depth (n) if not null.  The same code as the replay of k_render_rays_backward, so the two agree bit for bit.
template <bool DEPTH = false>
__global__ void __launch_bounds__(RAY_THREADS) k_render_rays(const __grid_constant__ BackwardParams P) {
    const int64_t r = blockIdx.x * (int64_t)RAY_THREADS + threadIdx.x;
    if (r >= P.nrays) return;
    double o[3], t_start, t_end;
    d3 d;
    double kt[RTGS_MAX_DEPTH];
    int ks[RTGS_MAX_DEPTH];
    const int cnt = load_ray(P, r, o, d, t_start, t_end) ? walk_layers<true>(P, o, d, t_start, t_end, kt, ks) : 0;
    double Y[15];
    replay_layers<DEPTH>(P, o, d, cnt, kt, ks, r, Y);   // no layer: rgb 0, T 1, depth 0
}

// Phases 1-3 per ray.  RAY_GRAD = false: the Gaussian gradients only.  RAY_GRAD = true: also dL/do and dL/dd, added
// by the ray's own thread to g_rays[r * 8 + 0..5] (no atomics: deterministic).
// at the occupancy of the matching k_render_backward instantiation.  DEPTH: dL_dD and replay_depth.
template <bool RAY_GRAD, bool DEPTH = false>
__global__ void __launch_bounds__(RAY_THREADS, RAY_GRAD ? 3 : 4)
    k_render_rays_backward(const __grid_constant__ BackwardParams P) {
    const int64_t r = blockIdx.x * (int64_t)RAY_THREADS + threadIdx.x;
    if (r >= P.nrays) return;
    double o[3], t_start, t_end;
    d3 d;
    double kt[RTGS_MAX_DEPTH];
    int ks[RTGS_MAX_DEPTH];
    const bool valid = load_ray(P, r, o, d, t_start, t_end);
    const int cnt = valid ? walk_layers<true>(P, o, d, t_start, t_end, kt, ks) : 0;
    double Y[15];
    const int L = replay_layers<DEPTH>(P, o, d, cnt, kt, ks, r, Y);
    if (!valid) return;
    const double gr[3] = {P.dL_drgb[r * 3 + 0], P.dL_drgb[r * 3 + 1], P.dL_drgb[r * 3 + 2]};
    const double B = P.dL_dT != nullptr ? (double)P.dL_dT[r] : 0.0;
    const double gDep = DEPTH && P.dL_dD != nullptr ? (double)P.dL_dD[r] : 0.0;
    if (gr[0] == 0.0 && gr[1] == 0.0 && gr[2] == 0.0 && B == 0.0 && gDep == 0.0) return;
    double gO[3] = {0.0, 0.0, 0.0}, gD[3] = {0.0, 0.0, 0.0};
    back_to_front<RAY_GRAD, DEPTH>(P, o, d, L, kt, ks, Y, gr, B, gO, gD, gDep);
    if constexpr (RAY_GRAD) {
        float* g = P.g_rays + r * 8;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            g[j] += (float)gO[j];
            g[3 + j] += (float)gD[j];
        }
    }
}

}  // namespace backward
}  // namespace rtgs_dev
