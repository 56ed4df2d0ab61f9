// K1 / K8: per-Gaussian EWA projection + SH colour, forward and backward, both constant sets.
//
// One thread per Gaussian.  Forward restates the arithmetic of
//   /root/reference/internal/utils/gaussian_projection.py:6-138   (gsplat mode; live-pinned by tests/golden)
//   /root/reference/internal/utils/sh_utils.py:57-112             (SH polynomials)
// and, for vanilla mode, the published preprocessCUDA of diff-gaussian-rasterization@59f5f77 (SURVEY §8c).
// Backward is hand-derived (DESIGN.md §K8) and checked against torch autograd through the oracle.
//
// HBM-bound: per visible Gaussian 268 B fwd / 552 B bwd at SH degree 3.  SH coefficients are streamed with
// 128-bit read-only loads (ld.global.nc), outputs written with 64/128-bit stores where the layout allows.
#include "common.cuh"
#include "onesweep.cuh"

namespace b200gs {

namespace {

constexpr float SH_C0 = 0.28209479177387814f;
constexpr float SH_C1 = 0.4886025119029199f;
__device__ constexpr float SH_C2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                                       -1.0925484305920792f, 0.5462742152960396f};
__device__ constexpr float SH_C3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                                       -0.4570457994644658f, 1.445305721320277f, -0.5900435899266435f};
__device__ constexpr float SH_C4[9] = {2.5033429417967046f, -1.7701307697799304f, 0.9461746957575601f, -0.6690465435572892f,
                                       0.10578554691520431f, -0.6690465435572892f, 0.47308734787878004f, -1.7701307697799304f,
                                       0.6258357354491761f};

// Every kernel that touches SH coefficients is instantiated for MC = 16 (degrees 0..3, the common case: 48 coefficient
// registers) and MC = 25 (degree 4, sh_utils.py:102-111: 75 registers); the launchers pick by the view's sh_degree.

// Loads the first ncoef*3 floats of one Gaussian's SH block into registers. 128-bit path when the block is 16B aligned.
template <int MC>
__device__ __forceinline__ void load_sh(const float* __restrict__ base, int ncoef, bool vec4, float* sh) {
    const int nf = ncoef * 3;
    if (vec4) {
        const float4* b4 = reinterpret_cast<const float4*>(base);
#pragma unroll
        for (int q = 0; q < MC * 3 / 4; ++q) {
            if (q * 4 < nf) {
                float4 t = __ldg(b4 + q);
                sh[q * 4 + 0] = t.x; sh[q * 4 + 1] = t.y; sh[q * 4 + 2] = t.z; sh[q * 4 + 3] = t.w;
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < MC * 3; ++q)
            if (q < nf) sh[q] = __ldg(base + q);
    }
}

// ---- arithmetic with the evaluation order written out ---------------------------------------------------------------------
// The same inline function compiled into two kernels is NOT guaranteed to round the same way: where a product has several uses (x*x,
// b*b, ...) nvcc's fmul+fadd -> fma contraction depends on the surrounding code (measured, round 2: the SH colours of the single-view
// K1 and of the multi-view K1 of the sharded renderer differed in the last bit for ~1 % of the splats -> a sharded image 1 ulp off
// the single-GPU image).  Everything the FORWARD projection computes therefore goes through these helpers: __fmul_rn / __fadd_rn /
// __fmaf_rn (and the double versions) are never contracted, split or reassociated, so every kernel that inlines the functions below
// produces the same bits (tests/test_gpu_sharded_kernels.py).
__device__ __forceinline__ float xm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float xa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float xf(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ double xm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xa(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xf(double a, double b, double c) { return __fma_rn(a, b, c); }

// unit view direction camera -> Gaussian and 1 / distance
__device__ __forceinline__ void view_dir(const float* p, const float* campos, float& dx, float& dy, float& dz, float& inv_len) {
    dx = xa(p[0], -campos[0]); dy = xa(p[1], -campos[1]); dz = xa(p[2], -campos[2]);
    inv_len = rsqrtf(xf(dz, dz, xf(dy, dy, xm(dx, dx))));
    dx = xm(dx, inv_len); dy = xm(dy, inv_len); dz = xm(dz, inv_len);
}

// basis values for unit direction (x,y,z); writes (deg+1)^2 entries (sh_utils.py:57-112)
template <int MC>
__device__ __forceinline__ void sh_basis(int deg, float x, float y, float z, float* b) {
    b[0] = SH_C0;
    if (deg > 0) {
        b[1] = xm(-SH_C1, y); b[2] = xm(SH_C1, z); b[3] = xm(-SH_C1, x);
        if (deg > 1) {
            const float xx = xm(x, x), yy = xm(y, y), zz = xm(z, z), xy = xm(x, y), yz = xm(y, z), xz = xm(x, z);
            const float xx_yy = xa(xx, -yy);
            b[4] = xm(SH_C2[0], xy); b[5] = xm(SH_C2[1], yz); b[6] = xm(SH_C2[2], xa(xf(2.0f, zz, -xx), -yy));
            b[7] = xm(SH_C2[3], xz); b[8] = xm(SH_C2[4], xx_yy);
            if (deg > 2) {
                const float t4 = xa(xf(4.0f, zz, -xx), -yy);          // 4 zz - xx - yy
                b[9] = xm(xm(SH_C3[0], y), xf(3.0f, xx, -yy)); b[10] = xm(xm(SH_C3[1], xy), z);
                b[11] = xm(xm(SH_C3[2], y), t4); b[12] = xm(xm(SH_C3[3], z), xf(-3.0f, yy, xf(-3.0f, xx, xm(2.0f, zz))));
                b[13] = xm(xm(SH_C3[4], x), t4); b[14] = xm(xm(SH_C3[5], z), xx_yy);
                b[15] = xm(xm(SH_C3[6], x), xf(-3.0f, yy, xx));
                if (MC > 16 && deg > 3) {
                    const float s7 = xf(7.0f, zz, -1.0f), t7 = xf(7.0f, zz, -3.0f);
                    b[16] = xm(xm(SH_C4[0], xy), xx_yy); b[17] = xm(xm(SH_C4[1], yz), xf(3.0f, xx, -yy));
                    b[18] = xm(xm(SH_C4[2], xy), s7); b[19] = xm(xm(SH_C4[3], yz), t7);
                    b[20] = xm(SH_C4[4], xf(zz, xf(35.0f, zz, -30.0f), 3.0f)); b[21] = xm(xm(SH_C4[5], xz), t7);
                    b[22] = xm(xm(SH_C4[6], xx_yy), s7); b[23] = xm(xm(SH_C4[7], xz), xf(-3.0f, yy, xx));
                    b[24] = xm(SH_C4[8], xf(xx, xf(-3.0f, yy, xx), -xm(yy, xf(3.0f, xx, -yy))));
                }
            }
        }
    }
}

// d(basis)/d(x,y,z)
template <int MC>
__device__ __forceinline__ void sh_basis_grad(int deg, float x, float y, float z, float* bx, float* by, float* bz) {
    bx[0] = by[0] = bz[0] = 0.f;
    if (deg > 0) {
        bx[1] = 0.f; by[1] = -SH_C1; bz[1] = 0.f;
        bx[2] = 0.f; by[2] = 0.f; bz[2] = SH_C1;
        bx[3] = -SH_C1; by[3] = 0.f; bz[3] = 0.f;
        if (deg > 1) {
            bx[4] = SH_C2[0] * y; by[4] = SH_C2[0] * x; bz[4] = 0.f;
            bx[5] = 0.f; by[5] = SH_C2[1] * z; bz[5] = SH_C2[1] * y;
            bx[6] = SH_C2[2] * -2.f * x; by[6] = SH_C2[2] * -2.f * y; bz[6] = SH_C2[2] * 4.f * z;
            bx[7] = SH_C2[3] * z; by[7] = 0.f; bz[7] = SH_C2[3] * x;
            bx[8] = SH_C2[4] * 2.f * x; by[8] = SH_C2[4] * -2.f * y; bz[8] = 0.f;
            if (deg > 2) {
                const float xx = x * x, yy = y * y, zz = z * z;
                bx[9] = SH_C3[0] * 6.f * x * y; by[9] = SH_C3[0] * (3.f * xx - 3.f * yy); bz[9] = 0.f;
                bx[10] = SH_C3[1] * y * z; by[10] = SH_C3[1] * x * z; bz[10] = SH_C3[1] * x * y;
                bx[11] = SH_C3[2] * -2.f * x * y; by[11] = SH_C3[2] * (4.f * zz - xx - 3.f * yy); bz[11] = SH_C3[2] * 8.f * y * z;
                bx[12] = SH_C3[3] * -6.f * x * z; by[12] = SH_C3[3] * -6.f * y * z; bz[12] = SH_C3[3] * (6.f * zz - 3.f * xx - 3.f * yy);
                bx[13] = SH_C3[4] * (4.f * zz - 3.f * xx - yy); by[13] = SH_C3[4] * -2.f * x * y; bz[13] = SH_C3[4] * 8.f * x * z;
                bx[14] = SH_C3[5] * 2.f * x * z; by[14] = SH_C3[5] * -2.f * y * z; bz[14] = SH_C3[5] * (xx - yy);
                bx[15] = SH_C3[6] * (3.f * xx - 3.f * yy); by[15] = SH_C3[6] * -6.f * x * y; bz[15] = 0.f;
                if (MC > 16 && deg > 3) {
                    const float xyz = x * y * z, s7 = 7.f * zz - 1.f, t7 = 7.f * zz - 3.f, u21 = 21.f * zz - 3.f;
                    bx[16] = SH_C4[0] * y * (3.f * xx - yy); by[16] = SH_C4[0] * x * (xx - 3.f * yy); bz[16] = 0.f;
                    bx[17] = SH_C4[1] * 6.f * xyz; by[17] = SH_C4[1] * 3.f * z * (xx - yy); bz[17] = SH_C4[1] * y * (3.f * xx - yy);
                    bx[18] = SH_C4[2] * y * s7; by[18] = SH_C4[2] * x * s7; bz[18] = SH_C4[2] * 14.f * xyz;
                    bx[19] = 0.f; by[19] = SH_C4[3] * z * t7; bz[19] = SH_C4[3] * y * u21;
                    bx[20] = 0.f; by[20] = 0.f; bz[20] = SH_C4[4] * z * (140.f * zz - 60.f);
                    bx[21] = SH_C4[5] * z * t7; by[21] = 0.f; bz[21] = SH_C4[5] * x * u21;
                    bx[22] = SH_C4[6] * 2.f * x * s7; by[22] = SH_C4[6] * -2.f * y * s7; bz[22] = SH_C4[6] * 14.f * z * (xx - yy);
                    bx[23] = SH_C4[7] * 3.f * z * (xx - yy); by[23] = SH_C4[7] * -6.f * xyz; bz[23] = SH_C4[7] * x * (xx - 3.f * yy);
                    bx[24] = SH_C4[8] * 4.f * x * (xx - 3.f * yy); by[24] = SH_C4[8] * 4.f * y * (yy - 3.f * xx); bz[24] = 0.f;
                }
            }
        }
    }
}

// Geometry shared by forward and backward.  R = double in the forward: the conic is the inverse of a 2x2 matrix whose
// condition number reaches 1e4 for elongated splats, so fp32 intermediates put ~1e-4 of noise on pixels (measured: two
// fp32 evaluation orders of the same formulas differ by 1.1e-4 on a 256x256 render).  Evaluating the ~150 flops per
// Gaussian in fp64 (inputs and outputs stay fp32) removes that noise for ~10 us per million Gaussians on B200.
template <typename R>
struct Proj {
    R tx, ty, tz;        // camera-space mean
    R cxp, cyp;          // clamped tx', ty' used in J
    bool clx, cly;       // clamp active
    R fx, fy;            // focal used by J
    R Rm[9];             // rotation from quaternion (row major)
    R s[3];              // scales * modifier
    R S3[6];             // cov3D upper triangle xx xy xz yy yz zz
    R T[6];              // T = J * Rw, rows 0,1 (2x3)
    R a, b, c, det;      // blurred cov2D and determinant
    R a0, c0, det0;      // un-blurred diag and determinant (gsplat compensation)
    R qr, qx, qy, qz;    // the unit quaternion Rm was built from (filled by the backward kernels)
};

template <typename R>
__device__ __forceinline__ void quat_to_rot(const R* q, R* Rm) {
    const R r = q[0], x = q[1], y = q[2], z = q[3];
    const R two = R(2), one = R(1);
    Rm[0] = xf(-two, xf(z, z, xm(y, y)), one); Rm[1] = xm(two, xf(-r, z, xm(x, y))); Rm[2] = xm(two, xf(r, y, xm(x, z)));
    Rm[3] = xm(two, xf(r, z, xm(x, y))); Rm[4] = xf(-two, xf(z, z, xm(x, x)), one); Rm[5] = xm(two, xf(-r, x, xm(y, z)));
    Rm[6] = xm(two, xf(-r, y, xm(x, z))); Rm[7] = xm(two, xf(r, x, xm(y, z))); Rm[8] = xf(-two, xf(y, y, xm(x, x)), one);
}

// The camera-independent half of the geometry: rotation, scaled axes, cov3D = (R S)(R S)^T.  The multi-view kernels of the sharded
// renderer evaluate it ONCE per Gaussian (scale_modifier of views[0]) and only project_view per camera.
template <typename R>
__device__ __forceinline__ void gaussian_cov3d(const R* sc, const R* q, float scale_modifier, Proj<R>& g) {
    quat_to_rot<R>(q, g.Rm);
#pragma unroll
    for (int k = 0; k < 3; ++k) g.s[k] = xm(sc[k], R(scale_modifier));
    R M[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) M[i * 3 + k] = xm(g.Rm[i * 3 + k], g.s[k]);
    g.S3[0] = xf(M[2], M[2], xf(M[1], M[1], xm(M[0], M[0])));
    g.S3[1] = xf(M[2], M[5], xf(M[1], M[4], xm(M[0], M[3])));
    g.S3[2] = xf(M[2], M[8], xf(M[1], M[7], xm(M[0], M[6])));
    g.S3[3] = xf(M[5], M[5], xf(M[4], M[4], xm(M[3], M[3])));
    g.S3[4] = xf(M[5], M[8], xf(M[4], M[7], xm(M[3], M[6])));
    g.S3[5] = xf(M[8], M[8], xf(M[7], M[7], xm(M[6], M[6])));
}

template <bool GSPLAT, typename R>
__device__ __forceinline__ void project_view(const B200gsView& v, const float* p, Proj<R>& g);

template <bool GSPLAT, typename R>
__device__ __forceinline__ void project_geometry(const B200gsView& v, const float* p, const R* sc, const R* q, Proj<R>& g) {
    gaussian_cov3d<R>(sc, q, v.scale_modifier, g);
    project_view<GSPLAT, R>(v, p, g);
}

// The per-camera half: camera-space mean, Jacobian, cov2D (+ blur), determinants.  g.S3 (and Rm, s for the backward) are inputs.
template <bool GSPLAT, typename R>
__device__ __forceinline__ void project_view(const B200gsView& v, const float* p, Proj<R>& g) {
    const float* V = v.viewmatrix;
    const R p0 = p[0], p1 = p[1], p2 = p[2];
    g.tx = xa(xf(p2, R(V[8]), xf(p1, R(V[4]), xm(p0, R(V[0])))), R(V[12]));
    g.ty = xa(xf(p2, R(V[9]), xf(p1, R(V[5]), xm(p0, R(V[1])))), R(V[13]));
    g.tz = xa(xf(p2, R(V[10]), xf(p1, R(V[6]), xm(p0, R(V[2])))), R(V[14]));

    R tanx, tany;
    if (GSPLAT) {
        g.fx = v.fx; g.fy = v.fy;
        tanx = xm(R(0.5), R(v.width)) / R(v.fx);
        tany = xm(R(0.5), R(v.height)) / R(v.fy);
    } else {
        tanx = v.tanfovx; tany = v.tanfovy;
        g.fx = R(v.width) / xm(R(2), tanx);
        g.fy = R(v.height) / xm(R(2), tany);
    }
    const R limx = xm(R(1.3), tanx), limy = xm(R(1.3), tany);
    const R txtz = g.tx / g.tz, tytz = g.ty / g.tz;
    g.clx = (txtz < -limx) || (txtz > limx);
    g.cly = (tytz < -limy) || (tytz > limy);
    g.cxp = xm(fmin(limx, fmax(-limx, txtz)), g.tz);
    g.cyp = xm(fmin(limy, fmax(-limy, tytz)), g.tz);
    const R itz = R(1) / g.tz;
    const R j00 = xm(g.fx, itz), j02 = xm(xm(-xm(g.fx, g.cxp), itz), itz);
    const R j11 = xm(g.fy, itz), j12 = xm(xm(-xm(g.fy, g.cyp), itz), itz);
    // T = J * Rw ; Rw[j][i] = V[i*4+j]
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        g.T[i] = xf(j02, R(V[i * 4 + 2]), xm(j00, R(V[i * 4 + 0])));
        g.T[3 + i] = xf(j12, R(V[i * 4 + 2]), xm(j11, R(V[i * 4 + 1])));
    }
    // cov2D = T S3 T^T
    const R* S = g.S3;
    const R* T = g.T;
    const R u0 = xf(S[2], T[2], xf(S[1], T[1], xm(S[0], T[0])));
    const R u1 = xf(S[4], T[2], xf(S[3], T[1], xm(S[1], T[0])));
    const R u2 = xf(S[5], T[2], xf(S[4], T[1], xm(S[2], T[0])));
    const R w0 = xf(S[2], T[5], xf(S[1], T[4], xm(S[0], T[3])));
    const R w1 = xf(S[4], T[5], xf(S[3], T[4], xm(S[1], T[3])));
    const R w2 = xf(S[5], T[5], xf(S[4], T[4], xm(S[2], T[3])));
    g.a0 = xf(T[2], u2, xf(T[1], u1, xm(T[0], u0)));
    g.b = xf(T[5], u2, xf(T[4], u1, xm(T[3], u0)));
    g.c0 = xf(T[5], w2, xf(T[4], w1, xm(T[3], w0)));
    const R bb = xm(g.b, g.b);
    g.det0 = xf(g.a0, g.c0, -bb);
    g.a = xa(g.a0, R(v.eps2d));
    g.c = xa(g.c0, R(v.eps2d));
    g.det = xf(g.a, g.c, -bb);
}

// Optional fused-activation ("raw parameter") operands: the model's exp / normalize / sigmoid activations and the
// dc|rest concatenation (vanilla_gaussian.py:345-358, gaussian.py:250-254) folded into K1 / K8.
struct RawIO {
    const float* opac_in;    // [n] opacity logits
    const float* shs_rest;   // [n, sh_stride-1, 3]; the `shs` argument then points at shs_dc [n,1,3]
    float* opac_out;         // [n] opacity handed to the blend kernels (sigmoid, x compensation when anti_aliased)
    const float* v_opac;     // [n] dL/d(opac_out) from the blend backward
    float* v_opac_logit;     // [n]
    float* v_shs_rest;       // [n, sh_stride-1, 3]; `v_shs` then receives the dc gradient [n,1,3]
    int anti_aliased;
    // backward of the sharded renderer: cotangents come as compacted [V,12] rows (b200gs.h row layout) addressed through
    // row_offsets[n] (exclusive scan of the visibility flags), and gradients are ACCUMULATED over the W cameras of a step
    const float* v_rows;
    const int32_t* row_offsets;
    int accumulate;
    float* v_mean2d;         // K8 (rows path, optional): [n, v_mean2d_cols] <- (dL/dmean2D.x, .y[, 0]) of every Gaussian, zeros for culled ones:
    int v_mean2d_cols;       // the `viewspace_points.grad` of the renderer contract, written here instead of by a fill + strided copy
};

template <bool RAW, typename R>
__device__ __forceinline__ void load_scale_quat(const float* __restrict__ scales, const float* __restrict__ quats, int64_t i, R* sc, R* q,
                                                R* inv_qnorm) {
    const float s0 = __ldg(scales + 3 * i), s1 = __ldg(scales + 3 * i + 1), s2 = __ldg(scales + 3 * i + 2);
    const float4 q4 = __ldg(reinterpret_cast<const float4*>(quats) + i);
    if (RAW) {
        sc[0] = exp(R(s0)); sc[1] = exp(R(s1)); sc[2] = exp(R(s2));
        const R w = q4.x, x = q4.y, y = q4.z, z = q4.w;
        const R inv = R(1) / fmax(sqrt(xf(z, z, xf(y, y, xf(x, x, xm(w, w))))), R(1e-12));  // F.normalize eps
        q[0] = xm(w, inv); q[1] = xm(x, inv); q[2] = xm(y, inv); q[3] = xm(z, inv);
        *inv_qnorm = inv;
    } else {
        sc[0] = s0; sc[1] = s1; sc[2] = s2;
        q[0] = q4.x; q[1] = q4.y; q[2] = q4.z; q[3] = q4.w;
        *inv_qnorm = R(1);
    }
}

// SH block of Gaussian i into registers: [K,3] contiguous, or dc [1,3] + rest [K-1,3] when RAW
template <bool RAW, int MC>
__device__ __forceinline__ void load_sh_any(const float* __restrict__ shs, const float* __restrict__ shs_rest, int64_t i, int stride,
                                            int ncoef, float* sh) {
    if (RAW) {
        sh[0] = __ldg(shs + 3 * i); sh[1] = __ldg(shs + 3 * i + 1); sh[2] = __ldg(shs + 3 * i + 2);
        const float* r = shs_rest + i * int64_t(stride - 1) * 3;
#pragma unroll
        for (int q = 3; q < MC * 3; ++q)
            if (q < ncoef * 3) sh[q] = __ldg(r + q - 3);
    } else {
        load_sh<MC>(shs + i * int64_t(stride) * 3, ncoef, ((stride * 3) & 3) == 0, sh);
    }
}

template <bool GSPLAT>
__device__ __forceinline__ float near_of(const B200gsView& v) {
    return v.near_plane > 0.f ? v.near_plane : (GSPLAT ? 0.01f : 0.2f);
}

// Destination of one view's projection outputs (element index `o` of every array).
struct ProjOut {
    float2* xy; float* depth; int32_t* radii; float* conic; float* comp; int32_t* tiles; float* cov3d; float* rgb; uint8_t* clamped;
};

// What one (view, Gaussian) projection produces (all zero when the Gaussian is culled)
struct ProjVals {
    float px, py, depth, cA, cB, cC, comp, opac;
    int32_t radius, ntiles;
};

// Projection of Gaussian (p, sc, q) into view v -> pv; returns the visibility.  cov3d (optional) is written at index o.
template <bool GSPLAT, bool RAW>
__device__ __forceinline__ bool project_one_view(const B200gsView& v, const RawIO& raw, int64_t i, int64_t o, const float* p, Proj<double>& g,
                                                 float* cov3d_out, ProjVals& pv);

template <bool GSPLAT, bool RAW>
__device__ __forceinline__ bool project_one(const B200gsView& v, const RawIO& raw, int64_t i, int64_t o, const float* p, const double* sc,
                                            const double* q, float* cov3d_out, ProjVals& pv) {
    Proj<double> g;
    gaussian_cov3d<double>(sc, q, v.scale_modifier, g);
    return project_one_view<GSPLAT, RAW>(v, raw, i, o, p, g, cov3d_out, pv);
}

// g: gaussian_cov3d already evaluated
template <bool GSPLAT, bool RAW>
__device__ __forceinline__ bool project_one_view(const B200gsView& v, const RawIO& raw, int64_t i, int64_t o, const float* p, Proj<double>& g,
                                                 float* cov3d_out, ProjVals& pv) {
    typedef double R;
    project_view<GSPLAT, R>(v, p, g);

    const float near = near_of<GSPLAT>(v);
    bool vis = GSPLAT ? (float(g.tz) >= near) : (float(g.tz) > near);
    if (!GSPLAT) vis = vis && (g.det != R(0));

    R pxd, pyd;
    if (GSPLAT) {
        const R iz = R(1) / xa(g.tz, R(1e-6));
        const R zn = xm(g.tz, iz);
        pxd = xf(zn, R(v.cx), xm(xm(g.tx, iz), R(v.fx)));
        pyd = xf(zn, R(v.cy), xm(xm(g.ty, iz), R(v.fy)));
    } else {
        const float* P = v.projmatrix;
        const R p0 = p[0], p1 = p[1], p2 = p[2];
        const R hx = xa(xf(p2, R(P[8]), xf(p1, R(P[4]), xm(p0, R(P[0])))), R(P[12]));
        const R hy = xa(xf(p2, R(P[9]), xf(p1, R(P[5]), xm(p0, R(P[1])))), R(P[13]));
        const R hw = xa(xf(p2, R(P[11]), xf(p1, R(P[7]), xm(p0, R(P[3])))), R(P[15]));
        const R iw = R(1) / xa(hw, R(0.0000001));
        pxd = xm(xf(xf(hx, iw, R(1)), R(v.width), R(-1)), R(0.5));
        pyd = xm(xf(xf(hy, iw, R(1)), R(v.height), R(-1)), R(0.5));
    }
    const float px = float(pxd), py = float(pyd);
    const R inv_det = R(1) / g.det;
    const R mid = xm(R(0.5), xa(g.a, g.c));
    const R sq = sqrt(fmax(R(0.1), xf(mid, mid, -g.det)));
    const R lam = fmax(xa(mid, sq), xa(mid, -sq));
    const float radius = float(ceil(xm(R(3), sqrt(lam))));
    const int grid_x = div_up(v.width, TILE), grid_y = div_up(v.height, TILE);
    int x0, y0, x1, y1;
    tile_rect<GSPLAT>(px, py, radius, grid_x, grid_y, x0, y0, x1, y1);
    const int ntiles = (x1 - x0) * (y1 - y0);
    vis = vis && (ntiles > 0) && (radius > 0.f);  // NaN radius compares false

    pv.px = pv.py = pv.depth = pv.cA = pv.cB = pv.cC = pv.comp = pv.opac = 0.f;
    pv.radius = pv.ntiles = 0;
    if (vis) {
        pv.px = px; pv.py = py;
        pv.depth = float(g.tz);
        pv.radius = (int32_t)radius;
        pv.cA = float(xm(g.c, inv_det));
        pv.cB = float(xm(-g.b, inv_det));
        pv.cC = float(xm(g.a, inv_det));
        pv.ntiles = ntiles;
        pv.comp = GSPLAT ? float(sqrt(fmax(xm(g.det0, inv_det), R(0)))) : 1.0f;
        if (RAW) {
            const float op = __frcp_rn(xa(1.0f, __expf(-__ldg(raw.opac_in + i))));
            pv.opac = (GSPLAT && raw.anti_aliased) ? xm(op, pv.comp) : op;
        }
    }
    if (cov3d_out) {
#pragma unroll
        for (int k = 0; k < 6; ++k) cov3d_out[6 * o + k] = vis ? float(g.S3[k]) : 0.f;
    }
    return vis;
}

// separate-array outputs of one projection at element o
template <bool RAW>
__device__ __forceinline__ void store_soa(const ProjOut& out, float* opac_out, int64_t o, const ProjVals& pv) {
    out.xy[o] = make_float2(pv.px, pv.py);
    out.depth[o] = pv.depth;
    out.radii[o] = pv.radius;
    out.conic[3 * o + 0] = pv.cA; out.conic[3 * o + 1] = pv.cB; out.conic[3 * o + 2] = pv.cC;
    if (out.tiles) out.tiles[o] = pv.ntiles;
    if (out.comp) out.comp[o] = pv.radius > 0 ? pv.comp : 0.f;
    if (RAW) opac_out[o] = pv.opac;
}

// max(SH colour + 0.5, 0) of a visible Gaussian seen from v.campos; bit c of *cl set where channel c was clamped
template <int MC>
__device__ __forceinline__ void sh_color_one(const B200gsView& v, const float* p, const float* sh, float& r, float& gc, float& bc, uint8_t& cl) {
    const int deg = v.sh_degree;
    const int ncoef = (deg + 1) * (deg + 1);
    float dx, dy, dz, inv_len;
    view_dir(p, v.campos, dx, dy, dz, inv_len);
    float bs[MC];
    sh_basis<MC>(deg, dx, dy, dz, bs);
    r = xm(bs[0], sh[0]); gc = xm(bs[0], sh[1]); bc = xm(bs[0], sh[2]);
#pragma unroll
    for (int k = 1; k < MC; ++k) {
        if (k < ncoef) {
            r = xf(bs[k], sh[3 * k + 0], r);
            gc = xf(bs[k], sh[3 * k + 1], gc);
            bc = xf(bs[k], sh[3 * k + 2], bc);
        }
    }
    r = xa(r, 0.5f); gc = xa(gc, 0.5f); bc = xa(bc, 0.5f);
    cl = 0;
    if (r < 0.f) { r = 0.f; cl |= 1; }
    if (gc < 0.f) { gc = 0.f; cl |= 2; }
    if (bc < 0.f) { bc = 0.f; cl |= 4; }
}

// rows_out (raw mode only): instead of the separate arrays, ONE [n,12] row per Gaussian (xy 0..1, depth 2, conic 3..5, compensation 6,
// blend opacity 7, rgb 8..10, radius bits 11) — three 128-bit stores; the binning and the blend kernels read the rows in place (one
// 48-byte record per splat instead of four separate sectors).  radii_out / clamped_out (what K8 needs) are still written.
template <bool GSPLAT, bool RAW, int MC>
__global__ void __launch_bounds__(256, 3) project_fwd_kernel(const __grid_constant__ B200gsView v, const RawIO raw, int64_t n,
                                                          const float* __restrict__ means, const float* __restrict__ scales,
                                                          const float* __restrict__ quats, const float* __restrict__ shs,
                                                          float2* __restrict__ xy_out, float* __restrict__ depth_out,
                                                          int32_t* __restrict__ radii_out, float* __restrict__ conic_out,
                                                          float* __restrict__ comp_out, int32_t* __restrict__ tiles_out,
                                                          float* __restrict__ cov3d_out, float* __restrict__ rgb_out,
                                                          uint8_t* __restrict__ clamped_out, float* __restrict__ rows_out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float p[3] = {__ldg(means + 3 * i), __ldg(means + 3 * i + 1), __ldg(means + 3 * i + 2)};
    double sc[3], q[4], inv_qn;
    load_scale_quat<RAW, double>(scales, quats, i, sc, q, &inv_qn);
    const ProjOut out{xy_out, depth_out, radii_out, conic_out, comp_out, tiles_out, cov3d_out, rgb_out, clamped_out};
    ProjVals pv;
    const bool vis = project_one<GSPLAT, RAW>(v, raw, i, i, p, sc, q, cov3d_out, pv);
    const bool rows = RAW && rows_out != nullptr;
    if (!rows) store_soa<RAW>(out, raw.opac_out, i, pv);
    float r = 0.f, gc = 0.f, bc = 0.f;
    uint8_t cl = 0;
    if (shs != nullptr) {
        if (vis) {
            const int deg = v.sh_degree;
            float sh[MC * 3];
            load_sh_any<RAW, MC>(shs, raw.shs_rest, i, v.sh_stride, (deg + 1) * (deg + 1), sh);
            sh_color_one<MC>(v, p, sh, r, gc, bc, cl);
        }
        if (!rows) { rgb_out[3 * i + 0] = r; rgb_out[3 * i + 1] = gc; rgb_out[3 * i + 2] = bc; }
        clamped_out[i] = cl;
    }
    if (rows) {
        float4* row = reinterpret_cast<float4*>(rows_out + i * B200GS_ROW_FLOATS);
        radii_out[i] = pv.radius;
        if (tiles_out) tiles_out[i] = pv.ntiles;
        row[0] = make_float4(pv.px, pv.py, pv.depth, pv.cA);             // zeros when culled (the mean2D columns are handed out)
        if (vis) row[1] = make_float4(pv.cB, pv.cC, pv.comp, pv.opac);
        row[2] = make_float4(r, gc, bc, __int_as_float(pv.radius));      // radius 0 = culled: all the kernels look at of such a row
    }
}

// The sharded renderer projects ONE shard into the W cameras of a step: one launch, the parameters (and the SH block, if any view
// sees the Gaussian) are read once per Gaussian instead of once per camera.  gsplat constants, raw parameters.  View j's outputs
// live at elements [j*n, (j+1)*n) of camera-major arrays.
struct ViewPack {
    B200gsView v[B200GS_MAX_VIEWS];
};

template <int MC>
__global__ void __launch_bounds__(256) project_fwd_multi_kernel(const __grid_constant__ ViewPack vp, int nviews, const RawIO raw, int64_t n,
                                                                const float* __restrict__ means, const float* __restrict__ scales,
                                                                const float* __restrict__ quats, const float* __restrict__ shs_dc,
                                                                float2* __restrict__ xy_out, float* __restrict__ depth_out,
                                                                int32_t* __restrict__ radii_out, float* __restrict__ conic_out,
                                                                float* __restrict__ rgb_out, uint8_t* __restrict__ clamped_out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float p[3] = {__ldg(means + 3 * i), __ldg(means + 3 * i + 1), __ldg(means + 3 * i + 2)};
    double sc[3], q[4], inv_qn;
    load_scale_quat<true, double>(scales, quats, i, sc, q, &inv_qn);
    Proj<double> g3;
    gaussian_cov3d<double>(sc, q, vp.v[0].scale_modifier, g3);      // once per Gaussian; project_one_view per camera
    const ProjOut out{xy_out, depth_out, radii_out, conic_out, nullptr, nullptr, nullptr, rgb_out, clamped_out};
    unsigned vismask = 0;
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        ProjVals pv;
        if (project_one_view<true, true>(vp.v[j], raw, i, int64_t(j) * n + i, p, g3, nullptr, pv)) vismask |= 1u << j;
        store_soa<true>(out, raw.opac_out, int64_t(j) * n + i, pv);
    }
    float sh[MC * 3];
    if (vismask) {
        const int deg = vp.v[0].sh_degree;
        load_sh_any<true, MC>(shs_dc, raw.shs_rest, i, vp.v[0].sh_stride, (deg + 1) * (deg + 1), sh);
    }
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        float r = 0.f, gc = 0.f, bc = 0.f;
        uint8_t cl = 0;
        if ((vismask >> j) & 1u) sh_color_one<MC>(vp.v[j], p, sh, r, gc, bc, cl);
        const int64_t o = int64_t(j) * n + i;
        rgb_out[3 * o + 0] = r; rgb_out[3 * o + 1] = gc; rgb_out[3 * o + 2] = bc;
        clamped_out[o] = cl;
    }
}

// K1 of a shard for all W cameras FUSED with the exchange's packing: the visible splats of camera j leave this kernel as [.,12]
// rows stored straight into block `dst.p[j]` (capacity `cap` rows) of the rank that owns camera j — a peer GPU's receive buffer
// mapped over NVLink, or a local send buffer — in Gaussian-index order (what keeps the sharded image bit-identical to the
// single-GPU one).  No intermediate arrays, no separate scan / pack / pad kernels: blocks take tickets, every warp compacts its
// visible lanes per camera into a shared-memory row tile (ballot), warp j runs camera j's chained scan over the blocks
// (decoupled look-back, one value per block and camera), and the block copies its rows out as contiguous runs.  Rows beyond
// `cap` are dropped and show up in d_count[j] (total visible of camera j; the caller compares with cap and redoes the step with
// the exact exchange).  What the backward needs stays local: radii, clamped, row_index (block-relative row j*cap + k, or -1
// when dropped) at [j*n + i], and the mean2D (the per-camera viewspace points the renderer hands out).
struct PackDst {
    float* p[B200GS_MAX_VIEWS];
};
constexpr int PACK_THREADS = 256;
constexpr int PACK_WARPS = PACK_THREADS / 32;

template <int MC>
__global__ void __launch_bounds__(PACK_THREADS, (MC <= 16 ? 3 : 2)) project_pack_multi_kernel(const __grid_constant__ ViewPack vp, int nviews, const RawIO raw, int64_t n,
                                                                        const float* __restrict__ means, const float* __restrict__ scales,
                                                                        const float* __restrict__ quats, const float* __restrict__ shs_dc,
                                                                        float2* __restrict__ xy_out, int32_t* __restrict__ radii_out,
                                                                        uint8_t* __restrict__ clamped_out, int32_t* __restrict__ row_index_out,
                                                                        const PackDst dst, int64_t cap, uint32_t* __restrict__ ticket,
                                                                        uint32_t* __restrict__ scan_state /*[nviews][gridDim.x]*/,
                                                                        int64_t* __restrict__ d_count) {
    extern __shared__ float4 s_rows[];                           // [nviews][PACK_THREADS slots][3]: slot = warp * 32 + rank among the warp's visible lanes
    __shared__ int s_cnt[B200GS_MAX_VIEWS][PACK_WARPS];          // visible lanes per (camera, warp)
    __shared__ uint32_t s_pre[B200GS_MAX_VIEWS][PACK_WARPS];     // global row (within the block of `cap`) of the warp's first row
    __shared__ int s_tile;
    const int tid = threadIdx.x;
    const unsigned lane = tid & 31u, w = tid >> 5;
    if (tid == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int64_t i = int64_t(t) * PACK_THREADS + tid;
    const bool live = i < n;
    float p[3] = {0.f, 0.f, 0.f};
    double sc[3] = {1.0, 1.0, 1.0}, q[4] = {1.0, 0.0, 0.0, 0.0}, inv_qn;
    if (live) {
        p[0] = __ldg(means + 3 * i); p[1] = __ldg(means + 3 * i + 1); p[2] = __ldg(means + 3 * i + 2);
        load_scale_quat<true, double>(scales, quats, i, sc, q, &inv_qn);
    }
    Proj<double> g3;
    gaussian_cov3d<double>(sc, q, vp.v[0].scale_modifier, g3);      // once per Gaussian; project_one_view per camera
    unsigned vismask = 0;
    unsigned long long kpos = 0;            // 8 bits per camera: this lane's rank among the warp's visible lanes
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        ProjVals pv;
        bool vis = false;
        if (live) vis = project_one_view<true, true>(vp.v[j], raw, i, 0, p, g3, nullptr, pv);
        const unsigned b = __ballot_sync(0xffffffffu, vis);
        const int k = __popc(b & ((1u << lane) - 1u));
        if (lane == 0) s_cnt[j][w] = __popc(b);
        if (live) {
            const int64_t o = int64_t(j) * n + i;
            xy_out[o] = make_float2(pv.px, pv.py);
            radii_out[o] = pv.radius;
        }
        if (vis) {
            vismask |= 1u << j;
            kpos |= (unsigned long long)k << (8 * j);
            float4* row = s_rows + (size_t(j) * PACK_THREADS + w * 32 + k) * 3;
            row[0] = make_float4(pv.px, pv.py, pv.depth, pv.cA);
            row[1] = make_float4(pv.cB, pv.cC, pv.comp, pv.opac);
            row[2].w = __int_as_float(pv.radius);
        }
    }
    float sh[MC * 3];
    if (vismask) {
        const int deg = vp.v[0].sh_degree;
        load_sh_any<true, MC>(shs_dc, raw.shs_rest, i, vp.v[0].sh_stride, (deg + 1) * (deg + 1), sh);
    }
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        uint8_t cl = 0;
        if ((vismask >> j) & 1u) {
            float r, gc, bc;
            sh_color_one<MC>(vp.v[j], p, sh, r, gc, bc, cl);
            float* row2 = reinterpret_cast<float*>(s_rows + (size_t(j) * PACK_THREADS + w * 32 + (int)((kpos >> (8 * j)) & 255ull)) * 3 + 2);
            row2[0] = r; row2[1] = gc; row2[2] = bc;
        }
        if (live) clamped_out[int64_t(j) * n + i] = cl;
    }
    __syncthreads();
    // warp j: camera j's block total -> chained scan over the blocks -> first row of every warp's run
    if ((int)w < nviews) {
        const int j = (int)w;
        const int c = (lane < PACK_WARPS) ? s_cnt[j][lane] : 0;
        int inc = c;
#pragma unroll
        for (int o = 1; o < PACK_WARPS; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)lane >= o) inc += v;
        }
        const int total = __shfl_sync(0xffffffffu, inc, PACK_WARPS - 1);
        const uint32_t base = sweep::chained_exclusive(scan_state + size_t(j) * gridDim.x, t, (uint32_t)total);
        if (lane < PACK_WARPS) s_pre[j][lane] = base + (uint32_t)(inc - c);
        if (lane == 0 && t == (int)gridDim.x - 1) d_count[j] = (int64_t)base + total;
    }
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        if (live) {
            int32_t ri = -1;
            if ((vismask >> j) & 1u) {
                const int64_t pos = (int64_t)s_pre[j][w] + (int64_t)((kpos >> (8 * j)) & 255ull);
                ri = pos < cap ? (int32_t)(int64_t(j) * cap + pos) : -1;
            }
            row_index_out[int64_t(j) * n + i] = ri;
        }
        // copy-out: 8 warps x 32 slots x 3 float4 per camera; consecutive threads -> consecutive 16-byte pieces of a warp's run
        float4* out = reinterpret_cast<float4*>(dst.p[j]);
        const float4* src = s_rows + size_t(j) * PACK_THREADS * 3;
#pragma unroll
        for (int it = 0; it < 3; ++it) {
            const int item = it * PACK_THREADS + tid;       // = (warp segment * 32 + r) * 3 + part
            const int seg = item / 96, r = (item - seg * 96) / 3, part = item - seg * 96 - r * 3;
            if (r < s_cnt[j][seg]) {
                const int64_t pos = (int64_t)s_pre[j][seg] + r;
                if (pos < cap) out[pos * 3 + part] = src[(seg * 32 + r) * 3 + part];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------------
constexpr int BWD_THREADS = 128;

// Cotangents of one view's projection outputs for one Gaussian
struct ProjCot {
    float vA, vB, vC;      // dL/dconic
    float2 vxy;            // dL/dmean2D (vanilla: NDC-scaled units)
    float vdepth;          // dL/ddepth (gsplat)
    float vcomp;           // dL/dcompensation (gsplat), incl. the part that reaches it through the blend opacity
};

// Adds view v's contribution to dL/dmean (dm), dL/dM-chain outputs: dL/dscale (activated scale, before the exp chain) and dL/dq
// (unit quaternion, before the normalisation chain).  g = project_geometry<GSPLAT, float>(v, p, sc, q).
template <bool GSPLAT>
__device__ __forceinline__ void geometry_backward(const B200gsView& v, const float* p, const Proj<float>& g, const ProjCot& c, float* dm,
                                                  float* dscale, float4& dq) {
    const float* V = v.viewmatrix;
    float dtx = 0.f, dty = 0.f, dtz = 0.f;  // dL/dt (camera)
    // ---- conic (+ compensation) -> blurred cov2D (a, b, c) ----------------------------------------------------
    const float inv_det = 1.0f / g.det;
    const float A = g.c * inv_det, B = -g.b * inv_det, C = g.a * inv_det;
    // X = -Q G Q, Q = [[A,B],[B,C]], G = [[vA, vB/2],[vB/2, vC]]
    const float hB = 0.5f * c.vB;
    const float m00 = A * c.vA + B * hB, m01 = A * hB + B * c.vC;
    const float m10 = B * c.vA + C * hB, m11 = B * hB + C * c.vC;
    float da = -(m00 * A + m01 * B);
    float db = -2.0f * (m00 * B + m01 * C);
    float dc = -(m10 * B + m11 * C);
    if (GSPLAT) {
        const float vc = c.vcomp;
        if (g.det0 > 0.f && vc != 0.f) {
            const float comp = sqrtf(g.det0 * inv_det);
            const float d_det0 = vc * 0.5f * comp / g.det0;
            const float d_det = -vc * 0.5f * comp * inv_det;
            da += d_det0 * g.c0 + d_det * g.c;
            dc += d_det0 * g.a0 + d_det * g.a;
            db += -2.0f * g.b * (d_det0 + d_det);
        }
    }
    // symmetric gradient wrt the 2x2 cov: [[da, db/2],[db/2, dc]]
    const float g00 = da, g01 = 0.5f * db, g11 = dc;
    const float* T = g.T;
    // dL/dSigma3 = T^T Gc T  (symmetric 3x3)
    float dS[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cidx = 0; cidx < 3; ++cidx)
            dS[r * 3 + cidx] = T[r] * (g00 * T[cidx] + g01 * T[3 + cidx]) + T[3 + r] * (g01 * T[cidx] + g11 * T[3 + cidx]);
    // dL/dT = 2 Gc T Sigma3 (2x3)
    const float* S = g.S3;
    const float Sf[9] = {S[0], S[1], S[2], S[1], S[3], S[4], S[2], S[4], S[5]};
    float TS0[3], TS1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        TS0[k] = T[0] * Sf[k] + T[1] * Sf[3 + k] + T[2] * Sf[6 + k];
        TS1[k] = T[3] * Sf[k] + T[4] * Sf[3 + k] + T[5] * Sf[6 + k];
    }
    float dT0[3], dT1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        dT0[k] = 2.0f * (g00 * TS0[k] + g01 * TS1[k]);
        dT1[k] = 2.0f * (g01 * TS0[k] + g11 * TS1[k]);
    }
    // T = J Rw -> dL/dJ = dL/dT Rw^T ; Rw[j][i] = V[i*4+j]
    const float dJ00 = dT0[0] * V[0] + dT0[1] * V[4] + dT0[2] * V[8];
    const float dJ02 = dT0[0] * V[2] + dT0[1] * V[6] + dT0[2] * V[10];
    const float dJ11 = dT1[0] * V[1] + dT1[1] * V[5] + dT1[2] * V[9];
    const float dJ12 = dT1[0] * V[2] + dT1[1] * V[6] + dT1[2] * V[10];
    const float itz = 1.0f / g.tz, itz2 = itz * itz, itz3 = itz2 * itz;
    const float dcx = -g.fx * itz2 * dJ02;  // dL/d(tx')
    const float dcy = -g.fy * itz2 * dJ12;
    dtz += -g.fx * itz2 * dJ00 - g.fy * itz2 * dJ11 + 2.0f * g.fx * g.cxp * itz3 * dJ02 + 2.0f * g.fy * g.cyp * itz3 * dJ12;
    if (!g.clx) dtx += dcx; else if (GSPLAT) dtz += dcx * g.cxp * itz;  // dgr drops the clamped branch's z-dependence
    if (!g.cly) dty += dcy; else if (GSPLAT) dtz += dcy * g.cyp * itz;

    // ---- mean2D / depth --------------------------------------------------------------------------------------
    if (GSPLAT) {
        const float iz = 1.0f / (g.tz + 1e-6f);
        dtx += v.fx * iz * c.vxy.x;
        dty += v.fy * iz * c.vxy.y;
        dtz += (-v.fx * g.tx * iz * iz + v.cx * 1e-6f * iz * iz) * c.vxy.x + (-v.fy * g.ty * iz * iz + v.cy * 1e-6f * iz * iz) * c.vxy.y;
        dtz += c.vdepth;
    } else {
        // v_xy is dL/d(ndc) (pixel gradient x 0.5 W/H), straight through the 4x4 full projection
        const float* P = v.projmatrix;
        const float hw = p[0] * P[3] + p[1] * P[7] + p[2] * P[11] + P[15];
        const float mw = 1.0f / (hw + 0.0000001f);
        const float mul1 = (p[0] * P[0] + p[1] * P[4] + p[2] * P[8] + P[12]) * mw * mw;
        const float mul2 = (p[0] * P[1] + p[1] * P[5] + p[2] * P[9] + P[13]) * mw * mw;
        dm[0] += (P[0] * mw - P[3] * mul1) * c.vxy.x + (P[1] * mw - P[3] * mul2) * c.vxy.y;
        dm[1] += (P[4] * mw - P[7] * mul1) * c.vxy.x + (P[5] * mw - P[7] * mul2) * c.vxy.y;
        dm[2] += (P[8] * mw - P[11] * mul1) * c.vxy.x + (P[9] * mw - P[11] * mul2) * c.vxy.y;
    }
    // t = p * V[:3,:3] + V[3,:3]  ->  dL/dp_i = sum_j V[i][j] dt_j
    dm[0] += V[0] * dtx + V[1] * dty + V[2] * dtz;
    dm[1] += V[4] * dtx + V[5] * dty + V[6] * dtz;
    dm[2] += V[8] * dtx + V[9] * dty + V[10] * dtz;

    // ---- Sigma3 = M M^T, M = R diag(s) ------------------------------------------------------------------------
    float M[9], dM[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k) M[r * 3 + k] = g.Rm[r * 3 + k] * g.s[k];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k)
            dM[r * 3 + k] = 2.0f * (dS[r * 3 + 0] * M[0 + k] + dS[r * 3 + 1] * M[3 + k] + dS[r * 3 + 2] * M[6 + k]);
    float dR[9];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        dscale[k] += v.scale_modifier * (g.Rm[k] * dM[k] + g.Rm[3 + k] * dM[3 + k] + g.Rm[6 + k] * dM[6 + k]);
#pragma unroll
        for (int r = 0; r < 3; ++r) dR[r * 3 + k] = dM[r * 3 + k] * g.s[k];
    }
    // Rm was built from the (unit) quaternion (r, x, y, z): recover it from the caller
    const float r = g.qr, x = g.qx, y = g.qy, z = g.qz;
    dq.x += 2.f * (-z * dR[1] + y * dR[2] + z * dR[3] - x * dR[5] - y * dR[6] + x * dR[7]);
    dq.y += 2.f * (y * dR[1] + z * dR[2] + y * dR[3] - 2.f * x * dR[4] - r * dR[5] + z * dR[6] + r * dR[7] - 2.f * x * dR[8]);
    dq.z += 2.f * (-2.f * y * dR[0] + x * dR[1] + r * dR[2] + x * dR[3] + z * dR[5] - r * dR[6] + z * dR[7] - 2.f * y * dR[8]);
    dq.w += 2.f * (-2.f * z * dR[0] - r * dR[1] + x * dR[2] + r * dR[3] - 2.f * z * dR[4] + y * dR[5] + x * dR[6] + y * dR[7]);
}

// SH-gradient rows of a warp's 32 Gaussians: staged in shared memory (odd row stride: conflict-free) and written back with
// fully coalesced 128-bit stores: every row must be written (zeros for culled Gaussians), so the warp's 32 rows are one
// contiguous 5.6-6 KB span of the output.  out[] holds this lane's 48 values (dc first); RAW: dc goes to v_shs, rest to dst_base.
// second half of store_sh_rows: the warp's staged rows (row of lane l at s_rows_warp + l * (rw | 1)) -> global memory, coalesced
template <bool RAW>
__device__ __forceinline__ void flush_sh_rows(const float* s_rows_warp, int rw, int64_t i, int64_t n, unsigned lane, float* __restrict__ dst_base,
                                              bool ACC) {
    const int rwp = rw | 1;
    __syncwarp();
    const int64_t i0 = i - lane;
    const int rows_valid = (i0 < n) ? (int)min((int64_t)32, n - i0) : 0;
    const int total = rows_valid * rw;
    float* dst = dst_base + i0 * rw;
    const float* sw = s_rows_warp;
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        for (int idx = lane; idx * 4 + 3 < total; idx += 32) {
            int f = idx * 4, r = f / rw, c = f - r * rw;
            float t[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                t[e] = sw[r * rwp + c];
                if (++c == rw) { c = 0; ++r; }
            }
            if (ACC) {
                const float4 old = reinterpret_cast<const float4*>(dst)[idx];
                t[0] += old.x; t[1] += old.y; t[2] += old.z; t[3] += old.w;
            }
            reinterpret_cast<float4*>(dst)[idx] = make_float4(t[0], t[1], t[2], t[3]);
        }
        for (int f = (total & ~3) + lane; f < total; f += 32) dst[f] = sw[(f / rw) * rwp + f % rw] + (ACC ? dst[f] : 0.f);
    } else {
        for (int f = lane; f < total; f += 32) dst[f] = sw[(f / rw) * rwp + f % rw] + (ACC ? dst[f] : 0.f);
    }
}

template <bool RAW, int MC>
__device__ __forceinline__ void store_sh_rows(float* s_rows_warp, const float* out, int64_t i, int64_t n, bool in_range, int stride3, unsigned lane,
                                              float* __restrict__ v_shs, float* __restrict__ v_shs_rest, bool ACC) {
    const int rw = RAW ? stride3 - 3 : stride3;          // floats per output row
    float* dst_base = RAW ? v_shs_rest : v_shs;
    if (RAW && in_range) {
        float o0 = out[0], o1 = out[1], o2 = out[2];
        if (ACC) { o0 += v_shs[3 * i]; o1 += v_shs[3 * i + 1]; o2 += v_shs[3 * i + 2]; }
        v_shs[3 * i] = o0; v_shs[3 * i + 1] = o1; v_shs[3 * i + 2] = o2;
    }
    if (rw <= MC * 3) {
        const int rwp = rw | 1;
        float* row = s_rows_warp + lane * rwp;
#pragma unroll
        for (int k = 0; k < MC * 3; ++k) {
            const int c = RAW ? k - 3 : k;
            if (c >= 0 && c < rw) row[c] = out[k];
        }
        flush_sh_rows<RAW>(s_rows_warp, rw, i, n, lane, dst_base, ACC);
    } else if (in_range) {  // wider coefficient storage than the kernel evaluates: plain per-thread rows
        float* o = dst_base + i * int64_t(rw);
#pragma unroll
        for (int k = RAW ? 3 : 0; k < MC * 3; ++k) o[RAW ? k - 3 : k] = out[k];
        for (int c = MC * 3 - (RAW ? 3 : 0); c < rw; ++c) o[c] = 0.f;
    }
}

template <bool GSPLAT, bool RAW, int MC>
__global__ void __launch_bounds__(BWD_THREADS, (MC <= 16 ? (GSPLAT ? 7 : 6) : 3)) project_bwd_kernel(const __grid_constant__ B200gsView v, const RawIO raw, int64_t n,
                                                          const float* __restrict__ means, const float* __restrict__ scales,
                                                          const float* __restrict__ quats, const float* __restrict__ shs,
                                                          const int32_t* __restrict__ radii, const uint8_t* __restrict__ clamped,
                                                          const float2* __restrict__ v_xy, const float* __restrict__ v_depth,
                                                          const float* __restrict__ v_conic, const float* __restrict__ v_comp,
                                                          const float* __restrict__ v_rgb, float* __restrict__ v_means,
                                                          float* __restrict__ v_scales, float4* __restrict__ v_quats,
                                                          float* __restrict__ v_shs) {
    __shared__ float s_rows[BWD_THREADS / 32][32 * (MC * 3 + 1)];
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const int warp = threadIdx.x >> 5;
    const bool in_range = i < n;
    const bool ROWS = RAW && (raw.v_rows != nullptr);
    const bool ACC = RAW && (raw.accumulate != 0);
    // a negative row index = the entry did not fit its fixed-size block (the caller redoes such a step): treated as culled
    const int64_t ri = (ROWS && in_range) ? (raw.row_offsets ? int64_t(raw.row_offsets[i]) : i) : 0;   // NULL offsets: row i
    const bool vis = in_range && (radii[i] > 0) && !(ROWS && ri < 0);
    const int stride3 = v.sh_stride * 3;
    float p[3] = {0.f, 0.f, 0.f};
    if (vis) { p[0] = __ldg(means + 3 * i); p[1] = __ldg(means + 3 * i + 1); p[2] = __ldg(means + 3 * i + 2); }
    const float* vrow = (ROWS && vis) ? raw.v_rows + ri * B200GS_ROW_FLOATS : nullptr;

    float dm[3] = {0.f, 0.f, 0.f};  // dL/dmean (world)

    // ---- SH colour -------------------------------------------------------------------------------------------
    if (v_shs != nullptr) {
        const int deg = v.sh_degree;
        const int ncoef = (deg + 1) * (deg + 1);
        float gr = 0.f, gg = 0.f, gb = 0.f, dx = 0.f, dy = 0.f, dz = 1.f, inv_len = 0.f;
        float bs[MC];
#pragma unroll
        for (int k = 0; k < MC; ++k) bs[k] = 0.f;
        if (vis) {
            const uint8_t cl = clamped[i];
            const float* crgb = ROWS ? vrow + B200GS_ROW_RGB : v_rgb + 3 * i;
            gr = (cl & 1) ? 0.f : __ldg(crgb + 0);
            gg = (cl & 2) ? 0.f : __ldg(crgb + 1);
            gb = (cl & 4) ? 0.f : __ldg(crgb + 2);
            view_dir(p, v.campos, dx, dy, dz, inv_len);
            sh_basis<MC>(deg, dx, dy, dz, bs);
        }
        if (vis && !GSPLAT && deg > 0) {
            // view direction -> mean (dgr back-propagates it; gsplat renderers detach the direction)
            // w_k = <sh_k, v_rgb> first (the 48 coefficients are consumed as they arrive: 16 live values instead of 48), then the basis
            // derivatives
            const float* c0 = RAW ? raw.shs_rest + i * int64_t(v.sh_stride - 1) * 3 - 3 : shs + i * int64_t(v.sh_stride) * 3;   // coefficient k at c0 + 3 k (k >= 1)
            float w[MC];
#pragma unroll
            for (int k = 1; k < MC; ++k) w[k] = (k < ncoef) ? __ldg(c0 + 3 * k) * gr + __ldg(c0 + 3 * k + 1) * gg + __ldg(c0 + 3 * k + 2) * gb : 0.f;
            float bx[MC], by[MC], bz[MC];
            sh_basis_grad<MC>(deg, dx, dy, dz, bx, by, bz);
            float ddx = 0.f, ddy = 0.f, ddz = 0.f;
#pragma unroll
            for (int k = 1; k < MC; ++k) {
                if (k < ncoef) { ddx += bx[k] * w[k]; ddy += by[k] * w[k]; ddz += bz[k] * w[k]; }
            }
            const float dot = dx * ddx + dy * ddy + dz * ddz;
            dm[0] += (ddx - dx * dot) * inv_len;
            dm[1] += (ddy - dy * dot) * inv_len;
            dm[2] += (ddz - dz * dot) * inv_len;
        }
        // SH-gradient row of this Gaussian (coefficient k, channel c: basis_k * v_rgb_c; zeros when culled) straight into the warp's
        // staging rows — 48 values that used to sit in registers until the store (96 registers, 5 blocks per SM) — then out coalesced
        const int rw = RAW ? stride3 - 3 : stride3;          // floats per output row
        if (rw <= MC * 3) {
            if (RAW && in_range) {
                float o0 = bs[0] * gr, o1 = bs[0] * gg, o2 = bs[0] * gb;
                if (ACC) { o0 += v_shs[3 * i]; o1 += v_shs[3 * i + 1]; o2 += v_shs[3 * i + 2]; }
                v_shs[3 * i] = o0; v_shs[3 * i + 1] = o1; v_shs[3 * i + 2] = o2;
            }
            float* row = s_rows[warp] + lane * (rw | 1);
#pragma unroll
            for (int k = RAW ? 1 : 0; k < MC; ++k) {
                const int c = RAW ? 3 * k - 3 : 3 * k;
                if (c < rw) {
                    const float bk = (k < ncoef) ? bs[k] : 0.f;
                    row[c] = bk * gr; row[c + 1] = bk * gg; row[c + 2] = bk * gb;
                }
            }
            flush_sh_rows<RAW>(s_rows[warp], rw, i, n, lane, RAW ? raw.v_shs_rest : v_shs, ACC);
        } else {   // wider coefficient storage than the kernel evaluates: the register path of store_sh_rows
            float out[MC * 3];
#pragma unroll
            for (int k = 0; k < MC; ++k) {
                const float bk = (k < ncoef) ? bs[k] : 0.f;
                out[3 * k + 0] = bk * gr; out[3 * k + 1] = bk * gg; out[3 * k + 2] = bk * gb;
            }
            store_sh_rows<RAW, MC>(s_rows[warp], out, i, n, in_range, stride3, lane, v_shs, raw.v_shs_rest, ACC);
        }
    }
    if (!in_range) return;
    if (RAW && raw.v_mean2d != nullptr) {
        float* m2 = raw.v_mean2d + i * raw.v_mean2d_cols;
        m2[0] = (ROWS && vis) ? __ldg(vrow) : 0.f;
        m2[1] = (ROWS && vis) ? __ldg(vrow + 1) : 0.f;
        if (raw.v_mean2d_cols > 2) m2[2] = 0.f;
    }
    if (!vis) {
        if (!ACC) {
            v_means[3 * i] = 0.f; v_means[3 * i + 1] = 0.f; v_means[3 * i + 2] = 0.f;
            v_scales[3 * i] = 0.f; v_scales[3 * i + 1] = 0.f; v_scales[3 * i + 2] = 0.f;
            v_quats[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (RAW) raw.v_opac_logit[i] = 0.f;
        }
        return;
    }
    float sc[3], q[4], inv_qn;
    load_scale_quat<RAW, float>(scales, quats, i, sc, q, &inv_qn);
    Proj<float> g;
    project_geometry<GSPLAT, float>(v, p, sc, q, g);
    g.qr = q[0]; g.qx = q[1]; g.qy = q[2]; g.qz = q[3];

    ProjCot c;
    const float* ccon = ROWS ? vrow + B200GS_ROW_CONIC : v_conic + 3 * i;
    c.vA = __ldg(ccon); c.vB = __ldg(ccon + 1); c.vC = __ldg(ccon + 2);
    c.vxy = ROWS ? make_float2(__ldg(vrow), __ldg(vrow + 1)) : v_xy[i];
    c.vdepth = 0.f;
    if (GSPLAT) c.vdepth = ROWS ? __ldg(vrow + B200GS_ROW_DEPTH) : (v_depth ? __ldg(v_depth + i) : 0.f);
    c.vcomp = (GSPLAT && v_comp != nullptr) ? __ldg(v_comp + i) : 0.f;
    if (RAW) {
        // blend opacity = sigmoid(logit) [* compensation]: split dL/d(opac_out) between the logit and the compensation
        const float o = 1.0f / (1.0f + expf(-__ldg(raw.opac_in + i)));
        const float vo = ROWS ? __ldg(vrow + B200GS_ROW_OPACITY) : __ldg(raw.v_opac + i);
        float v_sig = vo;
        if (GSPLAT && raw.anti_aliased) {
            const float comp = sqrtf(fmaxf(g.det0 / g.det, 0.f));
            v_sig = vo * comp;
            c.vcomp += vo * o;
        }
        raw.v_opac_logit[i] = v_sig * o * (1.0f - o) + (ACC ? raw.v_opac_logit[i] : 0.f);
    }
    float dscale[3] = {0.f, 0.f, 0.f};
    float4 dq = make_float4(0.f, 0.f, 0.f, 0.f);
    geometry_backward<GSPLAT>(v, p, g, c, dm, dscale, dq);

    if (ACC) { dm[0] += v_means[3 * i]; dm[1] += v_means[3 * i + 1]; dm[2] += v_means[3 * i + 2]; }
    v_means[3 * i] = dm[0]; v_means[3 * i + 1] = dm[1]; v_means[3 * i + 2] = dm[2];
#pragma unroll
    for (int k = 0; k < 3; ++k) v_scales[3 * i + k] = (RAW ? dscale[k] * sc[k] : dscale[k]) + (ACC ? v_scales[3 * i + k] : 0.f);   // d exp(x) = exp(x)
    if (RAW) {  // through q / |q|
        const float dot = dq.x * q[0] + dq.y * q[1] + dq.z * q[2] + dq.w * q[3];
        dq.x = (dq.x - q[0] * dot) * inv_qn; dq.y = (dq.y - q[1] * dot) * inv_qn;
        dq.z = (dq.z - q[2] * dot) * inv_qn; dq.w = (dq.w - q[3] * dot) * inv_qn;
    }
    if (ACC) {
        const float4 old = v_quats[i];
        dq.x += old.x; dq.y += old.y; dq.z += old.z; dq.w += old.w;
    }
    v_quats[i] = dq;
}

// Backward of project_fwd_multi_kernel: every thread walks the W cameras of the step, accumulates the parameter gradients of
// its Gaussian in registers and writes them ONCE (the per-camera launches read-modify-wrote 236 B per Gaussian and camera).
// Cotangents are [.,12] gradient rows (b200gs.h row layout); view j's rows start at v_rows[j] (possibly a peer GPU's buffer
// mapped over NVLink), entry (j, i) uses row row_index[j*n + i] of it.
struct RowSources {
    const float* rows[B200GS_MAX_VIEWS];
};

template <int MC>
__global__ void __launch_bounds__(BWD_THREADS) project_bwd_multi_kernel(const __grid_constant__ ViewPack vp, int nviews, const RawIO raw,
                                                                       const __grid_constant__ RowSources src, int64_t n,
                                                                       const float* __restrict__ means, const float* __restrict__ scales,
                                                                       const float* __restrict__ quats, const int32_t* __restrict__ radii,
                                                                       const uint8_t* __restrict__ clamped, const int32_t* __restrict__ row_index,
                                                                       float* __restrict__ v_means, float* __restrict__ v_scales,
                                                                       float4* __restrict__ v_quats, float* __restrict__ v_shs_dc) {
    __shared__ float s_rows[BWD_THREADS / 32][32 * (MC * 3 + 1)];
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const int warp = threadIdx.x >> 5;
    const bool in_range = i < n;
    const int stride3 = vp.v[0].sh_stride * 3;
    const int deg = vp.v[0].sh_degree;
    const int ncoef = (deg + 1) * (deg + 1);
    // SH-gradient accumulators over the cameras: the dc coefficient in registers, the rest in this lane's row of the staging buffer
    // (48 accumulator registers kept the kernel at 183 registers = 8 warps per SM); rows wider than the buffer keep the register path
    const int rw = stride3 - 3;                      // <= MC * 3: the launcher picks MC by the storage width
    float* my_row = s_rows[warp] + lane * (rw | 1);
    float dc_acc[3] = {0.f, 0.f, 0.f};
    for (int c = 0; c < rw; ++c) my_row[c] = 0.f;
    float dm[3] = {0.f, 0.f, 0.f}, dscale[3] = {0.f, 0.f, 0.f}, dlogit = 0.f;
    float4 dq = make_float4(0.f, 0.f, 0.f, 0.f);
    float p[3] = {0.f, 0.f, 0.f}, sc[3] = {1.f, 1.f, 1.f}, q[4] = {1.f, 0.f, 0.f, 0.f}, inv_qn = 1.f, o = 0.f;
    bool loaded = false;
    Proj<float> g;
#pragma unroll 1
    for (int j = 0; j < nviews; ++j) {
        const int64_t e = int64_t(j) * n + i;
        if (!in_range || radii[e] <= 0) continue;
        const int ri = row_index[e];
        if (ri < 0) continue;     // did not fit its fixed-size block: the caller redoes such a step
        const float* vrow = src.rows[j] + int64_t(ri) * B200GS_ROW_FLOATS;
        const float4 w0 = *reinterpret_cast<const float4*>(vrow), w1 = *reinterpret_cast<const float4*>(vrow + 4),
                     w2 = *reinterpret_cast<const float4*>(vrow + 8);
        if (!loaded) {
            p[0] = __ldg(means + 3 * i); p[1] = __ldg(means + 3 * i + 1); p[2] = __ldg(means + 3 * i + 2);
            load_scale_quat<true, float>(scales, quats, i, sc, q, &inv_qn);
            o = 1.0f / (1.0f + expf(-__ldg(raw.opac_in + i)));
            gaussian_cov3d<float>(sc, q, vp.v[0].scale_modifier, g);      // once per Gaussian; project_view per camera
            g.qr = q[0]; g.qx = q[1]; g.qy = q[2]; g.qz = q[3];
            loaded = true;
        }
        const B200gsView& v = vp.v[j];
        // SH colour
        {
            const uint8_t cl = clamped[e];
            const float gr = (cl & 1) ? 0.f : w2.x, gg = (cl & 2) ? 0.f : w2.y, gb = (cl & 4) ? 0.f : w2.z;
            float dx, dy, dz, inv_len;
            view_dir(p, v.campos, dx, dy, dz, inv_len);
            float bs[MC];
            sh_basis<MC>(deg, dx, dy, dz, bs);
            dc_acc[0] = fmaf(bs[0], gr, dc_acc[0]); dc_acc[1] = fmaf(bs[0], gg, dc_acc[1]); dc_acc[2] = fmaf(bs[0], gb, dc_acc[2]);
#pragma unroll
            for (int k = 1; k < MC; ++k) {
                if (k < ncoef && 3 * k < rw + 3) {
                    float* a = my_row + 3 * k - 3;
                    a[0] = fmaf(bs[k], gr, a[0]); a[1] = fmaf(bs[k], gg, a[1]); a[2] = fmaf(bs[k], gb, a[2]);
                }
            }
        }
        project_view<true, float>(v, p, g);
        ProjCot c;
        c.vxy = make_float2(w0.x, w0.y);
        c.vdepth = w0.z;
        c.vA = w0.w; c.vB = w1.x; c.vC = w1.y;
        c.vcomp = 0.f;
        const float vo = w1.w;
        float v_sig = vo;
        if (raw.anti_aliased) {
            const float comp = sqrtf(fmaxf(g.det0 / g.det, 0.f));
            v_sig = vo * comp;
            c.vcomp = vo * o;
        }
        dlogit += v_sig * o * (1.0f - o);
        geometry_backward<true>(v, p, g, c, dm, dscale, dq);
    }
    if (in_range) { v_shs_dc[3 * i] = dc_acc[0]; v_shs_dc[3 * i + 1] = dc_acc[1]; v_shs_dc[3 * i + 2] = dc_acc[2]; }
    flush_sh_rows<true>(s_rows[warp], rw, i, n, lane, raw.v_shs_rest, false);
    if (!in_range) return;
    v_means[3 * i] = dm[0]; v_means[3 * i + 1] = dm[1]; v_means[3 * i + 2] = dm[2];
#pragma unroll
    for (int k = 0; k < 3; ++k) v_scales[3 * i + k] = dscale[k] * sc[k];
    const float dot = dq.x * q[0] + dq.y * q[1] + dq.z * q[2] + dq.w * q[3];
    v_quats[i] = make_float4((dq.x - q[0] * dot) * inv_qn, (dq.y - q[1] * dot) * inv_qn, (dq.z - q[2] * dot) * inv_qn, (dq.w - q[3] * dot) * inv_qn);
    raw.v_opac_logit[i] = dlogit;
}

// ------------------------------------------------------------------------------------------------------------------
// standalone SH (gsplat.sh.spherical_harmonics)
// ------------------------------------------------------------------------------------------------------------------
template <int MC>
__global__ void __launch_bounds__(256) sh_fwd_kernel(int deg, int stride, int64_t n, const float* __restrict__ dirs,
                                                     const float* __restrict__ coeffs, float* __restrict__ rgb) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int ncoef = (deg + 1) * (deg + 1);
    float dx = __ldg(dirs + 3 * i), dy = __ldg(dirs + 3 * i + 1), dz = __ldg(dirs + 3 * i + 2);
    const float inv_len = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
    dx *= inv_len; dy *= inv_len; dz *= inv_len;
    float sh[MC * 3];
    load_sh<MC>(coeffs + i * int64_t(stride) * 3, ncoef, ((stride * 3) & 3) == 0, sh);
    float bs[MC];
    sh_basis<MC>(deg, dx, dy, dz, bs);
    float r = 0.f, g = 0.f, b = 0.f;
#pragma unroll
    for (int k = 0; k < MC; ++k)
        if (k < ncoef) { r += bs[k] * sh[3 * k]; g += bs[k] * sh[3 * k + 1]; b += bs[k] * sh[3 * k + 2]; }
    rgb[3 * i] = r; rgb[3 * i + 1] = g; rgb[3 * i + 2] = b;
}

template <int MC>
__global__ void __launch_bounds__(256) sh_bwd_kernel(int deg, int stride, int64_t n, const float* __restrict__ dirs,
                                                     const float* __restrict__ coeffs, const float* __restrict__ v_rgb,
                                                     float* __restrict__ v_coeffs, float* __restrict__ v_dirs) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int ncoef = (deg + 1) * (deg + 1);
    const int stride3 = stride * 3;
    const bool vec4 = (stride3 & 3) == 0;
    float dx = __ldg(dirs + 3 * i), dy = __ldg(dirs + 3 * i + 1), dz = __ldg(dirs + 3 * i + 2);
    const float inv_len = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);
    dx *= inv_len; dy *= inv_len; dz *= inv_len;
    const float gr = __ldg(v_rgb + 3 * i), gg = __ldg(v_rgb + 3 * i + 1), gb = __ldg(v_rgb + 3 * i + 2);
    float bs[MC];
    sh_basis<MC>(deg, dx, dy, dz, bs);
    float* o = v_coeffs + i * int64_t(stride3);
    for (int k = 0; k < stride; ++k) {
        const float bk = (k < ncoef) ? bs[k] : 0.f;
        o[3 * k] = bk * gr; o[3 * k + 1] = bk * gg; o[3 * k + 2] = bk * gb;
    }
    if (v_dirs != nullptr) {
        float ddx = 0.f, ddy = 0.f, ddz = 0.f;
        if (deg > 0) {
            float sh[MC * 3];
            load_sh<MC>(coeffs + i * int64_t(stride3), ncoef, vec4, sh);
            float bx[MC], by[MC], bz[MC];
            sh_basis_grad<MC>(deg, dx, dy, dz, bx, by, bz);
#pragma unroll
            for (int k = 1; k < MC; ++k)
                if (k < ncoef) {
                    const float w = sh[3 * k] * gr + sh[3 * k + 1] * gg + sh[3 * k + 2] * gb;
                    ddx += bx[k] * w; ddy += by[k] * w; ddz += bz[k] * w;
                }
            const float dot = dx * ddx + dy * ddy + dz * ddz;
            ddx = (ddx - dx * dot) * inv_len; ddy = (ddy - dy * dot) * inv_len; ddz = (ddz - dz * dot) * inv_len;
        }
        v_dirs[3 * i] = ddx; v_dirs[3 * i + 1] = ddy; v_dirs[3 * i + 2] = ddz;
    }
}

}  // namespace

int launch_project_fwd(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, float* xy, float* depth, int32_t* radii, float* conic, float* comp,
                       int32_t* tiles, float* cov3d, float* rgb, uint8_t* clamped, cudaStream_t s) {
    return launch_project_fwd_raw(v, n, means, scales, quats, nullptr, shs, nullptr, 0, xy, depth, radii, conic, comp, tiles, cov3d,
                                  rgb, clamped, nullptr, s, nullptr);
}

int launch_project_fwd_raw(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                           const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy,
                           float* depth, int32_t* radii, float* conic, float* comp, int32_t* tiles, float* cov3d, float* rgb,
                           uint8_t* clamped, float* opac_out, cudaStream_t s, float* rows) {
    if (n == 0) return B200GS_OK;
    const int threads = 256;
    const unsigned blocks = (unsigned)div_up64(n, threads);
    const bool raw_mode = opac_out != nullptr || rows != nullptr;
    RawIO raw{opac_logits, shs_rest, opac_out, nullptr, nullptr, nullptr, anti_aliased, nullptr, nullptr, 0};
#define B200GS_PF_ARGS v, raw, n, means, scales, quats, shs_dc, (float2*)xy, depth, radii, conic, comp, tiles, cov3d, rgb, clamped, rows
#define B200GS_PF_LAUNCH(MC)                                                                                    \
    do {                                                                                                         \
        if (v.mode == B200GS_MODE_GSPLAT) {                                                                      \
            if (raw_mode) project_fwd_kernel<true, true, MC><<<blocks, threads, 0, s>>>(B200GS_PF_ARGS);         \
            else project_fwd_kernel<true, false, MC><<<blocks, threads, 0, s>>>(B200GS_PF_ARGS);                 \
        } else {                                                                                                 \
            if (raw_mode) project_fwd_kernel<false, true, MC><<<blocks, threads, 0, s>>>(B200GS_PF_ARGS);        \
            else project_fwd_kernel<false, false, MC><<<blocks, threads, 0, s>>>(B200GS_PF_ARGS);                \
        }                                                                                                        \
    } while (0)
    if (shs_dc != nullptr && v.sh_degree > 3) B200GS_PF_LAUNCH(25);
    else B200GS_PF_LAUNCH(16);
#undef B200GS_PF_LAUNCH
#undef B200GS_PF_ARGS
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

int launch_project_bwd(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, const int32_t* radii, const uint8_t* clamped, const float* v_xy,
                       const float* v_depth, const float* v_conic, const float* v_comp, const float* v_rgb,
                       float* v_means, float* v_scales, float* v_quats, float* v_shs, cudaStream_t s) {
    return launch_project_bwd_raw(v, n, means, scales, quats, nullptr, shs, nullptr, 0, radii, clamped, v_xy, v_depth, v_conic,
                                  v_comp, v_rgb, nullptr, v_means, v_scales, v_quats, nullptr, v_shs, nullptr, s);
}

int launch_project_bwd_raw(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                           const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased,
                           const int32_t* radii, const uint8_t* clamped, const float* v_xy, const float* v_depth,
                           const float* v_conic, const float* v_comp, const float* v_rgb, const float* v_opac, float* v_means,
                           float* v_scales, float* v_quats, float* v_opac_logit, float* v_shs_dc, float* v_shs_rest,
                           cudaStream_t s, const float* v_rows, const int32_t* row_offsets, int accumulate, float* v_mean2d, int v_mean2d_cols) {
    if (n == 0) return B200GS_OK;
    const int threads = BWD_THREADS;
    const unsigned blocks = (unsigned)div_up64(n, threads);
    const bool raw_mode = v_opac_logit != nullptr;
    RawIO raw{opac_logits, shs_rest, nullptr, v_opac, v_opac_logit, v_shs_rest, anti_aliased, v_rows, row_offsets, accumulate, v_mean2d, v_mean2d_cols};
#define B200GS_PB_ARGS v, raw, n, means, scales, quats, shs_dc, radii, clamped, (const float2*)v_xy, v_depth, v_conic, v_comp, v_rgb, \
                       v_means, v_scales, (float4*)v_quats, v_shs_dc
#define B200GS_PB_LAUNCH(MC)                                                                                    \
    do {                                                                                                         \
        if (v.mode == B200GS_MODE_GSPLAT) {                                                                      \
            if (raw_mode) project_bwd_kernel<true, true, MC><<<blocks, threads, 0, s>>>(B200GS_PB_ARGS);         \
            else project_bwd_kernel<true, false, MC><<<blocks, threads, 0, s>>>(B200GS_PB_ARGS);                 \
        } else {                                                                                                 \
            if (raw_mode) project_bwd_kernel<false, true, MC><<<blocks, threads, 0, s>>>(B200GS_PB_ARGS);        \
            else project_bwd_kernel<false, false, MC><<<blocks, threads, 0, s>>>(B200GS_PB_ARGS);                \
        }                                                                                                        \
    } while (0)
    if (v_shs_dc != nullptr && v.sh_degree > 3) B200GS_PB_LAUNCH(25);
    else B200GS_PB_LAUNCH(16);
#undef B200GS_PB_LAUNCH
#undef B200GS_PB_ARGS
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

int launch_project_fwd_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                             const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy, float* depth,
                             int32_t* radii, float* conic, float* rgb, uint8_t* clamped, float* opac_out, cudaStream_t s) {
    if (n == 0 || n_views == 0) return B200GS_OK;
    ViewPack vp;
    for (int j = 0; j < n_views; ++j) vp.v[j] = views[j];
    for (int j = n_views; j < B200GS_MAX_VIEWS; ++j) vp.v[j] = views[0];
    RawIO raw{opac_logits, shs_rest, opac_out, nullptr, nullptr, nullptr, anti_aliased, nullptr, nullptr, 0};
    if (views[0].sh_degree > 3)
        project_fwd_multi_kernel<25><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(vp, n_views, raw, n, means, scales, quats, shs_dc, (float2*)xy, depth,
                                                                                radii, conic, rgb, clamped);
    else
        project_fwd_multi_kernel<16><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(vp, n_views, raw, n, means, scales, quats, shs_dc, (float2*)xy, depth,
                                                                                radii, conic, rgb, clamped);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

size_t project_pack_workspace_bytes(int n_views, int64_t n) {
    return 256 + (size_t)n_views * (size_t)div_up64(n > 0 ? n : 1, PACK_THREADS) * sizeof(uint32_t);
}

int launch_project_pack_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                              const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy, int32_t* radii,
                              uint8_t* clamped, int32_t* row_index, float* const* dst_rows, int64_t cap, void* workspace, size_t workspace_bytes,
                              int64_t* d_count, cudaStream_t s) {
    if (n_views == 0) return B200GS_OK;
    if (n == 0) {
        B200GS_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t) * (size_t)n_views, s));
        return B200GS_OK;
    }
    const size_t need = project_pack_workspace_bytes(n_views, n);
    if (workspace_bytes < need) {
        set_error("project_pack_multi: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return B200GS_EINVAL;
    }
    ViewPack vp;
    PackDst dst;
    for (int j = 0; j < B200GS_MAX_VIEWS; ++j) {
        vp.v[j] = views[j < n_views ? j : 0];
        dst.p[j] = j < n_views ? dst_rows[j] : nullptr;
    }
    RawIO raw{opac_logits, shs_rest, nullptr, nullptr, nullptr, nullptr, anti_aliased, nullptr, nullptr, 0};
    B200GS_CUDA(cudaMemsetAsync(workspace, 0, need, s));
    uint32_t* ticket = (uint32_t*)workspace;
    uint32_t* state = ticket + 64;
    const unsigned blocks = (unsigned)div_up64(n, PACK_THREADS);
    const size_t smem = (size_t)n_views * PACK_THREADS * 3 * sizeof(float4);
    static bool configured = false;         // raise the dynamic shared-memory limit once (8 cameras: 96 KB)
    if (!configured) {
        B200GS_CUDA(cudaFuncSetAttribute((const void*)project_pack_multi_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         B200GS_MAX_VIEWS * PACK_THREADS * 3 * (int)sizeof(float4)));
        B200GS_CUDA(cudaFuncSetAttribute((const void*)project_pack_multi_kernel<25>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         B200GS_MAX_VIEWS * PACK_THREADS * 3 * (int)sizeof(float4)));
        configured = true;
    }
    if (views[0].sh_degree > 3)
        project_pack_multi_kernel<25><<<blocks, PACK_THREADS, smem, s>>>(vp, n_views, raw, n, means, scales, quats, shs_dc, (float2*)xy, radii, clamped,
                                                                         row_index, dst, cap, ticket, state, d_count);
    else
        project_pack_multi_kernel<16><<<blocks, PACK_THREADS, smem, s>>>(vp, n_views, raw, n, means, scales, quats, shs_dc, (float2*)xy, radii, clamped,
                                                                         row_index, dst, cap, ticket, state, d_count);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

int launch_project_bwd_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                             const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, const int32_t* radii,
                             const uint8_t* clamped, const int32_t* row_index, const float* const* v_rows, float* v_means, float* v_scales,
                             float* v_quats, float* v_opac_logit, float* v_shs_dc, float* v_shs_rest, cudaStream_t s) {
    if (n == 0 || n_views == 0) return B200GS_OK;
    (void)shs_dc;
    ViewPack vp;
    RowSources src;
    static const float dummy[B200GS_ROW_FLOATS] = {0.f};
    for (int j = 0; j < B200GS_MAX_VIEWS; ++j) {
        vp.v[j] = views[j < n_views ? j : 0];
        src.rows[j] = (j < n_views && v_rows[j]) ? v_rows[j] : dummy;   // NULL only when no row of that view is ever read
    }
    RawIO raw{opac_logits, shs_rest, nullptr, nullptr, v_opac_logit, v_shs_rest, anti_aliased, nullptr, nullptr, 0};
    // the SH-gradient rows accumulate in the kernel's staging buffer: coefficient storage wider than 16 takes the 25-coefficient instantiation
    if (views[0].sh_stride > 25) {
        set_error("project_bwd_multi: sh_stride %d exceeds 25 coefficients", views[0].sh_stride);
        return B200GS_EINVAL;
    }
    if (views[0].sh_degree > 3 || views[0].sh_stride > 16)
        project_bwd_multi_kernel<25><<<(unsigned)div_up64(n, BWD_THREADS), BWD_THREADS, 0, s>>>(vp, n_views, raw, src, n, means, scales, quats, radii,
                                                                                                clamped, row_index, v_means, v_scales, (float4*)v_quats,
                                                                                                v_shs_dc);
    else
        project_bwd_multi_kernel<16><<<(unsigned)div_up64(n, BWD_THREADS), BWD_THREADS, 0, s>>>(vp, n_views, raw, src, n, means, scales, quats, radii,
                                                                                                clamped, row_index, v_means, v_scales, (float4*)v_quats,
                                                                                                v_shs_dc);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

int launch_sh_fwd(int degree, int stride, int64_t n, const float* dirs, const float* coeffs, float* rgb, cudaStream_t s) {
    if (n == 0) return B200GS_OK;
    if (degree > 3) sh_fwd_kernel<25><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(degree, stride, n, dirs, coeffs, rgb);
    else sh_fwd_kernel<16><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(degree, stride, n, dirs, coeffs, rgb);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

int launch_sh_bwd(int degree, int stride, int64_t n, const float* dirs, const float* coeffs, const float* v_rgb,
                  float* v_coeffs, float* v_dirs, cudaStream_t s) {
    if (n == 0) return B200GS_OK;
    if (degree > 3) sh_bwd_kernel<25><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(degree, stride, n, dirs, coeffs, v_rgb, v_coeffs, v_dirs);
    else sh_bwd_kernel<16><<<(unsigned)div_up64(n, 256), 256, 0, s>>>(degree, stride, n, dirs, coeffs, v_rgb, v_coeffs, v_dirs);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

}  // namespace b200gs
