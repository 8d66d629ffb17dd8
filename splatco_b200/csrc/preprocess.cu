// Per-Gaussian kernels: projection / EWA covariance / radii / tile counts (forward), the anchor
// prefilter, the block-sum scan that yields the instance count R, and the per-Gaussian backward
// chain.  Replaces upstream preprocessCUDA / filter_preprocessCUDA / InclusiveSum /
// computeCov2DCUDA+preprocessCUDA(bwd) [SURVEY.md Appendix A.2, A.5; reference call sites
// gaussian_renderer/__init__.py:163-171, 239-242].
//
// All of these are HBM-bound streaming kernels (SURVEY §8d: 48 B/anchor, 104 B/Gaussian,
// ~200 B/Gaussian): one Gaussian per thread, coalesced SoA reads, one packed 48-byte record written
// per Gaussian so the blend kernels fetch a splat with three 16-byte loads.
//
// Rounding contract: the chain that decides integers (radius, rect, tiles_touched, depth key) uses
// individually rounded __f*_rn operations in exactly the order of oracle/raster_oracle.c, so the
// integer outputs are bit-identical to the CPU oracle regardless of nvcc's FMA contraction.
#include <type_traits>

#include "camgrad.cuh"
#include "common.cuh"

namespace splatco {

// individually-rounded fp32 ops (no contraction possible)
__device__ __forceinline__ float MUL(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float ADD(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float SUB(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float DIV(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float SQRT(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ float DOT3(float a0, float b0, float a1, float b1, float a2, float b2) {
    return ADD(ADD(MUL(a0, b0), MUL(a1, b1)), MUL(a2, b2));
}

struct Proj {
    int radius;
    float depth, px, py;
    float conic[3];
    float rho;                // antialiasing opacity factor (project_one<true> only)
    int r0x, r0y, r1x, r1y;
    uint32_t tiles;
};

__device__ __forceinline__ void rect_of(float px, float py, int radius, int gx, int gy, int &r0x,
                                        int &r0y, int &r1x, int &r1y) {
    const float rf = (float)radius;
    // division by 16 is exact, so x * 0.0625f == x / 16.0f bit for bit
    r0x = min(gx, max(0, __float2int_rz(MUL(SUB(px, rf), 0.0625f))));
    r0y = min(gy, max(0, __float2int_rz(MUL(SUB(py, rf), 0.0625f))));
    r1x = min(gx, max(0, __float2int_rz(MUL(ADD(ADD(px, rf), 15.0f), 0.0625f))));
    r1y = min(gy, max(0, __float2int_rz(MUL(ADD(ADD(py, rf), 15.0f), 0.0625f))));
}

// view/proj are the 32 floats staged in shared memory by the caller.
// AA: also o.rho = sqrt(max(2.5e-5, det0 / det)), the ratio of the undilated to the dilated 2D covariance determinant
// (DESIGN.md §4.5c), on the same pinned-rounding chain as the conic.
template <bool AA = false>
__device__ __forceinline__ void project_one(float x, float y, float z, float sx, float sy, float sz,
                                            float4 q, float mod, const float *__restrict__ view,
                                            const float *__restrict__ proj, float tanfovx,
                                            float tanfovy, float focal_x, float focal_y, int H, int W,
                                            int gx, int gy, Proj &o) {
    o.radius = 0; o.tiles = 0; o.depth = 0.f; o.px = 0.f; o.py = 0.f;
    o.conic[0] = o.conic[1] = o.conic[2] = 0.f; o.r0x = o.r0y = o.r1x = o.r1y = 0;
    const float vx = ADD(ADD(ADD(MUL(view[0], x), MUL(view[4], y)), MUL(view[8], z)), view[12]);
    const float vy = ADD(ADD(ADD(MUL(view[1], x), MUL(view[5], y)), MUL(view[9], z)), view[13]);
    const float vz = ADD(ADD(ADD(MUL(view[2], x), MUL(view[6], y)), MUL(view[10], z)), view[14]);
    if (vz <= 0.2f) return;
    const float hx = ADD(ADD(ADD(MUL(proj[0], x), MUL(proj[4], y)), MUL(proj[8], z)), proj[12]);
    const float hy = ADD(ADD(ADD(MUL(proj[1], x), MUL(proj[5], y)), MUL(proj[9], z)), proj[13]);
    const float hw = ADD(ADD(ADD(MUL(proj[3], x), MUL(proj[7], y)), MUL(proj[11], z)), proj[15]);
    const float pw = DIV(1.0f, ADD(hw, 0.0000001f));
    const float ndc_x = MUL(hx, pw), ndc_y = MUL(hy, pw);

    const float s0 = MUL(mod, sx), s1 = MUL(mod, sy), s2 = MUL(mod, sz);
    const float qr = q.x, qx = q.y, qy = q.z, qz = q.w;
    float R[3][3];
    R[0][0] = SUB(1.0f, MUL(2.0f, ADD(MUL(qy, qy), MUL(qz, qz))));
    R[0][1] = MUL(2.0f, SUB(MUL(qx, qy), MUL(qr, qz)));
    R[0][2] = MUL(2.0f, ADD(MUL(qx, qz), MUL(qr, qy)));
    R[1][0] = MUL(2.0f, ADD(MUL(qx, qy), MUL(qr, qz)));
    R[1][1] = SUB(1.0f, MUL(2.0f, ADD(MUL(qx, qx), MUL(qz, qz))));
    R[1][2] = MUL(2.0f, SUB(MUL(qy, qz), MUL(qr, qx)));
    R[2][0] = MUL(2.0f, SUB(MUL(qx, qz), MUL(qr, qy)));
    R[2][1] = MUL(2.0f, ADD(MUL(qy, qz), MUL(qr, qx)));
    R[2][2] = SUB(1.0f, MUL(2.0f, ADD(MUL(qx, qx), MUL(qy, qy))));
    float M[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { M[i][0] = MUL(R[i][0], s0); M[i][1] = MUL(R[i][1], s1); M[i][2] = MUL(R[i][2], s2); }
    float S[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = i; j < 3; ++j) {
            S[i][j] = DOT3(M[i][0], M[j][0], M[i][1], M[j][1], M[i][2], M[j][2]);
            S[j][i] = S[i][j];
        }

    const float limx = MUL(1.3f, tanfovx), limy = MUL(1.3f, tanfovy);
    const float txtz = DIV(vx, vz), tytz = DIV(vy, vz);
    const float tx = MUL(fminf(limx, fmaxf(-limx, txtz)), vz);
    const float ty = MUL(fminf(limy, fmaxf(-limy, tytz)), vz);
    const float vz2 = MUL(vz, vz);
    const float J00 = DIV(focal_x, vz);
    const float J02 = DIV(-MUL(focal_x, tx), vz2);
    const float J11 = DIV(focal_y, vz);
    const float J12 = DIV(-MUL(focal_y, ty), vz2);
    float A0[3], A1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float r0 = view[4 * k + 0], r1 = view[4 * k + 1], r2 = view[4 * k + 2];
        A0[k] = ADD(MUL(J00, r0), MUL(J02, r2));
        A1[k] = ADD(MUL(J11, r1), MUL(J12, r2));
    }
    float B0[3], B1[3];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        B0[l] = DOT3(A0[0], S[0][l], A0[1], S[1][l], A0[2], S[2][l]);
        B1[l] = DOT3(A1[0], S[0][l], A1[1], S[1][l], A1[2], S[2][l]);
    }
    const float a0 = DOT3(B0[0], A0[0], B0[1], A0[1], B0[2], A0[2]);
    const float b = DOT3(B0[0], A1[0], B0[1], A1[1], B0[2], A1[2]);
    const float c0 = DOT3(B1[0], A1[0], B1[1], A1[1], B1[2], A1[2]);
    const float a = ADD(a0, 0.3f), c = ADD(c0, 0.3f);
    const float det = SUB(MUL(a, c), MUL(b, b));
    if (det == 0.0f) return;
    if constexpr (AA) o.rho = SQRT(fmaxf(2.5e-5f, DIV(SUB(MUL(a0, c0), MUL(b, b)), det)));
    const float det_inv = DIV(1.0f, det);
    const float mid = MUL(0.5f, ADD(a, c));
    const float sq = SQRT(fmaxf(0.1f, SUB(MUL(mid, mid), det)));
    const float l1 = ADD(mid, sq), l2 = SUB(mid, sq);
    const int radius = __float2int_rz(ceilf(MUL(3.0f, SQRT(fmaxf(l1, l2)))));
    const float px = MUL(SUB(MUL(ADD(ndc_x, 1.0f), (float)W), 1.0f), 0.5f);
    const float py = MUL(SUB(MUL(ADD(ndc_y, 1.0f), (float)H), 1.0f), 0.5f);
    int r0x, r0y, r1x, r1y;
    rect_of(px, py, radius, gx, gy, r0x, r0y, r1x, r1y);
    const int area = (r1x - r0x) * (r1y - r0y);
    if (area == 0) return;
    o.radius = radius; o.depth = vz; o.px = px; o.py = py;
    o.conic[0] = MUL(c, det_inv); o.conic[1] = -MUL(b, det_inv); o.conic[2] = MUL(a, det_inv);
    o.r0x = r0x; o.r0y = r0y; o.r1x = r1x; o.r1y = r1y;
    o.tiles = (uint32_t)area;
}

__device__ __forceinline__ void stage_cam(float *s_cam, const float *view, const float *proj) {
    if (threadIdx.x < 16) s_cam[threadIdx.x] = __ldg(view + threadIdx.x);
    else if (threadIdx.x < 32) s_cam[threadIdx.x] = __ldg(proj + threadIdx.x - 16);
    __syncthreads();
}

// ---- anchor prefilter -----------------------------------------------------------------------------
__global__ void __launch_bounds__(PRE_THREADS)
visible_filter_kernel(int N, const float *__restrict__ means3D, const float *__restrict__ scales,
                      int scale_stride, const float *__restrict__ rots, float mod,
                      const float *__restrict__ view, const float *__restrict__ proj, float tanfovx,
                      float tanfovy, float fx, float fy, int H, int W, int gx, int gy,
                      int32_t *__restrict__ radii) {
    __shared__ float s_cam[32];
    stage_cam(s_cam, view, proj);
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    if (i >= N) return;
    const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
    const float *sp = scales + (size_t)scale_stride * i;
    const float4 q = *reinterpret_cast<const float4 *>(rots + 4 * (size_t)i);
    Proj o;
    project_one(x, y, z, sp[0], sp[1], sp[2], q, mod, s_cam, s_cam + 16, tanfovx, tanfovy, fx, fy, H, W, gx, gy, o);
    radii[i] = o.radius;
}

// ---- anchor prefilter + stable compaction of the visible indices -----------------------------------------------
// prefilter_voxel returns a bool mask (gaussian_renderer/__init__.py:243-244) that render() immediately turns back
// into an index list with boolean indexing (:21-29).  The filter writes the mask, per-CTA counts, and (after the scan
// of the counts) the ascending index list itself, so the host needs neither torch.nonzero nor its two syncs.
__global__ void __launch_bounds__(PRE_THREADS)
visible_filter_mask_kernel(int N, const float *__restrict__ means3D, const float *__restrict__ scales,
                           int scale_stride, const float *__restrict__ rots, float mod,
                           const float *__restrict__ view, const float *__restrict__ proj, float tanfovx,
                           float tanfovy, float fx, float fy, int H, int W, int gx, int gy,
                           int32_t *__restrict__ radii, uint8_t *__restrict__ mask, uint32_t *__restrict__ block_sums) {
    __shared__ float s_cam[32];
    stage_cam(s_cam, view, proj);
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    int radius = 0;
    if (i < N) {
        const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
        const float *sp = scales + (size_t)scale_stride * i;
        const float4 q = *reinterpret_cast<const float4 *>(rots + 4 * (size_t)i);
        Proj o;
        project_one(x, y, z, sp[0], sp[1], sp[2], q, mod, s_cam, s_cam + 16, tanfovx, tanfovy, fx, fy, H, W, gx, gy, o);
        radius = o.radius;
        radii[i] = radius;
        mask[i] = radius > 0 ? 1 : 0;
    }
    const int cnt = __syncthreads_count(radius > 0);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = (uint32_t)cnt;
}

__global__ void __launch_bounds__(PRE_THREADS)
visible_compact_kernel(int N, const uint8_t *__restrict__ mask, const uint32_t *__restrict__ block_offsets,
                       int32_t *__restrict__ idx_out) {
    __shared__ uint32_t s_warp[PRE_THREADS / 32];
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const bool vis = i < N && mask[i];
    const uint32_t b = __ballot_sync(0xffffffffu, vis);
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int w = 0; w < PRE_THREADS / 32; ++w) woff += (w < (int)warp) ? s_warp[w] : 0u;
    if (vis) idx_out[block_offsets[blockIdx.x] + woff + __popc(b & lanemask_lt())] = i;
}

// ---- preprocess forward: also emits per-block tile-count sums (first level of the scan) ---------
// AA: the record's opacity is opacities[i] * rho (project_one<true>); everything else is that of the plain kernel.
template <bool AA>
__global__ void __launch_bounds__(PRE_THREADS)
preprocess_fwd_kernel(int P, const uint32_t *__restrict__ P_dev, const float *__restrict__ means3D, const float *__restrict__ scales,
                      int scale_stride, const float *__restrict__ rots,
                      const float *__restrict__ opacities, const float *__restrict__ colors, float mod,
                      const float *__restrict__ view, const float *__restrict__ proj, float tanfovx,
                      float tanfovy, float fx, float fy, int H, int W, int gx, int gy,
                      int32_t *__restrict__ radii, float4 *__restrict__ rec,
                      float *__restrict__ depths, uint32_t *__restrict__ tiles,
                      uint32_t *__restrict__ block_sums) {
    __shared__ float s_cam[32];
    __shared__ uint32_t s_warp[PRE_THREADS / 32];
    stage_cam(s_cam, view, proj);
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    uint32_t t = 0;
    // counted variant: the live row count is still on the device (decode's survivor count); rows in
    // [count, P) of the caller's upper-bound buffers are uninitialised and become invisible Gaussians
    const int live = P_dev ? min(P, (int)__ldg(P_dev)) : P;
    if (i >= live && i < P) { radii[i] = 0; tiles[i] = 0; }
    if (i < live) {
        const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
        const float *sp = scales + (size_t)scale_stride * i;
        const float4 q = *reinterpret_cast<const float4 *>(rots + 4 * (size_t)i);
        Proj o;
        project_one<AA>(x, y, z, sp[0], sp[1], sp[2], q, mod, s_cam, s_cam + 16, tanfovx, tanfovy, fx, fy, H, W, gx, gy, o);
        radii[i] = o.radius;
        tiles[i] = o.tiles;
        depths[i] = o.depth;
        t = o.tiles;
        float4 r0, r1, r2;
        if (o.radius > 0) {
            const float op = AA ? MUL(opacities[i], o.rho) : opacities[i];
            const float cr = colors[3 * (size_t)i], cg = colors[3 * (size_t)i + 1], cb = colors[3 * (size_t)i + 2];
            r0 = make_float4(o.px, o.py, o.conic[0], o.conic[1]);
            r1 = make_float4(o.conic[2], op, cr, cg);
            r2 = make_float4(cb, o.depth, __int_as_float(o.radius), 0.f);
        } else {
            r0 = r1 = r2 = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        rec[3 * (size_t)i] = r0; rec[3 * (size_t)i + 1] = r1; rec[3 * (size_t)i + 2] = r2;
    }
    // block sum of tiles_touched
    uint32_t s = t;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane_id() == 0) s_warp[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
#pragma unroll
        for (int w = 0; w < PRE_THREADS / 32; ++w) tot += s_warp[w];
        block_sums[blockIdx.x] = tot;
    }
}

// ---- per-Gaussian backward chain (fp32; tolerance-compared, so the compiler may contract) --------
// DEPTH: the blend's dL/dz_view (the trailing argument `const float *dL_ddepth`) is added to dL/dmeans3D through
// dz_view/dmean = (V[2], V[6], V[10]).
// Antialiasing: a trailing AAOpacity (after dL_ddepth when DEPTH) adds the opacity factor rho's term to dL/d(a, b, c)
// and rewrites dL_dopacity in place from dL/d(record opacity) to dL/dopacities (aa_rho_grad).
// The trailing arguments are a parameter pack, empty for the colour-only call, so that preprocess_bwd_kernel<false> keeps
// the parameter list -- and with it the code -- of the colour-only kernel.
struct AAOpacity {
    const float *opacities;
    float *dL_dopacity;
};
__device__ __forceinline__ const float *depth_grad_ptr(const float *p) { return p; }
__device__ __forceinline__ const float *depth_grad_ptr(const float *p, AAOpacity) { return p; }
__device__ __forceinline__ AAOpacity aa_args(AAOpacity a) { return a; }
__device__ __forceinline__ AAOpacity aa_args(const float *, AAOpacity a) { return a; }
template <typename... T> constexpr bool has_aa = (std::is_same<T, AAOpacity>::value || ... || false);

// rho = sqrt(max(2.5e-5, det0 / det)) with det0 = a0 c0 - b^2 of the undilated and det = a c - b^2 of the dilated
// (a = a0 + 0.3, c = c0 + 0.3) 2D covariance.  Where the clamp is inactive, adds dL/drho * drho/d(a, b, c) to
// (dL_da, dL_db, dL_dc), with the exact derivatives in cancellation-free form:
//     drho/da = (c0 det - det0 c) / (2 rho det^2) = 0.3 (c c0 + b^2) / (2 rho det^2)
//     drho/dc = (a0 det - det0 a) / (2 rho det^2) = 0.3 (a a0 + b^2) / (2 rho det^2)
//     drho/db = b (det0 - det) / (rho det^2)       = -0.3 b (a + c0) / (rho det^2)
// Returns rho.
__device__ __forceinline__ float aa_rho_grad(float a0, float b, float c0, float a, float c, float det, float dL_drho,
                                             float &dL_da, float &dL_db, float &dL_dc) {
    const float ratio = (a0 * c0 - b * b) / det;
    if (!(ratio > 2.5e-5f)) return sqrtf(2.5e-5f);
    const float rho = sqrtf(ratio);
    const float idet = 1.f / det;
    const float k = 0.15f * dL_drho / rho * idet * idet;        // 0.3 dL/drho / (2 rho det^2)
    dL_da += k * (c * c0 + b * b);
    dL_dc += k * (a * a0 + b * b);
    dL_db -= 2.f * k * b * (a + c0);
    return rho;
}

template <bool DEPTH, typename... DepthGrad>
__global__ void __launch_bounds__(PRE_THREADS)
preprocess_bwd_kernel(int P, const float *__restrict__ means3D, const float *__restrict__ scales,
                      int scale_stride, const float *__restrict__ rots, float mod,
                      const float *__restrict__ view, const float *__restrict__ proj, float tanfovx,
                      float tanfovy, float fx, float fy, const int32_t *__restrict__ radii,
                      const float *__restrict__ dL_dmean2D, const float *__restrict__ dL_dconic,
                      float *__restrict__ dL_dmeans3D, float *__restrict__ dL_dscales,
                      float *__restrict__ dL_drots, DepthGrad... dL_ddepth) {
    __shared__ float s_cam[32];
    stage_cam(s_cam, view, proj);
    const float *V = s_cam, *Pm = s_cam + 16;
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    if (i >= P) return;
    float gmx = 0.f, gmy = 0.f, gmz = 0.f, gs0 = 0.f, gs1 = 0.f, gs2 = 0.f;
    float4 gq = make_float4(0.f, 0.f, 0.f, 0.f);
    if (radii[i] > 0) {
        const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
        const float *sp = scales + (size_t)scale_stride * i;
        const float4 q = *reinterpret_cast<const float4 *>(rots + 4 * (size_t)i);
        // Rot[r][k] = V[4k + r]
        const float vx = V[0] * x + V[4] * y + V[8] * z + V[12];
        const float vy = V[1] * x + V[5] * y + V[9] * z + V[13];
        const float vz = V[2] * x + V[6] * y + V[10] * z + V[14];
        const float s[3] = { mod * sp[0], mod * sp[1], mod * sp[2] };
        const float qr = q.x, qx = q.y, qy = q.z, qz = q.w;
        float R[3][3];
        R[0][0] = 1.f - 2.f * (qy * qy + qz * qz); R[0][1] = 2.f * (qx * qy - qr * qz); R[0][2] = 2.f * (qx * qz + qr * qy);
        R[1][0] = 2.f * (qx * qy + qr * qz); R[1][1] = 1.f - 2.f * (qx * qx + qz * qz); R[1][2] = 2.f * (qy * qz - qr * qx);
        R[2][0] = 2.f * (qx * qz - qr * qy); R[2][1] = 2.f * (qy * qz + qr * qx); R[2][2] = 1.f - 2.f * (qx * qx + qy * qy);
        float M[3][3], S[3][3];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int k = 0; k < 3; ++k) M[a][k] = R[a][k] * s[k];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) S[a][b] = M[a][0] * M[b][0] + M[a][1] * M[b][1] + M[a][2] * M[b][2];
        const float limx = 1.3f * tanfovx, limy = 1.3f * tanfovy;
        const float txtz = vx / vz, tytz = vy / vz;
        const bool clx = (txtz < -limx) || (txtz > limx), cly = (tytz < -limy) || (tytz > limy);
        const float tx = fminf(limx, fmaxf(-limx, txtz)) * vz, ty = fminf(limy, fmaxf(-limy, tytz)) * vz;
        const float iz = 1.f / vz, iz2 = iz * iz, iz3 = iz2 * iz;
        const float J00 = fx * iz, J02 = -(fx * tx) * iz2, J11 = fy * iz, J12 = -(fy * ty) * iz2;
        float A[2][3], B[2][3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            A[0][k] = J00 * V[4 * k] + J02 * V[4 * k + 2];
            A[1][k] = J11 * V[4 * k + 1] + J12 * V[4 * k + 2];
        }
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int l = 0; l < 3; ++l) B[r][l] = A[r][0] * S[0][l] + A[r][1] * S[1][l] + A[r][2] * S[2][l];
        const float a = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2] + 0.3f;
        const float b = B[0][0] * A[1][0] + B[0][1] * A[1][1] + B[0][2] * A[1][2];
        const float c = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2] + 0.3f;
        const float denom = a * c - b * b;
        const float d2inv = 1.0f / (denom * denom + 0.0000001f);   // reference quirk (SURVEY A.5)
        const float gc0 = dL_dconic[3 * (size_t)i], gc1 = dL_dconic[3 * (size_t)i + 1], gc2 = dL_dconic[3 * (size_t)i + 2];
        float dL_da = d2inv * (-c * c * gc0 + 2.f * b * c * gc1 + (denom - a * c) * gc2);
        float dL_dc = d2inv * (-a * a * gc2 + 2.f * a * b * gc1 + (denom - a * c) * gc0);
        float dL_db = d2inv * 2.f * (b * c * gc0 - (denom + 2.f * b * b) * gc1 + a * b * gc2);
        if constexpr (has_aa<DepthGrad...>) {
            const AAOpacity aa = aa_args(dL_ddepth...);
            const float a0 = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2];
            const float c0 = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2];
            const float g = aa.dL_dopacity[i];
            const float rho = aa_rho_grad(a0, b, c0, a, c, denom, g * aa.opacities[i], dL_da, dL_db, dL_dc);
            aa.dL_dopacity[i] = g * rho;
        }
        const float G2[2][2] = { { dL_da, 0.5f * dL_db }, { 0.5f * dL_db, dL_dc } };
        // GA = G2 A (2x3);  dS = A^T GA;  dA = 2 G2 B
        float GA[2][3], dS[3][3], dA[2][3];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int l = 0; l < 3; ++l) {
                GA[r][l] = G2[r][0] * A[0][l] + G2[r][1] * A[1][l];
                dA[r][l] = 2.f * (G2[r][0] * B[0][l] + G2[r][1] * B[1][l]);
            }
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int l = 0; l < 3; ++l) dS[k][l] = A[0][k] * GA[0][l] + A[1][k] * GA[1][l];
        float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            dJ00 += dA[0][k] * V[4 * k]; dJ02 += dA[0][k] * V[4 * k + 2];
            dJ11 += dA[1][k] * V[4 * k + 1]; dJ12 += dA[1][k] * V[4 * k + 2];
        }
        const float dtx = clx ? 0.f : -fx * iz2 * dJ02;
        const float dty = cly ? 0.f : -fy * iz2 * dJ12;
        const float dtz = -fx * iz2 * dJ00 - fy * iz2 * dJ11 + 2.f * fx * tx * iz3 * dJ02 + 2.f * fy * ty * iz3 * dJ12;
        gmx = V[0] * dtx + V[1] * dty + V[2] * dtz;
        gmy = V[4] * dtx + V[5] * dty + V[6] * dtz;
        gmz = V[8] * dtx + V[9] * dty + V[10] * dtz;
        const float hx = Pm[0] * x + Pm[4] * y + Pm[8] * z + Pm[12];
        const float hy = Pm[1] * x + Pm[5] * y + Pm[9] * z + Pm[13];
        const float hw = Pm[3] * x + Pm[7] * y + Pm[11] * z + Pm[15];
        const float mw = 1.0f / (hw + 0.0000001f);
        const float mul1 = hx * mw * mw, mul2 = hy * mw * mw;
        const float g2x = dL_dmean2D[3 * (size_t)i], g2y = dL_dmean2D[3 * (size_t)i + 1];
        gmx += (Pm[0] * mw - Pm[3] * mul1) * g2x + (Pm[1] * mw - Pm[3] * mul2) * g2y;
        gmy += (Pm[4] * mw - Pm[7] * mul1) * g2x + (Pm[5] * mw - Pm[7] * mul2) * g2y;
        gmz += (Pm[8] * mw - Pm[11] * mul1) * g2x + (Pm[9] * mw - Pm[11] * mul2) * g2y;
        if constexpr (DEPTH) {
            const float gd = depth_grad_ptr(dL_ddepth...)[i];
            gmx = fmaf(V[2], gd, gmx); gmy = fmaf(V[6], gd, gmy); gmz = fmaf(V[10], gd, gmz);
        }
        // Sigma = M M^T: dM = 2 dS M;  M_ak = R_ak s_k
        float dR[3][3], gsv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            float acc = 0.f;
#pragma unroll
            for (int a2 = 0; a2 < 3; ++a2) {
                const float dM = 2.f * (dS[a2][0] * M[0][k] + dS[a2][1] * M[1][k] + dS[a2][2] * M[2][k]);
                acc += dM * R[a2][k];
                dR[a2][k] = dM * s[k];
            }
            gsv[k] = acc * mod;
        }
        gs0 = gsv[0]; gs1 = gsv[1]; gs2 = gsv[2];
        gq.x = 2.f * (-qz * dR[0][1] + qy * dR[0][2] + qz * dR[1][0] - qx * dR[1][2] - qy * dR[2][0] + qx * dR[2][1]);
        gq.y = 2.f * (qy * dR[0][1] + qz * dR[0][2] + qy * dR[1][0] - 2.f * qx * dR[1][1] - qr * dR[1][2] + qz * dR[2][0] + qr * dR[2][1] - 2.f * qx * dR[2][2]);
        gq.z = 2.f * (-2.f * qy * dR[0][0] + qx * dR[0][1] + qr * dR[0][2] + qx * dR[1][0] + qz * dR[1][2] - qr * dR[2][0] + qz * dR[2][1] - 2.f * qy * dR[2][2]);
        gq.w = 2.f * (-2.f * qz * dR[0][0] - qr * dR[0][1] + qx * dR[0][2] + qr * dR[1][0] - 2.f * qz * dR[1][1] + qy * dR[1][2] + qx * dR[2][0] + qy * dR[2][1]);
    }
    dL_dmeans3D[3 * (size_t)i] = gmx; dL_dmeans3D[3 * (size_t)i + 1] = gmy; dL_dmeans3D[3 * (size_t)i + 2] = gmz;
    dL_dscales[3 * (size_t)i] = gs0; dL_dscales[3 * (size_t)i + 1] = gs1; dL_dscales[3 * (size_t)i + 2] = gs2;
    *reinterpret_cast<float4 *>(dL_drots + 4 * (size_t)i) = gq;
}

// ---- camera gradients: dL/dviewmatrix and dL/dprojmatrix -----------------------------------------------------------
// Launched after preprocess_bwd_kernel, which stays as it is: this kernel re-derives the same chain from the same
// inputs (formulas and evaluation order of preprocess_bwd_kernel) and reduces, per CTA, the 32 camera floats
//     dV[4k+r]  += g[r] p~_k                         g = dL/dp_view = (dtx, dty, dtz + dL_ddepth),  p~ = (x, y, z, 1)
//     dV[4k]    += dA[0][k] J00,   dV[4k+1] += dA[1][k] J11,   dV[4k+2] += dA[0][k] J02 + dA[1][k] J12   (k < 3)
//     dPm[4k]   += g2x mw p~_k,    dPm[4k+1] += g2y mw p~_k,   dPm[4k+3] += -(g2x hx + g2y hy) mw^2 p~_k
// into part[blockIdx.x][0..31] (camgrad.cuh).  The forward never reads V[3,7,11,15] or Pm[2,6,10,14]: those stay 0.
// Antialiasing: a trailing AAOpacity adds the rho term to dL/d(a, b, c) as preprocess_bwd_kernel does.  This kernel only
// reads dL_dopacity, which must still hold dL/d(record opacity): it runs before the per-Gaussian kernel rewrites it.
template <typename... AA>
__global__ void __launch_bounds__(PRE_THREADS)
preprocess_bwd_camera_kernel(int P, const float *__restrict__ means3D, const float *__restrict__ scales,
                             int scale_stride, const float *__restrict__ rots, float mod,
                             const float *__restrict__ view, const float *__restrict__ proj, float tanfovx,
                             float tanfovy, float fx, float fy, const int32_t *__restrict__ radii,
                             const float *__restrict__ dL_dmean2D, const float *__restrict__ dL_dconic,
                             const float *__restrict__ dL_ddepth, float *__restrict__ part, AA... aa_opacity) {
    static_assert(PRE_THREADS == CAM_ROWS, "one camera partial per preprocess CTA");
    __shared__ float s_cam[32];
    stage_cam(s_cam, view, proj);
    const float *V = s_cam, *Pm = s_cam + 16;
    const int i = blockIdx.x * PRE_THREADS + threadIdx.x;
    float cg[CAM_COLS];
#pragma unroll
    for (int c = 0; c < CAM_COLS; ++c) cg[c] = 0.f;
    if (i < P && radii[i] > 0) {
        const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
        const float *sp = scales + (size_t)scale_stride * i;
        const float4 q = *reinterpret_cast<const float4 *>(rots + 4 * (size_t)i);
        const float vx = V[0] * x + V[4] * y + V[8] * z + V[12];
        const float vy = V[1] * x + V[5] * y + V[9] * z + V[13];
        const float vz = V[2] * x + V[6] * y + V[10] * z + V[14];
        const float s[3] = { mod * sp[0], mod * sp[1], mod * sp[2] };
        const float qr = q.x, qx = q.y, qy = q.z, qz = q.w;
        float R[3][3];
        R[0][0] = 1.f - 2.f * (qy * qy + qz * qz); R[0][1] = 2.f * (qx * qy - qr * qz); R[0][2] = 2.f * (qx * qz + qr * qy);
        R[1][0] = 2.f * (qx * qy + qr * qz); R[1][1] = 1.f - 2.f * (qx * qx + qz * qz); R[1][2] = 2.f * (qy * qz - qr * qx);
        R[2][0] = 2.f * (qx * qz - qr * qy); R[2][1] = 2.f * (qy * qz + qr * qx); R[2][2] = 1.f - 2.f * (qx * qx + qy * qy);
        float M[3][3], S[3][3];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int k = 0; k < 3; ++k) M[a][k] = R[a][k] * s[k];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) S[a][b] = M[a][0] * M[b][0] + M[a][1] * M[b][1] + M[a][2] * M[b][2];
        const float limx = 1.3f * tanfovx, limy = 1.3f * tanfovy;
        const float txtz = vx / vz, tytz = vy / vz;
        const bool clx = (txtz < -limx) || (txtz > limx), cly = (tytz < -limy) || (tytz > limy);
        const float tx = fminf(limx, fmaxf(-limx, txtz)) * vz, ty = fminf(limy, fmaxf(-limy, tytz)) * vz;
        const float iz = 1.f / vz, iz2 = iz * iz, iz3 = iz2 * iz;
        const float J00 = fx * iz, J02 = -(fx * tx) * iz2, J11 = fy * iz, J12 = -(fy * ty) * iz2;
        float A[2][3], B[2][3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            A[0][k] = J00 * V[4 * k] + J02 * V[4 * k + 2];
            A[1][k] = J11 * V[4 * k + 1] + J12 * V[4 * k + 2];
        }
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int l = 0; l < 3; ++l) B[r][l] = A[r][0] * S[0][l] + A[r][1] * S[1][l] + A[r][2] * S[2][l];
        const float a = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2] + 0.3f;
        const float b = B[0][0] * A[1][0] + B[0][1] * A[1][1] + B[0][2] * A[1][2];
        const float c = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2] + 0.3f;
        const float denom = a * c - b * b;
        const float d2inv = 1.0f / (denom * denom + 0.0000001f);
        const float gc0 = dL_dconic[3 * (size_t)i], gc1 = dL_dconic[3 * (size_t)i + 1], gc2 = dL_dconic[3 * (size_t)i + 2];
        float dL_da = d2inv * (-c * c * gc0 + 2.f * b * c * gc1 + (denom - a * c) * gc2);
        float dL_dc = d2inv * (-a * a * gc2 + 2.f * a * b * gc1 + (denom - a * c) * gc0);
        float dL_db = d2inv * 2.f * (b * c * gc0 - (denom + 2.f * b * b) * gc1 + a * b * gc2);
        if constexpr (sizeof...(AA) > 0) {
            const AAOpacity aa = aa_args(aa_opacity...);
            const float a0 = B[0][0] * A[0][0] + B[0][1] * A[0][1] + B[0][2] * A[0][2];
            const float c0 = B[1][0] * A[1][0] + B[1][1] * A[1][1] + B[1][2] * A[1][2];
            aa_rho_grad(a0, b, c0, a, c, denom, aa.dL_dopacity[i] * aa.opacities[i], dL_da, dL_db, dL_dc);
        }
        const float G2[2][2] = { { dL_da, 0.5f * dL_db }, { 0.5f * dL_db, dL_dc } };
        float dA[2][3];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int l = 0; l < 3; ++l) dA[r][l] = 2.f * (G2[r][0] * B[0][l] + G2[r][1] * B[1][l]);
        float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            dJ00 += dA[0][k] * V[4 * k]; dJ02 += dA[0][k] * V[4 * k + 2];
            dJ11 += dA[1][k] * V[4 * k + 1]; dJ12 += dA[1][k] * V[4 * k + 2];
        }
        const float dtx = clx ? 0.f : -fx * iz2 * dJ02;
        const float dty = cly ? 0.f : -fy * iz2 * dJ12;
        float dtz = -fx * iz2 * dJ00 - fy * iz2 * dJ11 + 2.f * fx * tx * iz3 * dJ02 + 2.f * fy * ty * iz3 * dJ12;
        if (dL_ddepth) dtz += dL_ddepth[i];
        const float hx = Pm[0] * x + Pm[4] * y + Pm[8] * z + Pm[12];
        const float hy = Pm[1] * x + Pm[5] * y + Pm[9] * z + Pm[13];
        const float hw = Pm[3] * x + Pm[7] * y + Pm[11] * z + Pm[15];
        const float mw = 1.0f / (hw + 0.0000001f);
        const float g2x = dL_dmean2D[3 * (size_t)i], g2y = dL_dmean2D[3 * (size_t)i + 1];
        const float ex = g2x * mw, ey = g2y * mw, ew = -(g2x * hx + g2y * hy) * mw * mw;
        const float ph[4] = { x, y, z, 1.f };
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            cg[4 * k] = dtx * ph[k]; cg[4 * k + 1] = dty * ph[k]; cg[4 * k + 2] = dtz * ph[k];
            cg[16 + 4 * k] = ex * ph[k]; cg[16 + 4 * k + 1] = ey * ph[k]; cg[16 + 4 * k + 3] = ew * ph[k];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            cg[4 * k] += dA[0][k] * J00;
            cg[4 * k + 1] += dA[1][k] * J11;
            cg[4 * k + 2] += dA[0][k] * J02 + dA[1][k] * J12;
        }
    }
    camera_block_partial(cg, part);
}

}  // namespace splatco

using namespace splatco;

extern "C" int splatco_visible_filter(int N, const float *means3D, const float *scales, int scale_stride,
                                      const float *rots, float scale_mod, const float *view,
                                      const float *proj, float tanfovx, float tanfovy, int H, int W,
                                      int32_t *radii_out, void *stream) {
    SPLATCO_REQUIRE(N >= 0 && H > 0 && W > 0, "visible_filter: bad sizes N=%d H=%d W=%d", N, H, W);
    if (N == 0) return 0;
    SPLATCO_REQUIRE(means3D && scales && rots && view && proj && radii_out, "visible_filter: null pointer");
    SPLATCO_REQUIRE(scale_stride >= 3, "visible_filter: scale_stride %d < 3", scale_stride);
    SPLATCO_REQUIRE(((uintptr_t)rots & 15) == 0, "visible_filter: rotations must be 16-byte aligned");
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    visible_filter_kernel<<<ceil_div(N, PRE_THREADS), PRE_THREADS, 0, (cudaStream_t)stream>>>(
        N, means3D, scales, scale_stride, rots, scale_mod, view, proj, tanfovx, tanfovy, fx, fy, H, W, gx, gy, radii_out);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" size_t splatco_visible_compact_ws_bytes(int N) {
    const size_t nb = (size_t)(N > 0 ? (N + PRE_THREADS - 1) / PRE_THREADS : 1);
    return 2 * align_up(nb * sizeof(uint32_t)) + align_up(sizeof(uint32_t));
}

extern "C" const int32_t *splatco_visible_compact_count_ptr(const void *ws, int N) {
    const size_t nb = (size_t)(N > 0 ? (N + PRE_THREADS - 1) / PRE_THREADS : 1);
    return ws ? reinterpret_cast<const int32_t *>((const char *)ws + 2 * align_up(nb * sizeof(uint32_t))) : nullptr;
}

extern "C" int splatco_visible_filter_compact(int N, const float *means3D, const float *scales, int scale_stride,
                                              const float *rots, float scale_mod, const float *view, const float *proj,
                                              float tanfovx, float tanfovy, int H, int W, int32_t *radii_out,
                                              uint8_t *mask_out, int32_t *idx_out, void *ws, int32_t *count_host,
                                              void *stream) {
    SPLATCO_REQUIRE(N >= 0 && H > 0 && W > 0, "visible_filter_compact: bad sizes N=%d H=%d W=%d", N, H, W);
    if (N == 0) { if (count_host) *count_host = 0; return 0; }
    SPLATCO_REQUIRE(means3D && scales && rots && view && proj && radii_out && mask_out && idx_out && ws,
                    "visible_filter_compact: null pointer");
    SPLATCO_REQUIRE(scale_stride >= 3, "visible_filter_compact: scale_stride %d < 3", scale_stride);
    SPLATCO_REQUIRE(((uintptr_t)rots & 15) == 0, "visible_filter_compact: rotations must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int nb = ceil_div(N, PRE_THREADS);
    char *b = (char *)ws;
    uint32_t *sums = (uint32_t *)b, *offs = (uint32_t *)(b + align_up((size_t)nb * 4)), *total = (uint32_t *)(b + 2 * align_up((size_t)nb * 4));
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    visible_filter_mask_kernel<<<nb, PRE_THREADS, 0, st>>>(N, means3D, scales, scale_stride, rots, scale_mod, view, proj, tanfovx,
                                                          tanfovy, fx, fy, H, W, gx, gy, radii_out, mask_out, sums);
    SPLATCO_CHECK_LAUNCH();
    scan_block_sums_kernel<<<1, 1024, 0, st>>>(nb, sums, offs, total);
    SPLATCO_CHECK_LAUNCH();
    visible_compact_kernel<<<nb, PRE_THREADS, 0, st>>>(N, mask_out, offs, idx_out);
    SPLATCO_CHECK_LAUNCH();
    if (count_host) SPLATCO_CHECK_CUDA(cudaMemcpyAsync(count_host, total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return 0;
}

template <bool AA>
static int preprocess_fwd_impl(int P, const uint32_t *P_dev, const float *means3D, const float *scales, int scale_stride,
                               const float *rots, const float *opacities, const float *colors,
                               float scale_mod, const float *view, const float *proj,
                               float tanfovx, float tanfovy, int H, int W, int32_t *radii_out,
                               void *geom, int32_t *num_rendered_host, void *stream) {
    SPLATCO_REQUIRE(P >= 0 && H > 0 && W > 0, "preprocess_fwd: bad sizes P=%d H=%d W=%d", P, H, W);
    cudaStream_t st = (cudaStream_t)stream;
    if (P == 0) {
        if (num_rendered_host) *num_rendered_host = 0;
        return 0;
    }
    SPLATCO_REQUIRE(means3D && scales && rots && opacities && colors && view && proj && radii_out && geom,
                    "preprocess_fwd: null pointer");
    SPLATCO_REQUIRE(scale_stride >= 3, "preprocess_fwd: scale_stride %d < 3", scale_stride);
    SPLATCO_REQUIRE(((uintptr_t)rots & 15) == 0 && ((uintptr_t)geom & 255) == 0,
                    "preprocess_fwd: rotations need 16-byte and geom 256-byte alignment");
    GeomWs g = geom_view(geom, P);
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    const int gx = ceil_div(W, TILE), gy = ceil_div(H, TILE);
    const int nb = ceil_div(P, PRE_THREADS);
    preprocess_fwd_kernel<AA><<<nb, PRE_THREADS, 0, st>>>(P, P_dev, means3D, scales, scale_stride, rots, opacities, colors,
                                                          scale_mod, view, proj, tanfovx, tanfovy, fx, fy, H, W,
                                                          gx, gy, radii_out, g.rec, g.depths, g.tiles, g.block_sums);
    SPLATCO_CHECK_LAUNCH();
    scan_block_sums_kernel<<<1, 1024, 0, st>>>(nb, g.block_sums, g.block_offsets, g.total);
    SPLATCO_CHECK_LAUNCH();
    if (num_rendered_host)
        SPLATCO_CHECK_CUDA(cudaMemcpyAsync(num_rendered_host, g.total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return 0;
}

extern "C" int splatco_preprocess_fwd(int P, const float *means3D, const float *scales, int scale_stride,
                                      const float *rots, const float *opacities, const float *colors,
                                      float scale_mod, const float *view, const float *proj,
                                      float tanfovx, float tanfovy, int H, int W, int32_t *radii_out,
                                      void *geom, int32_t *num_rendered_host, void *stream) {
    return preprocess_fwd_impl<false>(P, nullptr, means3D, scales, scale_stride, rots, opacities, colors, scale_mod, view, proj,
                               tanfovx, tanfovy, H, W, radii_out, geom, num_rendered_host, stream);
}

extern "C" int splatco_preprocess_fwd_counted(int P_max, const int32_t *P_dev, const float *means3D,
                                              const float *scales, int scale_stride, const float *rots,
                                              const float *opacities, const float *colors, float scale_mod,
                                              const float *view, const float *proj, float tanfovx,
                                              float tanfovy, int H, int W, int32_t *radii_out, void *geom,
                                              int32_t *num_rendered_host, void *stream) {
    SPLATCO_REQUIRE(P_dev, "preprocess_fwd_counted: null device count");
    return preprocess_fwd_impl<false>(P_max, reinterpret_cast<const uint32_t *>(P_dev), means3D, scales, scale_stride, rots,
                               opacities, colors, scale_mod, view, proj, tanfovx, tanfovy, H, W, radii_out, geom,
                               num_rendered_host, stream);
}

extern "C" int splatco_preprocess_fwd_aa(int P, const float *means3D, const float *scales, int scale_stride,
                                         const float *rots, const float *opacities, const float *colors,
                                         float scale_mod, const float *view, const float *proj,
                                         float tanfovx, float tanfovy, int H, int W, int32_t *radii_out,
                                         void *geom, int32_t *num_rendered_host, void *stream) {
    return preprocess_fwd_impl<true>(P, nullptr, means3D, scales, scale_stride, rots, opacities, colors, scale_mod, view,
                                     proj, tanfovx, tanfovy, H, W, radii_out, geom, num_rendered_host, stream);
}

extern "C" int splatco_preprocess_fwd_aa_counted(int P_max, const int32_t *P_dev, const float *means3D,
                                                 const float *scales, int scale_stride, const float *rots,
                                                 const float *opacities, const float *colors, float scale_mod,
                                                 const float *view, const float *proj, float tanfovx,
                                                 float tanfovy, int H, int W, int32_t *radii_out, void *geom,
                                                 int32_t *num_rendered_host, void *stream) {
    SPLATCO_REQUIRE(P_dev, "preprocess_fwd_aa_counted: null device count");
    return preprocess_fwd_impl<true>(P_max, reinterpret_cast<const uint32_t *>(P_dev), means3D, scales, scale_stride,
                                     rots, opacities, colors, scale_mod, view, proj, tanfovx, tanfovy, H, W, radii_out,
                                     geom, num_rendered_host, stream);
}

// AA: empty, or one AAOpacity (the antialiased backward), passed on to preprocess_bwd_kernel
template <bool DEPTH, typename... AA>
static int preprocess_bwd_impl(const char *name, int P, const float *means3D, const float *scales, int scale_stride,
                               const float *rots, float scale_mod, const float *view, const float *proj, float tanfovx,
                               float tanfovy, int H, int W, const int32_t *radii, const float *dL_dmean2D,
                               const float *dL_dconic, float *dL_dmeans3D, float *dL_dscales, float *dL_drots,
                               const float *dL_ddepth, void *stream, AA... aa) {
    SPLATCO_REQUIRE(P >= 0 && H > 0 && W > 0, "%s: bad sizes", name);
    if (P == 0) return 0;
    SPLATCO_REQUIRE(means3D && scales && rots && view && proj && radii && dL_dmean2D && dL_dconic &&
                    dL_dmeans3D && dL_dscales && dL_drots && (!DEPTH || dL_ddepth), "%s: null pointer", name);
    SPLATCO_REQUIRE(((uintptr_t)rots & 15) == 0 && ((uintptr_t)dL_drots & 15) == 0,
                    "%s: rotations / dL_drots must be 16-byte aligned", name);
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    if constexpr (DEPTH)
        preprocess_bwd_kernel<true, const float *, AA...><<<ceil_div(P, PRE_THREADS), PRE_THREADS, 0, (cudaStream_t)stream>>>(
            P, means3D, scales, scale_stride, rots, scale_mod, view, proj, tanfovx, tanfovy, fx, fy, radii,
            dL_dmean2D, dL_dconic, dL_dmeans3D, dL_dscales, dL_drots, dL_ddepth, aa...);
    else
        preprocess_bwd_kernel<false, AA...><<<ceil_div(P, PRE_THREADS), PRE_THREADS, 0, (cudaStream_t)stream>>>(
            P, means3D, scales, scale_stride, rots, scale_mod, view, proj, tanfovx, tanfovy, fx, fy, radii,
            dL_dmean2D, dL_dconic, dL_dmeans3D, dL_dscales, dL_drots, aa...);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" int splatco_preprocess_bwd(int P, const float *means3D, const float *scales, int scale_stride,
                                      const float *rots, float scale_mod, const float *view,
                                      const float *proj, float tanfovx, float tanfovy, int H, int W,
                                      const int32_t *radii, const float *dL_dmean2D,
                                      const float *dL_dconic, float *dL_dmeans3D, float *dL_dscales,
                                      float *dL_drots, void *stream) {
    return preprocess_bwd_impl<false>("preprocess_bwd", P, means3D, scales, scale_stride, rots, scale_mod, view, proj,
                                      tanfovx, tanfovy, H, W, radii, dL_dmean2D, dL_dconic, dL_dmeans3D, dL_dscales,
                                      dL_drots, nullptr, stream);
}

extern "C" int splatco_preprocess_bwd_depth(int P, const float *means3D, const float *scales, int scale_stride,
                                            const float *rots, float scale_mod, const float *view,
                                            const float *proj, float tanfovx, float tanfovy, int H, int W,
                                            const int32_t *radii, const float *dL_dmean2D,
                                            const float *dL_dconic, float *dL_dmeans3D, float *dL_dscales,
                                            float *dL_drots, const float *dL_ddepth, void *stream) {
    return preprocess_bwd_impl<true>("preprocess_bwd_depth", P, means3D, scales, scale_stride, rots, scale_mod, view,
                                     proj, tanfovx, tanfovy, H, W, radii, dL_dmean2D, dL_dconic, dL_dmeans3D, dL_dscales,
                                     dL_drots, dL_ddepth, stream);
}

extern "C" size_t splatco_camera_grad_ws_bytes(int n) { return camera_grad_ws_bytes(n); }

extern "C" int splatco_preprocess_bwd_camera(int P, const float *means3D, const float *scales, int scale_stride,
                                             const float *rots, float scale_mod, const float *view,
                                             const float *proj, float tanfovx, float tanfovy, int H, int W,
                                             const int32_t *radii, const float *dL_dmean2D,
                                             const float *dL_dconic, float *dL_dmeans3D, float *dL_dscales,
                                             float *dL_drots, const float *dL_ddepth, void *ws, float *dL_dview,
                                             float *dL_dproj, void *stream) {
    SPLATCO_REQUIRE(P >= 0 && H > 0 && W > 0, "preprocess_bwd_camera: bad sizes");
    SPLATCO_REQUIRE(dL_dview && dL_dproj && (P == 0 || ws), "preprocess_bwd_camera: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (P == 0) {
        SPLATCO_CHECK_CUDA(cudaMemsetAsync(dL_dview, 0, 16 * sizeof(float), st));
        SPLATCO_CHECK_CUDA(cudaMemsetAsync(dL_dproj, 0, 16 * sizeof(float), st));
        return 0;
    }
    // the per-Gaussian outputs: exactly the camera-off call
    const int rc = dL_ddepth ? preprocess_bwd_impl<true>("preprocess_bwd_camera", P, means3D, scales, scale_stride, rots,
                                                         scale_mod, view, proj, tanfovx, tanfovy, H, W, radii, dL_dmean2D,
                                                         dL_dconic, dL_dmeans3D, dL_dscales, dL_drots, dL_ddepth, stream)
                             : preprocess_bwd_impl<false>("preprocess_bwd_camera", P, means3D, scales, scale_stride, rots,
                                                          scale_mod, view, proj, tanfovx, tanfovy, H, W, radii, dL_dmean2D,
                                                          dL_dconic, dL_dmeans3D, dL_dscales, dL_drots, nullptr, stream);
    if (rc) return rc;
    const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
    const int nb = ceil_div(P, PRE_THREADS);
    float *part = (float *)ws;
    preprocess_bwd_camera_kernel<><<<nb, PRE_THREADS, 0, st>>>(P, means3D, scales, scale_stride, rots, scale_mod, view, proj,
                                                             tanfovx, tanfovy, fx, fy, radii, dL_dmean2D, dL_dconic,
                                                             dL_ddepth, part);
    SPLATCO_CHECK_LAUNCH();
    camera_sum_kernel<<<1, 1024, 0, st>>>(nb, 32, 16, 1.0f, part, dL_dview, dL_dproj);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" int splatco_preprocess_bwd_aa(int P, const float *means3D, const float *scales, int scale_stride,
                                         const float *rots, float scale_mod, const float *view,
                                         const float *proj, float tanfovx, float tanfovy, int H, int W,
                                         const int32_t *radii, const float *dL_dmean2D,
                                         const float *dL_dconic, float *dL_dmeans3D, float *dL_dscales,
                                         float *dL_drots, const float *opacities, float *dL_dopacity,
                                         const float *dL_ddepth, void *ws, float *dL_dview, float *dL_dproj,
                                         void *stream) {
    SPLATCO_REQUIRE(P >= 0 && H > 0 && W > 0, "preprocess_bwd_aa: bad sizes");
    const bool camera = dL_dview || dL_dproj;
    SPLATCO_REQUIRE(!camera || (dL_dview && dL_dproj && (P == 0 || ws)), "preprocess_bwd_aa: camera outputs need "
                    "dL_dview, dL_dproj and ws together");
    cudaStream_t st = (cudaStream_t)stream;
    if (P == 0) {
        if (camera) {
            SPLATCO_CHECK_CUDA(cudaMemsetAsync(dL_dview, 0, 16 * sizeof(float), st));
            SPLATCO_CHECK_CUDA(cudaMemsetAsync(dL_dproj, 0, 16 * sizeof(float), st));
        }
        return 0;
    }
    SPLATCO_REQUIRE(opacities && dL_dopacity, "preprocess_bwd_aa: null pointer");
    const AAOpacity aa{opacities, dL_dopacity};
    if (camera) {
        // before the per-Gaussian kernel: it reads dL_dopacity as the blend wrote it
        SPLATCO_REQUIRE(means3D && scales && rots && view && proj && radii && dL_dmean2D && dL_dconic,
                        "preprocess_bwd_aa: null pointer");
        SPLATCO_REQUIRE(((uintptr_t)rots & 15) == 0, "preprocess_bwd_aa: rotations must be 16-byte aligned");
        const float fx = (float)W / (2.0f * tanfovx), fy = (float)H / (2.0f * tanfovy);
        const int nb = ceil_div(P, PRE_THREADS);
        float *part = (float *)ws;
        preprocess_bwd_camera_kernel<AAOpacity><<<nb, PRE_THREADS, 0, st>>>(
            P, means3D, scales, scale_stride, rots, scale_mod, view, proj, tanfovx, tanfovy, fx, fy, radii, dL_dmean2D,
            dL_dconic, dL_ddepth, part, aa);
        SPLATCO_CHECK_LAUNCH();
        camera_sum_kernel<<<1, 1024, 0, st>>>(nb, 32, 16, 1.0f, part, dL_dview, dL_dproj);
        SPLATCO_CHECK_LAUNCH();
    }
    return dL_ddepth ? preprocess_bwd_impl<true>("preprocess_bwd_aa", P, means3D, scales, scale_stride, rots, scale_mod,
                                                 view, proj, tanfovx, tanfovy, H, W, radii, dL_dmean2D, dL_dconic,
                                                 dL_dmeans3D, dL_dscales, dL_drots, dL_ddepth, stream, aa)
                     : preprocess_bwd_impl<false>("preprocess_bwd_aa", P, means3D, scales, scale_stride, rots, scale_mod,
                                                  view, proj, tanfovx, tanfovy, H, W, radii, dL_dmean2D, dL_dconic,
                                                  dL_dmeans3D, dL_dscales, dL_drots, nullptr, stream, aa);
}
