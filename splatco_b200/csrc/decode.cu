// Anchor decode (generate_neural_gaussians) forward + backward on sm_100a.
// Reference being replaced (file:line in /root/reference):
//   gaussian_renderer/__init__.py:18-116   gather visible rows, geo features, MLP heads, mask, compaction
//   scene/gaussian_model.py:149-169        FeaturePlanes.forward  (sum over levels of BN+Linear branches)
//   scene/grids.py:146-201                 tri-plane bilinear gather (grid_sample, align_corners=True, zeros)
//   scene/gaussian_model.py:307-337        opacity / cov / colour heads
//
// v1 structure (fp32 throughout, the reference's numerics): the decode is expressed as
//   gather(+BN batch statistics) -> fold BN into the Linear weights -> a chain of small row-major GEMMs
//   (hand-written SIMT SGEMM below) with fused epilogues -> mask/scan/compaction,
// and the backward as the transposed chain plus split-K weight-gradient GEMMs.  BatchNorm in train mode
// needs grid-wide statistics before the first Linear, and its backward needs two grid-wide sums; both
// reduce to the column sums S0 and the matrices S1 = dY^T X accumulated by the same GEMM kernel, so no
// separate BN kernels exist (derivation in DESIGN.md §decode).
#include "common.cuh"

namespace splatco {

constexpr int KO = 10;                 // n_offsets the kernels are specialised for
constexpr int FD = 32;                 // feat_dim
constexpr int GD = FD + 3 + 3 * KO + 6;  // 71: [feat | anchor | offsets | scaling]
constexpr int XI = 100;                // x100 = [feat 32 | dir 3 | dist 1 | geo 64]
constexpr int HD = 96;                 // 3 heads x 32 hidden
constexpr int ZD = 112;                // 10 + 70 + 30 outputs, padded to 112
constexpr int DEC_MAX_DP = 96;

inline int ru4(int x) { return (x + 3) & ~3; }

struct DecDims {
    int V, rc, level, DP, LDX;
};
inline DecDims dec_dims(int V, int rc, int level) {
    DecDims d;
    d.V = V; d.rc = rc; d.level = level;
    d.DP = rc * (level == 0 ? 6 : (level == 1 ? 9 : 12));
    d.LDX = ru4(d.DP + GD);
    return d;
}

}  // namespace splatco
#include "decode_tc.cuh"
#include "decode_tc_bwd.cuh"
namespace splatco {

// ---- forward workspace -------------------------------------------------------------------------------
enum FwdChunk { F_X, F_STATS, F_MU, F_RSTD, F_WPT, F_WCT, F_BGEO, F_W1T, F_B1E, F_W2T, F_B2, F_WPG, F_WCG,
                F_XIN, F_H, F_Z, F_MASKBITS, F_OFFS, F_BSUM, F_BOFF, F_TOTAL, F_XT, F_BA, F_W1B, F_W2B, F_W2R, F_W1R, F_WPCR, F_NCHUNK };

static size_t dec_fwd_offsets(const DecDims &d, size_t off[F_NCHUNK + 1]) {
    const size_t V = (size_t)(d.V > 0 ? d.V : 0);
    const size_t nb = (V + 255) / 256;
    size_t o = 0;
    auto put = [&](int c, size_t bytes) { off[c] = o; o += align_up(bytes); };
    put(F_X, V * d.LDX * 4);
    put(F_STATS, 2 * (size_t)d.LDX * 8);
    put(F_MU, d.LDX * 4); put(F_RSTD, d.LDX * 4);
    put(F_WPT, DEC_MAX_DP * 32 * 4); put(F_WCT, GD * 32 * 4); put(F_BGEO, 64 * 4);
    put(F_W1T, XI * HD * 4); put(F_B1E, HD * 4);
    put(F_W2T, HD * ZD * 4); put(F_B2, ZD * 4);
    put(F_WPG, 32 * DEC_MAX_DP * 4); put(F_WCG, 32 * GD * 4);
    put(F_XIN, V * XI * 4); put(F_H, V * HD * 4); put(F_Z, V * ZD * 4);
    put(F_MASKBITS, V * 4); put(F_OFFS, V * 4); put(F_BSUM, nb * 4); put(F_BOFF, nb * 4); put(F_TOTAL, 4);
    // tensor-core path: X in 128-row tile / 16-byte chunk layout, pre-split weight tiles
    const size_t ntiles = (V + TC_ROWS - 1) / TC_ROWS;
    put(F_XT, d.rc <= TC_MAX_RC ? ntiles * tc_tile_chunks(d.DP) * TC_CHUNK : 0);
    put(F_BA, 2 * TC_BA_HALF); put(F_W1B, 2 * TC_W1_HALF); put(F_W2B, 2 * TC_W2_HALF);
    put(F_W2R, 2 * TCB_W2R_HALF); put(F_W1R, 2 * TCB_W1R_HALF); put(F_WPCR, 2 * TCB_WPC_HALF);   // backward-chain weight tiles
    off[F_NCHUNK] = o;
    return o;
}

// ---- backward workspace ------------------------------------------------------------------------------
enum BwdChunk { B_DZ, B_DH, B_DX, B_DXH, B_DGA, B_GW2T, B_GB2, B_GW1T, B_GB1, B_S1, B_S0, B_M1, B_M2, B_NCHUNK };

static size_t dec_bwd_offsets(const DecDims &d, size_t off[B_NCHUNK + 1]) {
    const size_t V = (size_t)(d.V > 0 ? d.V : 0);
    size_t o = 0;
    auto put = [&](int c, size_t bytes) { off[c] = o; o += align_up(bytes); };
    put(B_DZ, V * ZD * 4); put(B_DH, V * HD * 4); put(B_DX, V * XI * 4); put(B_DXH, V * d.LDX * 4);
    put(B_DGA, V * 40 * 4);
    put(B_GW2T, HD * ZD * 4); put(B_GB2, ZD * 4); put(B_GW1T, XI * HD * 4); put(B_GB1, HD * 4);
    put(B_S1, 32 * (size_t)d.LDX * 4); put(B_S0, 64 * 4); put(B_M1, d.LDX * 4); put(B_M2, d.LDX * 4);
    off[B_NCHUNK] = o;
    return o;
}

// =======================================================================================================
// Generic SIMT SGEMM: C[M,N] (+)= epi( sum_k A(m,k) B(k,n) ),  64x32 tile, 256 threads, 2x4 per thread.
//   A(m,k) = TA ? A[k*lda+m] : A[m*lda+k]      B(k,n) = TB ? B[n*ldb+k] : B[k*ldb+n]
//   gridDim.z > 1 => split-K over chunks of `kchunk`, results atomically added (C pre-zeroed, no epilogue).
// =======================================================================================================
constexpr int GBM = 64, GBN = 32, GBK = 16;

template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
sgemm_kernel(int M, int N, int K, const float *__restrict__ A, int lda, const float *__restrict__ B, int ldb,
             float *__restrict__ C, int ldc, const float *__restrict__ bias, int relu,
             const float *__restrict__ gate, int ldg, int kchunk) {
    __shared__ float As[GBK][GBM + 4];
    __shared__ float Bs[GBK][GBN + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * GBM, n0 = blockIdx.y * GBN;
    const int kbeg = kchunk > 0 ? blockIdx.z * kchunk : 0;
    const int kend = kchunk > 0 ? min(K, kbeg + kchunk) : K;
    const int ty = tid >> 3, tx = tid & 7;       // rows ty*2..+1, cols tx*4..+3
    float acc[2][4] = {};
    for (int k0 = kbeg; k0 < kend; k0 += GBK) {
        // A tile: 64 x 16
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + i * 256;
            int m, k;
            if (TA) { m = e & 63; k = e >> 6; } else { k = e & 15; m = e >> 4; }
            const int gm = m0 + m, gk = k0 + k;
            float v = 0.f;
            if (gm < M && gk < kend) v = TA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
            As[k][m] = v;
        }
        // B tile: 16 x 32
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int e = tid + i * 256;
            int n, k;
            if (TB) { k = e & 15; n = e >> 4; } else { n = e & 31; k = e >> 5; }
            const int gn = n0 + n, gk = k0 + k;
            float v = 0.f;
            if (gn < N && gk < kend) v = TB ? B[(size_t)gn * ldb + gk] : B[(size_t)gk * ldb + gn];
            Bs[k][n] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GBK; ++k) {
            const float a0 = As[k][ty * 2], a1 = As[k][ty * 2 + 1];
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            acc[0][0] = fmaf(a0, b.x, acc[0][0]); acc[0][1] = fmaf(a0, b.y, acc[0][1]);
            acc[0][2] = fmaf(a0, b.z, acc[0][2]); acc[0][3] = fmaf(a0, b.w, acc[0][3]);
            acc[1][0] = fmaf(a1, b.x, acc[1][0]); acc[1][1] = fmaf(a1, b.y, acc[1][1]);
            acc[1][2] = fmaf(a1, b.z, acc[1][2]); acc[1][3] = fmaf(a1, b.w, acc[1][3]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int gm = m0 + ty * 2 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            float v = acc[i][j];
            if (kchunk > 0) { atomicAdd(&C[(size_t)gm * ldc + gn], v); continue; }
            if (bias) v += bias[gn];
            if (relu) v = fmaxf(v, 0.f);
            if (gate) v = gate[(size_t)gm * ldg + gn] > 0.f ? v : 0.f;
            C[(size_t)gm * ldc + gn] = v;
        }
    }
}

template <bool TA, bool TB>
static int sgemm(cudaStream_t st, int M, int N, int K, const float *A, int lda, const float *B, int ldb, float *C,
                 int ldc, const float *bias = nullptr, int relu = 0, const float *gate = nullptr, int ldg = 0,
                 int kchunk = 0) {
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    dim3 grid(ceil_div(M, GBM), ceil_div(N, GBN), kchunk > 0 ? ceil_div(K, kchunk) : 1);
    sgemm_kernel<TA, TB><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, C, ldc, bias, relu, gate, ldg, kchunk);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

// column sums: out[n] += sum_m A[m*lda + n]   (out pre-zeroed)
__global__ void __launch_bounds__(128)
colsum_kernel(int M, int N, const float *__restrict__ A, int lda, float *__restrict__ out, int rows_per_cta) {
    const int n = blockIdx.y * 128 + threadIdx.x;
    if (n >= N) return;
    const int mbeg = blockIdx.x * rows_per_cta, mend = min(M, mbeg + rows_per_cta);
    float s = 0.f;
    for (int m = mbeg; m < mend; ++m) s += A[(size_t)m * lda + n];
    atomicAdd(&out[n], s);
}

// =======================================================================================================
// Gather: one warp per visible anchor; lanes run over output channels so that X rows are written
// coalesced; BN batch statistics (sum, sum of squares) accumulated per lane, reduced per CTA, then fp64 atomics.
// =======================================================================================================
struct DecPtrs {
    const float *anchor_feat, *anchor, *offset, *scaling;
    const int32_t *vis;
    const float *plane[3][3];
    const float *att[3];
    int E[3];
    const float *mn, *mx, *cam;      // device pointers (3 floats each)
    const float *noise;
    float noise_q;                   // != 0: add U(-.5,.5) * noise_q to the plane features of levels >= 1, generated here
    unsigned long long noise_seed;
    int packed;                      // 1: planes are [E,E,8] channel-last (splatco_pack_planes), 0: [rc,E,E]
};

struct Bilin { int i00, i01, i10, i11; float w00, w01, w10, w11; };

// u indexes plane rows (size E), v indexes columns (size E): what grid_sample(align_corners=True) does
__device__ __forceinline__ Bilin bilin_setup(float u, float v, int E) {
    const float fu = (u + 1.f) * 0.5f * (float)(E - 1);
    const float fv = (v + 1.f) * 0.5f * (float)(E - 1);
    const float u0f = floorf(fu), v0f = floorf(fv);
    const int u0 = (int)u0f, v0 = (int)v0f, u1 = u0 + 1, v1 = v0 + 1;
    const float wu1 = fu - u0f, wv1 = fv - v0f, wu0 = 1.f - wu1, wv0 = 1.f - wv1;
    const bool iu0 = u0 >= 0 && u0 < E, iu1 = u1 >= 0 && u1 < E, iv0 = v0 >= 0 && v0 < E, iv1 = v1 >= 0 && v1 < E;
    Bilin b;
    b.i00 = (iu0 && iv0) ? u0 * E + v0 : -1; b.w00 = wu0 * wv0;
    b.i01 = (iu0 && iv1) ? u0 * E + v1 : -1; b.w01 = wu0 * wv1;
    b.i10 = (iu1 && iv0) ? u1 * E + v0 : -1; b.w10 = wu1 * wv0;
    b.i11 = (iu1 && iv1) ? u1 * E + v1 : -1; b.w11 = wu1 * wv1;
    return b;
}
// ts = texel stride in floats (1 for [rc,E,E] planes, 8 for channel-last planes)
__device__ __forceinline__ float bilin_fetch(const float *__restrict__ p, const Bilin &b, int ts) {
    float r = 0.f;
    if (b.i00 >= 0) r = fmaf(__ldg(p + (size_t)b.i00 * ts), b.w00, r);
    if (b.i01 >= 0) r = fmaf(__ldg(p + (size_t)b.i01 * ts), b.w01, r);
    if (b.i10 >= 0) r = fmaf(__ldg(p + (size_t)b.i10 * ts), b.w10, r);
    if (b.i11 >= 0) r = fmaf(__ldg(p + (size_t)b.i11 * ts), b.w11, r);
    return r;
}
__device__ __forceinline__ void bilin_scatter(float *__restrict__ p, const Bilin &b, float g, int ts) {
    if (b.i00 >= 0) atomicAdd(p + (size_t)b.i00 * ts, g * b.w00);
    if (b.i01 >= 0) atomicAdd(p + (size_t)b.i01 * ts, g * b.w01);
    if (b.i10 >= 0) atomicAdd(p + (size_t)b.i10 * ts, g * b.w10);
    if (b.i11 >= 0) atomicAdd(p + (size_t)b.i11 * ts, g * b.w11);
}

// channel c of the plane block -> (level, plane 0..2, attended?, channel within plane)
__device__ __forceinline__ void plane_channel(int c, int rc, int &lvl, int &pl, int &att, int &ch) {
    if (c < 6 * rc) { lvl = 0; const int g = c / rc; pl = g >> 1; att = g & 1; ch = c - g * rc; }
    else if (c < 9 * rc) { lvl = 1; const int cc = c - 6 * rc; pl = cc / rc; att = 0; ch = cc - pl * rc; }
    else { lvl = 2; const int cc = c - 9 * rc; pl = cc / rc; att = 0; ch = cc - pl * rc; }
}

__device__ __forceinline__ void norm_coords(const DecPtrs &p, float ax, float ay, float az, float ind[3]) {
    const float m0 = __ldg(p.mn), m1 = __ldg(p.mn + 1), m2 = __ldg(p.mn + 2);
    ind[0] = (ax - m0) / (__ldg(p.mx) - m0) * 2.f - 1.f;
    ind[1] = (ay - m1) / (__ldg(p.mx + 1) - m1) * 2.f - 1.f;
    ind[2] = (az - m2) / (__ldg(p.mx + 2) - m2) * 2.f - 1.f;
}
// plane 0 = xy (rows X, cols Y), 1 = xz (rows X, cols Z), 2 = yz (rows Y, cols Z)   [grids.py:148-150]
__device__ __forceinline__ void plane_axes(int pl, const float ind[3], float &u, float &v) {
    u = pl == 2 ? ind[1] : ind[0];
    v = pl == 0 ? ind[1] : ind[2];
}

// What plane column c samples: resolved once per CTA into shared memory (16 bytes per column) instead of once per
// (anchor, column) in registers -- plane_channel() costs two integer divisions and the base-pointer selection a chain
// of selects, ~50 instructions per use, and both kernels below are bound by instructions in flight.
struct __align__(16) ColDesc { const float *base; int E; int axis; };
__device__ __forceinline__ void build_col_table(ColDesc *tab, int DP, int rc, const int *E, const float *const (*plane)[3],
                                                const float *const *att, int packed) {
    for (int c = threadIdx.x; c < DP; c += blockDim.x) {
        int lvl, pl, a, ch;
        plane_channel(c, rc, lvl, pl, a, ch);
        const float *b = a ? att[pl] : plane[lvl][pl];
        ColDesc d;
        d.E = E[lvl];
        d.axis = pl;
        d.base = b ? b + (packed ? (size_t)ch : (size_t)ch * d.E * d.E) : nullptr;
        tab[c] = d;
    }
    __syncthreads();
}

// U(-0.5, 0.5) from a counter-based generator: two rounds of a 64-bit mix (splitmix64 finaliser) of (seed, element
// index).  The reference draws torch.empty_like(feat).uniform_(-0.5, 0.5) * Q (scene/grids.py:159-164): any
// independent uniform stream is equivalent; this one is reproducible from torch's seed and the call counter.
__device__ __forceinline__ float uniform_pm_half(unsigned long long seed, unsigned long long idx) {
    unsigned long long z = seed + idx * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (float)(unsigned)(z >> 40) * (1.0f / 16777216.0f) - 0.5f;        // 24 random bits
}

constexpr int GATHER_WARPS = 8;

__global__ void __launch_bounds__(GATHER_WARPS * 32, 3)
dec_gather_kernel(DecPtrs p, int V, int rc, int DP, int LDX, float *__restrict__ X, float *__restrict__ XIN,
                  double *__restrict__ stats, float *__restrict__ XT) {
    extern __shared__ float s_red[];     // [GATHER_WARPS][2][LDX]
    __shared__ ColDesc s_col[DEC_MAX_DP];
    build_col_table(s_col, DP, rc, p.E, p.plane, p.att, p.packed);
    const int ts = p.packed ? 8 : 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps_total = gridDim.x * GATHER_WARPS;
    constexpr int MAXC = 6;              // ceil((96+71)/32)
    float sum[MAXC], sq[MAXC];
#pragma unroll
    for (int j = 0; j < MAXC; ++j) sum[j] = sq[j] = 0.f;
    const int ncols = DP + GD;
    for (int v = blockIdx.x * GATHER_WARPS + warp; v < V; v += nwarps_total) {
        const int i = p.vis[v];
        const float ax = __ldg(p.anchor + 3 * (size_t)i), ay = __ldg(p.anchor + 3 * (size_t)i + 1), az = __ldg(p.anchor + 3 * (size_t)i + 2);
        float ind[3];
        norm_coords(p, ax, ay, az, ind);
        float *xrow = X + (size_t)v * LDX;
        // phase 1: every load of this anchor (up to 4 texels x 6 column groups per lane) with no store in between,
        // so they are all in flight together; phase 2 writes the row.  (One group's loads at a time made the
        // plane-texel latency the critical path: ncu showed ~40 % of the stall samples on these lines.)
        float vals[MAXC];
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane + 32 * j;
            float val = 0.f;
            if (c < DP) {
                const ColDesc cd = s_col[c];
                float u, w;
                plane_axes(cd.axis, ind, u, w);
                // (channel-last planes: the rc channels of a texel share one 32-byte sector)
                val = bilin_fetch(cd.base, bilin_setup(u, w, cd.E), ts);
                if (c >= 6 * rc) {
                    if (p.noise) val += __ldg(p.noise + (size_t)v * (DP - 6 * rc) + (c - 6 * rc));
                    else if (p.noise_q != 0.f) val = fmaf(uniform_pm_half(p.noise_seed, (unsigned long long)v * DP + c), p.noise_q, val);
                }
            } else if (c < ncols) {
                const int g = c - DP;
                if (g < FD) val = __ldg(p.anchor_feat + (size_t)i * FD + g);
                else if (g < FD + 3) val = g == FD ? ax : (g == FD + 1 ? ay : az);
                else if (g < FD + 3 + 3 * KO) val = __ldg(p.offset + (size_t)i * 3 * KO + (g - FD - 3));
                else val = __ldg(p.scaling + (size_t)i * 6 + (g - FD - 3 - 3 * KO));
            }
            vals[j] = val;
        }
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane + 32 * j;
            if (c >= ncols) break;
            const float val = vals[j];
            xrow[c] = val;
            if (XT) {       // tile / chunk layout for the tensor-core kernel: [tile][chunk][row][4]; g starts on a fresh chunk
                const int cc = c < DP ? c : ((DP + 3) & ~3) + (c - DP);
                const size_t cell = ((size_t)(v >> 7) * tc_tile_chunks(DP) + (cc >> 2)) * TC_ROWS + (v & 127);
                XT[cell * 4 + (cc & 3)] = val;
            }
            sum[j] += val; sq[j] = fmaf(val, val, sq[j]);
        }
        if (XT) {           // zero the padding of the last P chunk and the g pad column (garbage * 0 could be NaN)
            const int npc = (DP + 3) >> 2;
            const size_t tb = (size_t)(v >> 7) * tc_tile_chunks(DP);
            if (lane < 4 * npc - DP) XT[((tb + npc - 1) * TC_ROWS + (v & 127)) * 4 + (DP & 3) + lane] = 0.f;
            if (lane == 0) XT[((tb + npc + 17) * TC_ROWS + (v & 127)) * 4 + 3] = 0.f;
        }
        if (lane < LDX - ncols) xrow[ncols + lane] = 0.f;       // zero the row padding
        // x100 head: feat | dir | dist   (gaussian_renderer/__init__.py:34-38,55)
        float *xin = XIN + (size_t)v * XI;
        xin[lane] = __ldg(p.anchor_feat + (size_t)i * FD + lane);
        if (lane < 4) {
            const float vx = ax - __ldg(p.cam), vy = ay - __ldg(p.cam + 1), vz = az - __ldg(p.cam + 2);
            const float dist = sqrtf(vx * vx + vy * vy + vz * vz);
            const float dd = lane == 0 ? vx / dist : (lane == 1 ? vy / dist : (lane == 2 ? vz / dist : dist));
            xin[FD + lane] = dd;
            if (XT) XT[(((size_t)(v >> 7) * tc_tile_chunks(DP) + ((DP + 3) >> 2) + 18) * TC_ROWS + (v & 127)) * 4 + lane] = dd;
        }
    }
    // CTA reduction of the statistics, then one fp64 atomic per channel per CTA
    float *mine = s_red + (size_t)warp * 2 * LDX;
#pragma unroll
    for (int j = 0; j < MAXC; ++j) {
        const int c = lane + 32 * j;
        if (c < ncols) { mine[c] = sum[j]; mine[LDX + c] = sq[j]; }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
        double s = 0.0, q = 0.0;
#pragma unroll
        for (int w = 0; w < GATHER_WARPS; ++w) { s += (double)s_red[(size_t)w * 2 * LDX + c]; q += (double)s_red[(size_t)w * 2 * LDX + LDX + c]; }
        atomicAdd(&stats[c], s);
        atomicAdd(&stats[LDX + c], q);
    }
}

// =======================================================================================================
// Fold kernel (one CTA): batch mean / rstd, running-stat update, BN folded into the Linear weights,
// head weights re-laid out as [K][N] GEMM operands.
// =======================================================================================================
struct DecWeights {
    const float *bn_w[3], *bn_b[3], *lin_w[3], *lin_b[3];        // plane branch per level
    const float *cbn_w[3], *cbn_b[3], *clin_w[3], *clin_b[3];    // context branch per level
    float *bn_rm[3], *bn_rv[3], *cbn_rm[3], *cbn_rv[3];          // running stats (updated in place; may be null)
    long long *bn_nbt[3], *cbn_nbt[3];
    const float *w1[3], *b1[3], *w2[3], *b2[3];                  // opacity, cov, colour heads
    const float *app_vec;
    int use_dist[3];
    int app_dim;
    float eps, momentum;
};

__device__ __forceinline__ int level_dim(int l, int rc) { return l == 0 ? 6 * rc : 3 * rc; }
__device__ __forceinline__ int level_base(int l, int rc) { return l == 0 ? 0 : (l == 1 ? 6 * rc : 9 * rc); }

// Launched with several CTAs: every output depends only on the batch statistics and the source weights, so
// each CTA first derives mean / rstd of all channels into shared memory and then takes a grid-stride share of
// every table; the BatchNorm running statistics are updated by CTA 0 alone.
constexpr int FOLD_CTAS = 16;
__global__ void __launch_bounds__(256)
dec_fold_kernel(DecWeights w, int V_host, const int32_t *__restrict__ Vdev, int rc, int level, int DP, int LDX, const double *__restrict__ stats,
                float *__restrict__ mu, float *__restrict__ rstd, float *__restrict__ WpT, float *__restrict__ WcT,
                float *__restrict__ bgeo, float *__restrict__ W1T, float *__restrict__ b1e, float *__restrict__ W2T,
                float *__restrict__ b2, float *__restrict__ WpG, float *__restrict__ WcG, int update_running) {
    __shared__ float s_mu[DEC_MAX_DP + GD + 4], s_rstd[DEC_MAX_DP + GD + 4];
    const int V = Vdev ? __ldg(Vdev) : V_host;          // (row count still on the device: splatco_decode_desc::V_dev)
    const int tid = threadIdx.x;
    const int gtid = blockIdx.x * 256 + tid, nthr = gridDim.x * 256;
    const int ncols = DP + GD;
    const bool first = blockIdx.x == 0;
    for (int c = tid; c < LDX; c += 256) {
        if (c >= ncols) { s_mu[c] = 0.f; s_rstd[c] = 0.f; if (first) { mu[c] = 0.f; rstd[c] = 0.f; } continue; }
        const double mean = stats[c] / (double)V;
        double var = stats[LDX + c] / (double)V - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mu[c] = (float)mean;
        s_rstd[c] = (float)(1.0 / sqrt(var + (double)w.eps));
        if (!first) continue;
        mu[c] = s_mu[c]; rstd[c] = s_rstd[c];
        if (update_running && V >= 2) {       // (V < 2 is an error the caller raises; with V_dev it is only known here)
            const float unb = (float)(V > 1 ? var * (double)V / (double)(V - 1) : var);
            const float m = w.momentum;
            if (c < DP) {
                int l = c < 6 * rc ? 0 : (c < 9 * rc ? 1 : 2);
                const int cl = c - level_base(l, rc);
                if (w.bn_rm[l]) w.bn_rm[l][cl] = (1.f - m) * w.bn_rm[l][cl] + m * (float)mean;
                if (w.bn_rv[l]) w.bn_rv[l][cl] = (1.f - m) * w.bn_rv[l][cl] + m * unb;
            } else {
                const int g = c - DP;
                for (int l = 0; l <= level; ++l) {
                    if (w.cbn_rm[l]) w.cbn_rm[l][g] = (1.f - m) * w.cbn_rm[l][g] + m * (float)mean;
                    if (w.cbn_rv[l]) w.cbn_rv[l][g] = (1.f - m) * w.cbn_rv[l][g] + m * unb;
                }
            }
        }
    }
    if (first && update_running && V >= 2 && tid == 0)
        for (int l = 0; l <= level; ++l) {
            if (w.bn_nbt[l]) *w.bn_nbt[l] += 1;
            if (w.cbn_nbt[l]) *w.cbn_nbt[l] += 1;
        }
    __syncthreads();
    // plane branch
    for (int e = gtid; e < DP * 32; e += nthr) {
        const int c = e >> 5, o = e & 31;
        const int l = c < 6 * rc ? 0 : (c < 9 * rc ? 1 : 2);
        const int d = level_dim(l, rc), cl = c - level_base(l, rc);
        const float gw = w.bn_w[l][cl] * w.lin_w[l][o * d + cl];
        WpG[o * DP + c] = gw;
        WpT[c * 32 + o] = gw * s_rstd[c];
    }
    // context branch (all active levels normalise the same g with the same batch statistics)
    for (int e = gtid; e < GD * 32; e += nthr) {
        const int g = e >> 5, o = e & 31;
        float gw = 0.f;
        for (int l = 0; l <= level; ++l) gw = fmaf(w.cbn_w[l][g], w.clin_w[l][o * GD + g], gw);
        WcG[o * GD + g] = gw;
        WcT[g * 32 + o] = gw * s_rstd[DP + g];
    }
    // geo bias: Linear bias + beta through the Linear - mean through the folded weights; one warp per output,
    // the warps of the whole grid share the 64 outputs
    {
        const int lane = tid & 31, gw_id = gtid >> 5, nwarps = nthr >> 5;
        for (int out = gw_id; out < 64; out += nwarps) {
            const int o = out & 31;
            float b = 0.f;
            if (out < 32) {
                for (int l = 0; l <= level; ++l) {
                    const int d = level_dim(l, rc), base = level_base(l, rc);
                    for (int cl = lane; cl < d; cl += 32) {
                        const float lw = w.lin_w[l][o * d + cl];
                        b = fmaf(w.bn_b[l][cl], lw, b);
                        b = fmaf(-s_mu[base + cl], w.bn_w[l][cl] * lw * s_rstd[base + cl], b);
                    }
                }
            } else {
                for (int g = lane; g < GD; g += 32) {
                    float gwsum = 0.f;
                    for (int l = 0; l <= level; ++l) {
                        const float lw = w.clin_w[l][o * GD + g];
                        b = fmaf(w.cbn_b[l][g], lw, b);
                        gwsum = fmaf(w.cbn_w[l][g], lw, gwsum);
                    }
                    b = fmaf(-s_mu[DP + g], gwsum * s_rstd[DP + g], b);
                }
            }
#pragma unroll
            for (int dd = 16; dd > 0; dd >>= 1) b += __shfl_xor_sync(0xffffffffu, b, dd);
            if (lane == 0) {
                float bias = 0.f;
                for (int l = 0; l <= level; ++l) bias += out < 32 ? w.lin_b[l][o] : w.clin_b[l][o];
                bgeo[out] = b + bias;
            }
        }
    }
    // hidden layer: x100 = [feat 32 | dir 3 | dist 1 | geo 64]; per-head torch layout is
    // [feat | dir | (dist) | geo | (appearance, colour head only)]
    for (int e = gtid; e < XI * HD; e += nthr) {
        const int k = e / HD, n = e - k * HD;
        const int hd = n >> 5, o = n & 31;
        const int dd = w.use_dist[hd];
        const int in_h = 35 + dd + 64 + (hd == 2 ? w.app_dim : 0);
        float v;
        if (k < 35) v = w.w1[hd][o * in_h + k];
        else if (k == 35) v = dd ? w.w1[hd][o * in_h + 35] : 0.f;
        else v = w.w1[hd][o * in_h + 35 + dd + (k - 36)];
        W1T[e] = v;
    }
    for (int n = gtid; n < HD; n += nthr) {
        const int hd = n >> 5, o = n & 31;
        float b = w.b1[hd][o];
        if (hd == 2 && w.app_dim > 0) {
            const int dd = w.use_dist[2];
            const int in_h = 35 + dd + 64 + w.app_dim;
            for (int a = 0; a < w.app_dim; ++a) b = fmaf(w.w1[2][o * in_h + 35 + dd + 64 + a], w.app_vec[a], b);
        }
        b1e[n] = b;
    }
    // output layer as one block-diagonal [96][112] operand: cols [opacity 0..9 | cov 10..79 | colour 80..109]
    for (int e = gtid; e < HD * ZD; e += nthr) {
        const int i = e / ZD, j = e - i * ZD;
        const int hd_i = i >> 5, ii = i & 31;
        float v = 0.f;
        if (j < KO) { if (hd_i == 0) v = w.w2[0][j * 32 + ii]; }
        else if (j < 8 * KO) { if (hd_i == 1) v = w.w2[1][(j - KO) * 32 + ii]; }
        else if (j < 11 * KO) { if (hd_i == 2) v = w.w2[2][(j - 8 * KO) * 32 + ii]; }
        W2T[e] = v;
    }
    for (int j = gtid; j < ZD; j += nthr) {
        float v = 0.f;
        if (j < KO) v = w.b2[0][j];
        else if (j < 8 * KO) v = w.b2[1][j - KO];
        else if (j < 11 * KO) v = w.b2[2][j - 8 * KO];
        b2[j] = v;
    }
}

// =======================================================================================================
// Head activations, opacity mask, per-anchor survivor counts (first scan level)
// =======================================================================================================
// One thread per Z element (coalesced); a CTA covers 32 rows.  block_sums (one per 256 rows, pre-zeroed)
// receives the survivor counts for the scan.
constexpr int ACT_ROWS = 32;
__global__ void __launch_bounds__(256)
dec_heads_act_kernel(int V, float *__restrict__ Z, float *__restrict__ neural_opacity, uint8_t *__restrict__ mask_out,
                     uint32_t *__restrict__ maskbits, uint32_t *__restrict__ block_sums) {
    __shared__ uint32_t s_bits[ACT_ROWS];
    if (threadIdx.x < ACT_ROWS) s_bits[threadIdx.x] = 0;
    __syncthreads();
    const int row0 = blockIdx.x * ACT_ROWS;
    const int nrows = min(ACT_ROWS, V - row0);
    float *zb = Z + (size_t)row0 * ZD;
    for (int e = threadIdx.x; e < nrows * ZD; e += 256) {
        const int r = e / ZD, j = e - r * ZD;
        const float x = zb[e];
        if (j < KO) {
            const float t = tanhf(x);
            zb[e] = t;
            const size_t o = (size_t)(row0 + r) * KO + j;
            neural_opacity[o] = t;
            const bool m = t > 0.f;
            mask_out[o] = m ? 1 : 0;
            if (m) atomicOr(&s_bits[r], 1u << j);
        } else if (j >= 8 * KO && j < 11 * KO) {
            zb[e] = 1.f / (1.f + expf(-x));
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int r = threadIdx.x;
        uint32_t bits = 0;
        if (r < nrows) { bits = s_bits[r]; maskbits[row0 + r] = bits; }
        uint32_t s = __popc(bits);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (r == 0 && s) atomicAdd(&block_sums[row0 / 256], s);
    }
}

// exclusive per-anchor offsets from maskbits + scanned block offsets (same 256-wide partition)
__global__ void __launch_bounds__(256)
dec_offsets_kernel(int V_host, const int32_t *__restrict__ Vdev, const uint32_t *__restrict__ maskbits,
                   const uint32_t *__restrict__ block_offsets, uint32_t *__restrict__ offs) {
    __shared__ uint32_t s_warp[8];
    const int V = Vdev ? __ldg(Vdev) : V_host;
    const int v = blockIdx.x * 256 + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t c = v < V ? __popc(maskbits[v]) : 0u;
    uint32_t inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t n = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (uint32_t)d) inc += n; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) woff += (w < (int)warp) ? s_warp[w] : 0u;
    if (v < V) offs[v] = block_offsets[blockIdx.x] + woff + inc - c;
}

// compaction + post-processing (gaussian_renderer/__init__.py:96-111), one thread per (anchor, offset)
__global__ void __launch_bounds__(256)
dec_compact_kernel(int V, int LDX, int DP, const float *__restrict__ X, const float *__restrict__ Z,
                   const uint32_t *__restrict__ maskbits, const uint32_t *__restrict__ offs,
                   float *__restrict__ xyz, float *__restrict__ color, float *__restrict__ opacity,
                   float *__restrict__ scaling, float *__restrict__ rot) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= V * KO) return;
    const int v = t / KO, k = t - v * KO;
    const uint32_t bits = maskbits[v];
    if (!((bits >> k) & 1u)) return;
    const size_t j = offs[v] + __popc(bits & ((1u << k) - 1u));
    const float *g = X + (size_t)v * LDX + DP;       // [feat 32 | anchor 3 | offsets 30 | scaling 6]
    const float *z = Z + (size_t)v * ZD;
    const float *s6 = g + FD + 3 + 3 * KO;
    const float *of = g + FD + 3 + 3 * k;
    xyz[3 * j] = g[FD] + of[0] * s6[0];
    xyz[3 * j + 1] = g[FD + 1] + of[1] * s6[1];
    xyz[3 * j + 2] = g[FD + 2] + of[2] * s6[2];
    color[3 * j] = z[8 * KO + 3 * k]; color[3 * j + 1] = z[8 * KO + 3 * k + 1]; color[3 * j + 2] = z[8 * KO + 3 * k + 2];
    opacity[j] = z[k];
    const float *sr = z + KO + 7 * k;
    scaling[3 * j] = s6[3] / (1.f + expf(-sr[0]));
    scaling[3 * j + 1] = s6[4] / (1.f + expf(-sr[1]));
    scaling[3 * j + 2] = s6[5] / (1.f + expf(-sr[2]));
    const float n = fmaxf(sqrtf(sr[3] * sr[3] + sr[4] * sr[4] + sr[5] * sr[5] + sr[6] * sr[6]), 1e-12f);
    rot[4 * j] = sr[3] / n; rot[4 * j + 1] = sr[4] / n; rot[4 * j + 2] = sr[5] / n; rot[4 * j + 3] = sr[6] / n;
}

// =======================================================================================================
// Backward elementwise stages
// =======================================================================================================
// un-compaction: upstream gradients of the five compacted outputs -> dZ rows (pre-activation) and the
// direct (non-MLP) gradients of anchor / offsets / scaling.  One thread per (visible anchor, offset):
// a CTA covers 32 anchors x 10 offsets, so the 110 dZ entries of a row are written by 10 adjacent
// threads; the per-anchor sums over offsets (anchor 3 + scaling 6) are reduced in shared memory.
constexpr int UNC_ROWS = 32;
__global__ void __launch_bounds__(UNC_ROWS * KO)
dec_bwd_uncompact_kernel(int V, int LDX, int DP, const float *__restrict__ X, const float *__restrict__ Z,
                         const uint32_t *__restrict__ maskbits, const uint32_t *__restrict__ offs,
                         const float *__restrict__ d_xyz, const float *__restrict__ d_color,
                         const float *__restrict__ d_opacity, const float *__restrict__ d_scaling,
                         const float *__restrict__ d_rot, const float *__restrict__ d_nopac,
                         float *__restrict__ DZ, float *__restrict__ DGA) {
    __shared__ float s_sum[UNC_ROWS][9];
    const int tid = threadIdx.x;
    if (tid < UNC_ROWS * 9) (&s_sum[0][0])[tid] = 0.f;
    __syncthreads();
    const int vl = tid / KO, k = tid - vl * KO;
    const int v = blockIdx.x * UNC_ROWS + vl;
    if (v < V) {
        const uint32_t bits = maskbits[v];
        const float *g = X + (size_t)v * LDX + DP;
        const float *z = Z + (size_t)v * ZD;
        const float *s6 = g + FD + 3 + 3 * KO;
        float *dz = DZ + (size_t)v * ZD;
        float *dga = DGA + (size_t)v * 40;          // [anchor 3 | offsets 30 | scaling 6 | pad]
        const bool m = (bits >> k) & 1u;
        const float no = z[k];
        float dno = d_nopac ? d_nopac[(size_t)v * KO + k] : 0.f;
        float dof[3] = {0.f, 0.f, 0.f}, dc[3] = {0.f, 0.f, 0.f}, dsr[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (m) {
            const size_t j = offs[v] + __popc(bits & ((1u << k) - 1u));
            dno += d_opacity[j];
            const float gx = d_xyz[3 * j], gy = d_xyz[3 * j + 1], gz = d_xyz[3 * j + 2];
            const float *of = g + FD + 3 + 3 * k;
            dof[0] = gx * s6[0]; dof[1] = gy * s6[1]; dof[2] = gz * s6[2];
            atomicAdd(&s_sum[vl][0], gx); atomicAdd(&s_sum[vl][1], gy); atomicAdd(&s_sum[vl][2], gz);
            atomicAdd(&s_sum[vl][3], gx * of[0]); atomicAdd(&s_sum[vl][4], gy * of[1]); atomicAdd(&s_sum[vl][5], gz * of[2]);
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const float c = z[8 * KO + 3 * k + q];
                dc[q] = d_color[3 * j + q] * c * (1.f - c);
            }
            const float *sr = z + KO + 7 * k;
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const float sg = 1.f / (1.f + expf(-sr[q]));
                const float gsc = d_scaling[3 * j + q];
                dsr[q] = gsc * s6[3 + q] * sg * (1.f - sg);
                atomicAdd(&s_sum[vl][6 + q], gsc * sg);
            }
            const float nrm = sqrtf(sr[3] * sr[3] + sr[4] * sr[4] + sr[5] * sr[5] + sr[6] * sr[6]);
            const float n = fmaxf(nrm, 1e-12f);
            const float r0 = sr[3] / n, r1 = sr[4] / n, r2 = sr[5] / n, r3 = sr[6] / n;
            const float g0 = d_rot[4 * j], g1 = d_rot[4 * j + 1], g2 = d_rot[4 * j + 2], g3 = d_rot[4 * j + 3];
            if (nrm > 1e-12f) {
                const float dot = r0 * g0 + r1 * g1 + r2 * g2 + r3 * g3;
                dsr[3] = (g0 - r0 * dot) / n; dsr[4] = (g1 - r1 * dot) / n;
                dsr[5] = (g2 - r2 * dot) / n; dsr[6] = (g3 - r3 * dot) / n;
            } else {
                dsr[3] = g0 / n; dsr[4] = g1 / n; dsr[5] = g2 / n; dsr[6] = g3 / n;
            }
        }
        dz[k] = dno * (1.f - no * no);
#pragma unroll
        for (int q = 0; q < 7; ++q) dz[KO + 7 * k + q] = dsr[q];
#pragma unroll
        for (int q = 0; q < 3; ++q) { dz[8 * KO + 3 * k + q] = dc[q]; dga[3 + 3 * k + q] = dof[q]; }
        if (k == 0) { dz[11 * KO] = 0.f; dz[11 * KO + 1] = 0.f; dga[39] = 0.f; }
    }
    __syncthreads();
    if (v < V && k < 9) {
        // s_sum: [0..2] anchor, [3..5] scaling[0..2] (from xyz), [6..8] scaling[3..5]
        float *dga = DGA + (size_t)v * 40;
        const float val = s_sum[vl][k];
        if (k < 3) dga[k] = val; else dga[33 + (k - 3)] = val;
    }
}

// S0/S1 -> parameter gradients of the BN+Linear branches and the per-channel BN-backward constants m1, m2.
struct DecWeightGrads {
    float *bn_w[3], *bn_b[3], *lin_w[3], *lin_b[3];
    float *cbn_w[3], *cbn_b[3], *clin_w[3], *clin_b[3];
    float *w1[3], *b1[3], *w2[3], *b2[3];
    float *app_vec;
};

constexpr int BWD_FOLD_CTAS = 4, BWD_FOLD_SECTIONS = 11;
__global__ void __launch_bounds__(256)
dec_bwd_fold_kernel(DecWeights w, DecWeightGrads gw, int V, int rc, int level, int DP, int LDX,
                    const float *__restrict__ mu, const float *__restrict__ rstd, const float *__restrict__ WpG,
                    const float *__restrict__ WcG, const float *__restrict__ S1raw /*[32][LDX]*/,
                    const float *__restrict__ S0 /*[64]*/, const float *__restrict__ gW1T, const float *__restrict__ gb1,
                    const float *__restrict__ gW2T, const float *__restrict__ gb2, float *__restrict__ m1,
                    float *__restrict__ m2) {
    // Every output is independent: blockIdx.y selects one SECTION of the outputs (BN-backward constants, one level's plane
    // branch, one level's context branch, one head, the appearance vector) so that the sections -- each a short chain of
    // dependent global loads -- run side by side instead of one after the other in every CTA.
    const int tid = blockIdx.x * 256 + threadIdx.x, nthr = gridDim.x * 256;
    const int sec = blockIdx.y;
    const int ncols = DP + GD;
    const float invV = 1.f / (float)V;
    // S1[o][c] = sum_rows dgeo[o] * xhat[c] = rstd[c] * (S1raw[o][c] - mu[c] * S0branch[o])
    if (sec == 0)
    for (int c = tid; c < LDX; c += nthr) {
        if (c >= ncols) { m1[c] = 0.f; m2[c] = 0.f; continue; }
        const bool pl = c < DP;
        const float *WG = pl ? WpG : WcG;
        const int ldw = pl ? DP : GD, cc = pl ? c : c - DP;
        const float *S0b = pl ? S0 : S0 + 32;
        float a1 = 0.f, a2 = 0.f;
        for (int o = 0; o < 32; ++o) {
            const float s1 = rstd[c] * (S1raw[o * LDX + c] - mu[c] * S0b[o]);
            a1 = fmaf(WG[o * ldw + cc], S0b[o], a1);
            a2 = fmaf(WG[o * ldw + cc], s1, a2);
        }
        m1[c] = a1 * invV;
        m2[c] = a2 * invV;
    }
    // plane branch parameter grads
    for (int l = 0; l <= level; ++l) {
        const int d = level_dim(l, rc), base = level_base(l, rc);
        if (sec == 1 + l) {
        for (int e = tid; e < 32 * d; e += nthr) {
            const int o = e / d, cl = e - o * d, c = base + cl;
            const float s1 = rstd[c] * (S1raw[o * LDX + c] - mu[c] * S0[o]);
            if (gw.lin_w[l]) gw.lin_w[l][o * d + cl] += w.bn_w[l][cl] * s1 + w.bn_b[l][cl] * S0[o];
        }
        for (int cl = tid; cl < d; cl += nthr) {
            const int c = base + cl;
            float gg = 0.f, gb = 0.f;
            for (int o = 0; o < 32; ++o) {
                const float s1 = rstd[c] * (S1raw[o * LDX + c] - mu[c] * S0[o]);
                gg = fmaf(w.lin_w[l][o * d + cl], s1, gg);
                gb = fmaf(w.lin_w[l][o * d + cl], S0[o], gb);
            }
            if (gw.bn_w[l]) gw.bn_w[l][cl] += gg;
            if (gw.bn_b[l]) gw.bn_b[l][cl] += gb;
        }
        if (tid < 32 && gw.lin_b[l]) gw.lin_b[l][tid] += S0[tid];      // tid is grid-wide: only CTA 0 has tid < 32
        }
        if (sec != 4 + l) continue;
        // context branch
        for (int e = tid; e < 32 * GD; e += nthr) {
            const int o = e / GD, g = e - o * GD, c = DP + g;
            const float s1 = rstd[c] * (S1raw[o * LDX + c] - mu[c] * S0[32 + o]);
            if (gw.clin_w[l]) gw.clin_w[l][o * GD + g] += w.cbn_w[l][g] * s1 + w.cbn_b[l][g] * S0[32 + o];
        }
        for (int g = tid; g < GD; g += nthr) {
            const int c = DP + g;
            float gg = 0.f, gb = 0.f;
            for (int o = 0; o < 32; ++o) {
                const float s1 = rstd[c] * (S1raw[o * LDX + c] - mu[c] * S0[32 + o]);
                gg = fmaf(w.clin_w[l][o * GD + g], s1, gg);
                gb = fmaf(w.clin_w[l][o * GD + g], S0[32 + o], gb);
            }
            if (gw.cbn_w[l]) gw.cbn_w[l][g] += gg;
            if (gw.cbn_b[l]) gw.cbn_b[l][g] += gb;
        }
        if (tid < 32 && gw.clin_b[l]) gw.clin_b[l][tid] += S0[32 + tid];
    }
    // heads: un-fold gW1T[k][n] / gW2T[i][j] into torch layouts
    for (int hd = 0; hd < 3; ++hd) {
        if (sec != 7 + hd) continue;
        const int dd = w.use_dist[hd];
        const int app = hd == 2 ? w.app_dim : 0;
        const int in_h = 35 + dd + 64 + app;
        if (gw.w1[hd])
            for (int e = tid; e < 32 * in_h; e += nthr) {
                const int o = e / in_h, col = e - o * in_h;
                const int n = hd * 32 + o;
                float v;
                if (col < 35) v = gW1T[col * HD + n];
                else if (dd && col == 35) v = gW1T[35 * HD + n];
                else if (col < 35 + dd + 64) v = gW1T[(36 + col - 35 - dd) * HD + n];
                else v = gb1[n] * w.app_vec[col - 35 - dd - 64];
                gw.w1[hd][e] += v;
            }
        if (gw.b1[hd] && tid < 32) gw.b1[hd][tid] += gb1[hd * 32 + tid];
        const int nout = hd == 0 ? KO : (hd == 1 ? 7 * KO : 3 * KO);
        const int j0 = hd == 0 ? 0 : (hd == 1 ? KO : 8 * KO);
        if (gw.w2[hd])
            for (int e = tid; e < nout * 32; e += nthr) {
                const int j = e >> 5, ii = e & 31;
                gw.w2[hd][e] += gW2T[(hd * 32 + ii) * ZD + j0 + j];
            }
        if (gw.b2[hd])
            for (int j = tid; j < nout; j += nthr) gw.b2[hd][j] += gb2[j0 + j];
    }
    if (sec == 10 && gw.app_vec && w.app_dim > 0) {
        const int dd = w.use_dist[2];
        const int in_h = 35 + dd + 64 + w.app_dim;
        for (int a = tid; a < w.app_dim; a += nthr) {
            float s = 0.f;
            for (int o = 0; o < 32; ++o) s = fmaf(w.w1[2][o * in_h + 35 + dd + 64 + a], gb1[64 + o], s);
            gw.app_vec[a] += s;
        }
    }
}

// Final input gradients: BN backward through the folded branch (dx = rstd (dxhat - m1 - xhat m2)),
// bilinear scatter into the plane gradients, and the per-anchor rows of the N-row gradient tensors.
// One warp per visible anchor (same mapping as the gather).
struct DecInputGrads {
    float *anchor_feat, *anchor, *offset, *scaling;     // [N,*], visible rows accumulated (fire-and-forget REDs: a
                                                        // read-modify-write would stall on its own load)
    float *plane[3][3];
    float *att[3];
};

__global__ void __launch_bounds__(GATHER_WARPS * 32)
dec_bwd_inputs_kernel(DecPtrs p, DecInputGrads gi, int V, int rc, int DP, int LDX, const float *__restrict__ X,
                      const float *__restrict__ XIN, const float *__restrict__ mu, const float *__restrict__ rstd,
                      const float *__restrict__ m1, const float *__restrict__ m2, const float *__restrict__ DXH,
                      const float *__restrict__ DX, const float *__restrict__ DGA) {
    __shared__ ColDesc s_col[DEC_MAX_DP];
    build_col_table(s_col, DP, rc, p.E, gi.plane, gi.att, p.packed);        // bases of the plane GRADIENTS (may be null)
    const int ts = p.packed ? 8 : 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps_total = gridDim.x * GATHER_WARPS;
    const int ncols = DP + GD;
    for (int v = blockIdx.x * GATHER_WARPS + warp; v < V; v += nwarps_total) {
        const int i = p.vis[v];
        const float ax = __ldg(p.anchor + 3 * (size_t)i), ay = __ldg(p.anchor + 3 * (size_t)i + 1), az = __ldg(p.anchor + 3 * (size_t)i + 2);
        float ind[3];
        norm_coords(p, ax, ay, az, ind);
        const float *xrow = X + (size_t)v * LDX, *dxh = DXH + (size_t)v * LDX;
        const float *dx100 = DX + (size_t)v * XI, *dga = DGA + (size_t)v * 40, *xin = XIN + (size_t)v * XI;
        // direction / distance gradient -> anchor (every lane computes all three components)
        float dv0, dv1, dv2;
        {
            const float d0 = xin[FD], d1 = xin[FD + 1], d2 = xin[FD + 2], dist = xin[FD + 3];
            const float g0 = dx100[FD], g1 = dx100[FD + 1], g2 = dx100[FD + 2], gd = dx100[FD + 3];
            const float dot = d0 * g0 + d1 * g1 + d2 * g2;
            dv0 = (g0 - d0 * dot) / dist + gd * d0;
            dv1 = (g1 - d1 * dot) / dist + gd * d1;
            dv2 = (g2 - d2 * dot) / dist + gd * d2;
        }
        // all row loads of the (at most 6) channel groups are issued before any of them is consumed: the
        // kernel is bound by L2 / HBM latency, not by instruction issue
        constexpr int MAXC = 6;
        float dxs[MAXC];
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane + 32 * j;
            dxs[j] = 0.f;
            if (c < ncols) {
                const float r = __ldg(rstd + c);
                const float xh = (__ldg(xrow + c) - __ldg(mu + c)) * r;
                dxs[j] = r * (__ldg(dxh + c) - __ldg(m1 + c) - xh * __ldg(m2 + c));
            }
        }
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane + 32 * j;
            if (c >= ncols) break;
            const float dx = dxs[j];
            if (c < DP) {
                const ColDesc cd = s_col[c];
                if (cd.base) {
                    float u, w;
                    plane_axes(cd.axis, ind, u, w);
                    bilin_scatter(const_cast<float *>(cd.base), bilin_setup(u, w, cd.E), dx, ts);
                }
            } else {
                const int g = c - DP;
                if (g < FD) atomicAdd(&gi.anchor_feat[(size_t)i * FD + g], dx + dx100[g]);
                else if (g < FD + 3) {
                    const int q = g - FD;
                    atomicAdd(&gi.anchor[3 * (size_t)i + q], dx + dga[q] + (q == 0 ? dv0 : (q == 1 ? dv1 : dv2)));
                }
                else if (g < FD + 3 + 3 * KO) atomicAdd(&gi.offset[(size_t)i * 3 * KO + (g - FD - 3)], dx + dga[3 + (g - FD - 3)]);
                else atomicAdd(&gi.scaling[(size_t)i * 6 + (g - FD - 3 - 3 * KO)], dx + dga[33 + (g - FD - 3 - 3 * KO)]);
            }
        }
    }
}

}  // namespace splatco
#include "decode2.cuh"

using namespace splatco;

namespace {

struct FwdView {
    float *X, *mu, *rstd, *WpT, *WcT, *bgeo, *W1T, *b1e, *W2T, *b2, *WpG, *WcG, *XIN, *H, *Z;
    double *stats;
    uint32_t *maskbits, *offs, *bsum, *boff, *total;
    float *XT;
    uint8_t *BA, *W1B, *W2B, *W2R, *W1R, *WPCR;
};
FwdView fwd_view(void *ws, const DecDims &d) {
    size_t off[F_NCHUNK + 1];
    dec_fwd_offsets(d, off);
    char *b = (char *)ws;
    FwdView v;
    v.X = (float *)(b + off[F_X]); v.stats = (double *)(b + off[F_STATS]);
    v.mu = (float *)(b + off[F_MU]); v.rstd = (float *)(b + off[F_RSTD]);
    v.WpT = (float *)(b + off[F_WPT]); v.WcT = (float *)(b + off[F_WCT]); v.bgeo = (float *)(b + off[F_BGEO]);
    v.W1T = (float *)(b + off[F_W1T]); v.b1e = (float *)(b + off[F_B1E]);
    v.W2T = (float *)(b + off[F_W2T]); v.b2 = (float *)(b + off[F_B2]);
    v.WpG = (float *)(b + off[F_WPG]); v.WcG = (float *)(b + off[F_WCG]);
    v.XIN = (float *)(b + off[F_XIN]); v.H = (float *)(b + off[F_H]); v.Z = (float *)(b + off[F_Z]);
    v.maskbits = (uint32_t *)(b + off[F_MASKBITS]); v.offs = (uint32_t *)(b + off[F_OFFS]);
    v.bsum = (uint32_t *)(b + off[F_BSUM]); v.boff = (uint32_t *)(b + off[F_BOFF]);
    v.total = (uint32_t *)(b + off[F_TOTAL]);
    v.XT = (float *)(b + off[F_XT]);
    v.BA = (uint8_t *)(b + off[F_BA]); v.W1B = (uint8_t *)(b + off[F_W1B]); v.W2B = (uint8_t *)(b + off[F_W2B]);
    v.W2R = (uint8_t *)(b + off[F_W2R]); v.W1R = (uint8_t *)(b + off[F_W1R]); v.WPCR = (uint8_t *)(b + off[F_WPCR]);
    return v;
}

struct BwdView {
    float *DZ, *DH, *DX, *DXH, *DGA, *gW2T, *gb2, *gW1T, *gb1, *S1, *S0, *m1, *m2;
    char *acc_begin; size_t acc_bytes;
};
BwdView bwd_view(void *ws, const DecDims &d) {
    size_t off[B_NCHUNK + 1];
    dec_bwd_offsets(d, off);
    char *b = (char *)ws;
    BwdView v;
    v.DZ = (float *)(b + off[B_DZ]); v.DH = (float *)(b + off[B_DH]); v.DX = (float *)(b + off[B_DX]);
    v.DXH = (float *)(b + off[B_DXH]); v.DGA = (float *)(b + off[B_DGA]);
    v.gW2T = (float *)(b + off[B_GW2T]); v.gb2 = (float *)(b + off[B_GB2]);
    v.gW1T = (float *)(b + off[B_GW1T]); v.gb1 = (float *)(b + off[B_GB1]);
    v.S1 = (float *)(b + off[B_S1]); v.S0 = (float *)(b + off[B_S0]);
    v.m1 = (float *)(b + off[B_M1]); v.m2 = (float *)(b + off[B_M2]);
    v.acc_begin = b + off[B_GW2T]; v.acc_bytes = off[B_M1] - off[B_GW2T];
    return v;
}

int check_desc(const splatco_decode_desc *d) {
    SPLATCO_REQUIRE(d, "decode: null descriptor");
    SPLATCO_REQUIRE(d->K == KO, "decode: n_offsets=%d unsupported (kernels are specialised for %d)", d->K, KO);
    SPLATCO_REQUIRE(d->level >= 0 && d->level <= 2, "decode: activate_level %d out of range", d->level);
    SPLATCO_REQUIRE(d->rc >= 1 && d->rc * 12 <= DEC_MAX_DP, "decode: channels per plane %d unsupported", d->rc);
    SPLATCO_REQUIRE(d->V >= 0 && d->N >= d->V, "decode: bad sizes N=%d V=%d", d->N, d->V);
    SPLATCO_REQUIRE(d->app_dim >= 0 && (d->app_dim == 0 || d->app_vec), "decode: appearance vector missing");
    SPLATCO_REQUIRE(d->plane_layout == 0 || (d->plane_layout == 1 && d->rc <= 8), "decode: bad plane_layout %d", d->plane_layout);
    if (d->V == 0) return 0;
    SPLATCO_REQUIRE(d->anchor_feat && d->anchor && d->offset && d->scaling && d->vis, "decode: null input");
    SPLATCO_REQUIRE(d->xyz_min && d->xyz_max && d->cam, "decode: null bbox / camera pointer");
    for (int l = 0; l <= d->level; ++l) {
        SPLATCO_REQUIRE(d->E[l] >= 2, "decode: plane edge %d too small", d->E[l]);
        for (int p = 0; p < 3; ++p) SPLATCO_REQUIRE(d->plane[3 * l + p], "decode: null plane (level %d)", l);
        SPLATCO_REQUIRE(d->bn_w[l] && d->bn_b[l] && d->lin_w[l] && d->lin_b[l] && d->cbn_w[l] && d->cbn_b[l] &&
                        d->clin_w[l] && d->clin_b[l], "decode: null BN/Linear parameter (level %d)", l);
    }
    for (int p = 0; p < 3; ++p) SPLATCO_REQUIRE(d->att[p], "decode: null attended plane");
    for (int h = 0; h < 3; ++h)
        SPLATCO_REQUIRE(d->w1[h] && d->b1[h] && d->w2[h] && d->b2[h], "decode: null head parameter");
    return 0;
}

DecPtrs make_ptrs(const splatco_decode_desc *d) {
    DecPtrs p;
    p.anchor_feat = d->anchor_feat; p.anchor = d->anchor; p.offset = d->offset; p.scaling = d->scaling;
    p.vis = d->vis;
    for (int l = 0; l < 3; ++l) {
        p.E[l] = d->E[l];
        for (int q = 0; q < 3; ++q) p.plane[l][q] = d->plane[3 * l + q];
    }
    for (int q = 0; q < 3; ++q) p.att[q] = d->att[q];
    p.mn = d->xyz_min; p.mx = d->xyz_max; p.cam = d->cam;
    p.noise = d->noise;
    p.noise_q = d->noise_q;
    p.noise_seed = d->noise_seed;
    p.packed = d->plane_layout;
    return p;
}

DecWeights make_weights(const splatco_decode_desc *d) {
    DecWeights w;
    for (int l = 0; l < 3; ++l) {
        w.bn_w[l] = d->bn_w[l]; w.bn_b[l] = d->bn_b[l]; w.lin_w[l] = d->lin_w[l]; w.lin_b[l] = d->lin_b[l];
        w.cbn_w[l] = d->cbn_w[l]; w.cbn_b[l] = d->cbn_b[l]; w.clin_w[l] = d->clin_w[l]; w.clin_b[l] = d->clin_b[l];
        w.bn_rm[l] = d->bn_rm[l]; w.bn_rv[l] = d->bn_rv[l]; w.cbn_rm[l] = d->cbn_rm[l]; w.cbn_rv[l] = d->cbn_rv[l];
        w.bn_nbt[l] = (long long *)d->bn_nbt[l]; w.cbn_nbt[l] = (long long *)d->cbn_nbt[l];
        w.w1[l] = d->w1[l]; w.b1[l] = d->b1[l]; w.w2[l] = d->w2[l]; w.b2[l] = d->b2[l];
        w.use_dist[l] = d->use_dist[l];
    }
    w.app_vec = d->app_vec; w.app_dim = d->app_dim; w.eps = d->bn_eps; w.momentum = d->bn_momentum;
    return w;
}

int gather_grid(int V) { return min(ceil_div(V, GATHER_WARPS), 148 * 8); }

}  // namespace

static size_t v1_decode_fwd_ws_bytes(int V, int rc, int level) {
    size_t off[F_NCHUNK + 1];
    return dec_fwd_offsets(dec_dims(V, rc, level), off);
}
static size_t v1_decode_bwd_ws_bytes(int V, int rc, int level) {
    size_t off[B_NCHUNK + 1];
    return dec_bwd_offsets(dec_dims(V, rc, level), off);
}

static const int32_t *v1_decode_count_ptr(const void *ws, int V, int rc, int level) {
    if (!ws) return nullptr;
    return reinterpret_cast<const int32_t *>(fwd_view(const_cast<void *>(ws), dec_dims(V, rc, level)).total);
}

static int v1_decode_fwd(const splatco_decode_desc *d, void *ws, float *neural_opacity, uint8_t *mask,
                                  int32_t *M_host, void *stream) {
    if (check_desc(d)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (d->V == 0) { if (M_host) *M_host = 0; return 0; }
    SPLATCO_REQUIRE(d->V >= 2, "decode: BatchNorm in train mode needs more than 1 visible anchor (got %d)", d->V);
    SPLATCO_REQUIRE(ws && neural_opacity && mask, "decode_fwd: null pointer");
    const DecDims dd = dec_dims(d->V, d->rc, d->level);
    const int V = d->V;
    FwdView f = fwd_view(ws, dd);
    const DecPtrs p = make_ptrs(d);
    const DecWeights w = make_weights(d);
    SPLATCO_CHECK_CUDA(cudaMemsetAsync(f.stats, 0, 2 * (size_t)dd.LDX * sizeof(double), st));
    const bool use_tc = dd.rc <= TC_MAX_RC;     // tensor-core path (3 rc <= 16 plane chunks fit its shared-memory map)
    dec_gather_kernel<<<gather_grid(V), GATHER_WARPS * 32, GATHER_WARPS * 2 * dd.LDX * sizeof(float), st>>>(
        p, V, dd.rc, dd.DP, dd.LDX, f.X, f.XIN, f.stats, use_tc ? f.XT : nullptr);
    SPLATCO_CHECK_LAUNCH();
    dec_fold_kernel<<<FOLD_CTAS, 256, 0, st>>>(w, V, nullptr, dd.rc, dd.level, dd.DP, dd.LDX, f.stats, f.mu, f.rstd, f.WpT, f.WcT,
                                       f.bgeo, f.W1T, f.b1e, f.W2T, f.b2, f.WpG, f.WcG, d->update_running);
    SPLATCO_CHECK_LAUNCH();
    const int nb = ceil_div(V, 256);
    SPLATCO_CHECK_CUDA(cudaMemsetAsync(f.bsum, 0, (size_t)nb * sizeof(uint32_t), st));
    if (use_tc) {
        // fused tcgen05 path: geo -> hidden -> heads -> activations in one persistent kernel
        dec_tc_pack_kernel<<<12, 256, 0, st>>>(dd.DP, f.WpT, f.WcT, f.W1T, f.W2T, f.BA, f.W1B, f.W2B);
        SPLATCO_CHECK_LAUNCH();
        dec_tc_pack_bwd_kernel<<<12, 256, 0, st>>>(dd.DP, f.W2T, f.W1T, f.WpG, f.WcG, f.W2R, f.W1R, f.WPCR);   // for the backward
        SPLATCO_CHECK_LAUNCH();
        static unsigned char attr_dev[64];       // cudaFuncSetAttribute is per device
    const int attr_i = current_device() & 63;
        if (!attr_dev[attr_i]) {
            SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(dec_tc_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM));
            attr_dev[attr_i] = 1;
        }
        const int ntiles = ceil_div(V, TC_ROWS);
        dec_tc_fwd_kernel<<<min(ntiles, 148), TC_THREADS, TC_SMEM, st>>>(V, dd.DP, f.XT, f.BA, f.W1B, f.W2B, f.bgeo, f.b1e, f.b2,
                                                                     f.XIN, f.H, f.Z, neural_opacity, mask, f.maskbits, f.bsum);
        SPLATCO_CHECK_LAUNCH();
    } else {
        // SIMT fp32 chain (plane grids with more than 5 channels per plane)
        // geo = [ (P - mu) Wp' | (g - mu) Wc' ] + bias, written straight into x100 columns 36..99
        if (sgemm<false, false>(st, V, 32, dd.DP, f.X, dd.LDX, f.WpT, 32, f.XIN + 36, XI, f.bgeo)) return -2;
        if (sgemm<false, false>(st, V, 32, GD, f.X + dd.DP, dd.LDX, f.WcT, 32, f.XIN + 68, XI, f.bgeo + 32)) return -2;
        if (sgemm<false, false>(st, V, HD, XI, f.XIN, XI, f.W1T, HD, f.H, HD, f.b1e, 1)) return -2;
        if (sgemm<false, false>(st, V, ZD, HD, f.H, HD, f.W2T, ZD, f.Z, ZD, f.b2)) return -2;
        dec_heads_act_kernel<<<ceil_div(V, ACT_ROWS), 256, 0, st>>>(V, f.Z, neural_opacity, mask, f.maskbits, f.bsum);
        SPLATCO_CHECK_LAUNCH();
    }
    scan_block_sums_kernel<<<1, 1024, 0, st>>>(nb, f.bsum, f.boff, f.total);
    SPLATCO_CHECK_LAUNCH();
    dec_offsets_kernel<<<nb, 256, 0, st>>>(V, nullptr, f.maskbits, f.boff, f.offs);
    SPLATCO_CHECK_LAUNCH();
    if (M_host) SPLATCO_CHECK_CUDA(cudaMemcpyAsync(M_host, f.total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return 0;
}

static int v1_decode_emit(const splatco_decode_desc *d, const void *ws, int M, float *xyz, float *color,
                                   float *opacity, float *scaling, float *rot, void *stream) {
    if (check_desc(d)) return -1;
    if (d->V == 0 || M == 0) return 0;
    SPLATCO_REQUIRE(ws && xyz && color && opacity && scaling && rot, "decode_emit: null pointer");
    const DecDims dd = dec_dims(d->V, d->rc, d->level);
    FwdView f = fwd_view(const_cast<void *>(ws), dd);
    dec_compact_kernel<<<ceil_div(d->V * KO, 256), 256, 0, (cudaStream_t)stream>>>(
        d->V, dd.LDX, dd.DP, f.X, f.Z, f.maskbits, f.offs, xyz, color, opacity, scaling, rot);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

static int v1_decode_bwd(const splatco_decode_desc *d, const void *fwd_ws, void *bwd_ws, int M,
                                  const float *d_xyz, const float *d_color, const float *d_opacity,
                                  const float *d_scaling, const float *d_rot, const float *d_neural_opacity,
                                  const splatco_decode_grads *g, void *stream) {
    if (check_desc(d)) return -1;
    if (d->V == 0) return 0;
    SPLATCO_REQUIRE(fwd_ws && bwd_ws && g, "decode_bwd: null pointer");
    SPLATCO_REQUIRE(M == 0 || (d_xyz && d_color && d_opacity && d_scaling && d_rot), "decode_bwd: null upstream gradient");
    SPLATCO_REQUIRE(g->anchor_feat && g->anchor && g->offset && g->scaling, "decode_bwd: null per-anchor gradient");
    cudaStream_t st = (cudaStream_t)stream;
    const DecDims dd = dec_dims(d->V, d->rc, d->level);
    const int V = d->V, DP = dd.DP, LDX = dd.LDX;
    FwdView f = fwd_view(const_cast<void *>(fwd_ws), dd);
    BwdView b = bwd_view(bwd_ws, dd);
    const DecPtrs p = make_ptrs(d);
    const DecWeights w = make_weights(d);
    DecWeightGrads gw;
    DecInputGrads gi;
    for (int l = 0; l < 3; ++l) {
        gw.bn_w[l] = g->bn_w[l]; gw.bn_b[l] = g->bn_b[l]; gw.lin_w[l] = g->lin_w[l]; gw.lin_b[l] = g->lin_b[l];
        gw.cbn_w[l] = g->cbn_w[l]; gw.cbn_b[l] = g->cbn_b[l]; gw.clin_w[l] = g->clin_w[l]; gw.clin_b[l] = g->clin_b[l];
        gw.w1[l] = g->w1[l]; gw.b1[l] = g->b1[l]; gw.w2[l] = g->w2[l]; gw.b2[l] = g->b2[l];
        for (int q = 0; q < 3; ++q) gi.plane[l][q] = g->plane[3 * l + q];
        gi.att[l] = g->att[l];
    }
    gw.app_vec = g->app_vec;
    gi.anchor_feat = g->anchor_feat; gi.anchor = g->anchor; gi.offset = g->offset; gi.scaling = g->scaling;
    const int KCH = 512;            // split-K chunk: V/512 slices x (M/64 x N/32) tiles keep all 148 SMs busy

    SPLATCO_CHECK_CUDA(cudaMemsetAsync(b.acc_begin, 0, b.acc_bytes, st));
    dec_bwd_uncompact_kernel<<<ceil_div(V, UNC_ROWS), UNC_ROWS * KO, 0, st>>>(V, LDX, DP, f.X, f.Z, f.maskbits, f.offs, d_xyz, d_color,
                                                              d_opacity, d_scaling, d_rot, d_neural_opacity, b.DZ, b.DGA);
    SPLATCO_CHECK_LAUNCH();
    const bool use_tc = dd.rc <= TC_MAX_RC;
    if (use_tc) {
        // row chain on tensor cores: dH = (dZ W2).[H>0], dX = dH W1, dxhat = dgeo (gamma W); gb2, gb1, S0 in its epilogues
        static unsigned char attr_dev[64];       // cudaFuncSetAttribute is per device
    const int attr_i = current_device() & 63;
        if (!attr_dev[attr_i]) {
            SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(dec_tc_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TCB_SMEM));
            attr_dev[attr_i] = 1;
        }
        dec_tc_bwd_kernel<<<min(ceil_div(V, TC_ROWS), 148), TC_THREADS, TCB_SMEM, st>>>(V, DP, LDX, b.DZ, f.H, f.W2R, f.W1R, f.WPCR,
                                                                                    b.DH, b.DX, b.DXH, b.gb2, b.gb1, b.S0);
        SPLATCO_CHECK_LAUNCH();
    } else {
        // SIMT chain.  W2 is block-diagonal: three narrow GEMMs instead of one dense 96 x 112.
        for (int hd = 0; hd < 3; ++hd) {
            const int j0 = hd == 0 ? 0 : (hd == 1 ? KO : 8 * KO), nj = hd == 0 ? KO : (hd == 1 ? 7 * KO : 3 * KO), i0 = 32 * hd;
            if (sgemm<false, true>(st, V, 32, nj, b.DZ + j0, ZD, f.W2T + (size_t)i0 * ZD + j0, ZD, b.DH + i0, HD, nullptr, 0,
                                   f.H + i0, HD)) return -2;
        }
        if (sgemm<false, true>(st, V, XI, HD, b.DH, HD, f.W1T, HD, b.DX, XI)) return -2;
        if (sgemm<false, false>(st, V, DP, 32, b.DX + 36, XI, f.WpG, DP, b.DXH, LDX)) return -2;
        if (sgemm<false, false>(st, V, GD, 32, b.DX + 68, XI, f.WcG, GD, b.DXH + DP, LDX)) return -2;
        colsum_kernel<<<dim3(ceil_div(V, 128), 1), 128, 0, st>>>(V, ZD, b.DZ, ZD, b.gb2, 128);
        SPLATCO_CHECK_LAUNCH();
        colsum_kernel<<<dim3(ceil_div(V, 128), 1), 128, 0, st>>>(V, HD, b.DH, HD, b.gb1, 128);
        SPLATCO_CHECK_LAUNCH();
        colsum_kernel<<<dim3(ceil_div(V, 128), 1), 128, 0, st>>>(V, 64, b.DX + 36, XI, b.S0, 128);
        SPLATCO_CHECK_LAUNCH();
    }
    // weight gradients: gW2T += H^T dZ (block-diagonal), gW1T += X100^T dH, S1raw = dgeo^T X (both branches)
    {
        WgGroup grp;
        grp.count = 0;
        auto add = [&](int M, int N, const float *A, int lda, const float *B, int ldb, float *C, int ldc) {
            WgProblem &q = grp.p[grp.count++];
            q.A = A; q.B = B; q.C = C; q.M = M; q.N = N; q.lda = lda; q.ldb = ldb; q.ldc = ldc;
            q.shape = M > 32 ? 4 : (N <= 16 ? 0 : (N <= 32 ? 1 : (N <= 64 ? 2 : 3)));
        };
        for (int hd = 0; hd < 3; ++hd) {
            const int j0 = hd == 0 ? 0 : (hd == 1 ? KO : 8 * KO), nj = hd == 0 ? KO : (hd == 1 ? 7 * KO : 3 * KO), i0 = 32 * hd;
            add(32, nj, f.H + i0, HD, b.DZ + j0, ZD, b.gW2T + (size_t)i0 * ZD + j0, ZD);
        }
        add(XI, HD, f.XIN, XI, b.DH, HD, b.gW1T, HD);
        add(32, DP, b.DX + 36, XI, f.X, LDX, b.S1, LDX);
        add(32, GD, b.DX + 68, XI, f.X + DP, LDX, b.S1 + DP, LDX);
        // deal ~2 CTAs per SM to the problems in proportion to their (padded) FMA counts
        static const int kWork[5] = {2 * 1, 2 * 2, 2 * 4, 2 * 5, 8 * 6};
        int total = 0;
        for (int i = 0; i < grp.count; ++i) total += kWork[grp.p[i].shape];
        // (narrow outputs run far below the FMA rate, so no CTA gets more than 768 rows whatever its share)
        const int budget = 2 * 148, max_slices = max(1, ceil_div(V, 2 * WG_KB)), min_slices = ceil_div(V, 768);
        int ctas = 0;
        for (int i = 0; i < grp.count; ++i) {
            WgProblem &q = grp.p[i];
            q.nslices = min(max_slices, max(min_slices, budget * kWork[q.shape] / total));
            q.cta0 = ctas;
            ctas += q.nslices;
        }
        dec_wgrad_kernel<<<ctas, 256, 0, st>>>(grp, V);
        SPLATCO_CHECK_LAUNCH();
    }
    dec_bwd_fold_kernel<<<dim3(BWD_FOLD_CTAS, BWD_FOLD_SECTIONS), 256, 0, st>>>(w, gw, V, dd.rc, dd.level, DP, LDX, f.mu, f.rstd, f.WpG, f.WcG, b.S1, b.S0,
                                           b.gW1T, b.gb1, b.gW2T, b.gb2, b.m1, b.m2);
    SPLATCO_CHECK_LAUNCH();
    dec_bwd_inputs_kernel<<<gather_grid(V), GATHER_WARPS * 32, 0, st>>>(p, gi, V, dd.rc, DP, LDX, f.X, f.XIN, f.mu, f.rstd,
                                                                        b.m1, b.m2, b.DXH, b.DX, b.DGA);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

// ---- channel-last copies of the feature planes --------------------------------------------------------------
// [rc,E,E] (the reference's nn.Parameter layout, scene/grids.py:122-125) <-> [E,E,8]: one 32-byte sector per texel.
// Built once per iteration by the host (decode.py caches it across the mv views), like TriPlaneAttention.
namespace splatco {
__global__ void __launch_bounds__(256)
pack_planes_kernel(int rc, int npix, const float *__restrict__ a, const float *__restrict__ b, const float *__restrict__ c,
                   float *__restrict__ pa, float *__restrict__ pb, float *__restrict__ pc) {
    const float *src = blockIdx.y == 0 ? a : (blockIdx.y == 1 ? b : c);
    float *dst = blockIdx.y == 0 ? pa : (blockIdx.y == 1 ? pb : pc);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < npix; i += gridDim.x * 256) {
        float v[8];
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) v[ch] = ch < rc ? __ldg(src + (size_t)ch * npix + i) : 0.f;
        float4 *o = reinterpret_cast<float4 *>(dst + (size_t)i * 8);
        o[0] = make_float4(v[0], v[1], v[2], v[3]);
        o[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
}
__global__ void __launch_bounds__(256)
unpack_planes_add_kernel(int rc, int npix, const float *__restrict__ pa, const float *__restrict__ pb,
                         const float *__restrict__ pc, float *__restrict__ a, float *__restrict__ b, float *__restrict__ c) {
    const float *src = blockIdx.y == 0 ? pa : (blockIdx.y == 1 ? pb : pc);
    float *dst = blockIdx.y == 0 ? a : (blockIdx.y == 1 ? b : c);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < npix; i += gridDim.x * 256) {
        const float4 *in = reinterpret_cast<const float4 *>(src + (size_t)i * 8);
        const float4 lo = __ldg(in), hi = __ldg(in + 1);
        const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
        for (int ch = 0; ch < 8; ++ch)
            if (ch < rc && v[ch] != 0.f) dst[(size_t)ch * npix + i] += v[ch];
    }
}
}  // namespace splatco

extern "C" int splatco_pack_planes(int rc, int E, const float *xy, const float *xz, const float *yz, float *pxy,
                                   float *pxz, float *pyz, void *stream) {
    SPLATCO_REQUIRE(rc >= 1 && rc <= 8 && E >= 1 && (int64_t)E * E < 0x7fffffff, "pack_planes: bad sizes rc=%d E=%d", rc, E);
    SPLATCO_REQUIRE(xy && xz && yz && pxy && pxz && pyz, "pack_planes: null pointer");
    SPLATCO_REQUIRE((((uintptr_t)pxy | (uintptr_t)pxz | (uintptr_t)pyz) & 31) == 0, "pack_planes: outputs need 32-byte alignment");
    const int npix = E * E;
    pack_planes_kernel<<<dim3(min(148 * 8, ceil_div(npix, 256)), 3), 256, 0, (cudaStream_t)stream>>>(rc, npix, xy, xz, yz, pxy, pxz, pyz);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

extern "C" int splatco_unpack_planes_add(int rc, int E, const float *gpxy, const float *gpxz, const float *gpyz,
                                         float *gxy, float *gxz, float *gyz, void *stream) {
    SPLATCO_REQUIRE(rc >= 1 && rc <= 8 && E >= 1 && (int64_t)E * E < 0x7fffffff, "unpack_planes_add: bad sizes rc=%d E=%d", rc, E);
    SPLATCO_REQUIRE(gpxy && gpxz && gpyz && gxy && gxz && gyz, "unpack_planes_add: null pointer");
    const int npix = E * E;
    unpack_planes_add_kernel<<<dim3(min(148 * 8, ceil_div(npix, 256)), 3), 256, 0, (cudaStream_t)stream>>>(rc, npix, gpxy, gpxz, gpyz,
                                                                                                          gxy, gxz, gyz);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

// =====================================================================================================================
// v2 host side (decode2.cuh) and the dispatch between the two implementations.
//   v2: plane grids with at most 5 channels per plane (num_channels <= 15, the reference's configurations)
//   v1: everything else, or when forced with splatco_decode_set_impl(1) / SPLATCO_DECODE_IMPL=1 (A/B timing, debugging)
// =====================================================================================================================
namespace {

int g_decode_impl = 0;      // 0: not read yet, 1: v1, 2: v2
int g_decode_profile = 0;
cudaEvent_t g_prof_ev[64][4];          // per device: fwd begin / end, bwd begin / end
unsigned char g_prof_have[64];
void prof_record(int which, cudaStream_t st) {
    if (g_decode_profile != 1) return;
    const int d = current_device() & 63;
    if (!g_prof_have[d]) {
        for (int i = 0; i < 4; ++i) cudaEventCreate(&g_prof_ev[d][i]);
        g_prof_have[d] = 1;
    }
    cudaEventRecord(g_prof_ev[d][which], st);
}
int decode_impl() {
    if (!g_decode_impl) {
        const char *e = getenv("SPLATCO_DECODE_IMPL");
        g_decode_impl = (e && e[0] == '1') ? 1 : 2;
    }
    return g_decode_impl;
}
bool use_v2(int rc) { return decode_impl() == 2 && rc >= 1 && rc <= 5; }

enum F2Chunk { G_STATS, G_MU, G_RSTD, G_WPT, G_WCT, G_BGEO, G_W1T, G_B1E, G_W2T, G_B2, G_WPG, G_WCG, G_XT, G_HT, G_ZT,
               G_MASKBITS, G_OFFS, G_BSUM, G_BOFF, G_TOTAL, G_W1S, G_W1R, G_W2B, G_B2BLK, G_W2R, G_NCHUNK };

size_t d2_fwd_offsets(const D2Dims &d, size_t off[G_NCHUNK + 1]) {
    const size_t V = (size_t)(d.V > 0 ? d.V : 0);
    const size_t nb = (V + 255) / 256, nt = (size_t)d.ntiles;
    size_t o = 0;
    auto put = [&](int c, size_t bytes) { off[c] = o; o += align_up(bytes); };
    put(G_STATS, 2 * (size_t)d.LDX * 8);
    put(G_MU, d.LDX * 4); put(G_RSTD, d.LDX * 4);
    put(G_WPT, DEC_MAX_DP * 32 * 4); put(G_WCT, GD * 32 * 4); put(G_BGEO, 64 * 4);
    put(G_W1T, XI * HD * 4); put(G_B1E, HD * 4);
    put(G_W2T, HD * ZD * 4); put(G_B2, ZD * 4);
    put(G_WPG, 32 * DEC_MAX_DP * 4); put(G_WCG, 32 * GD * 4);
    put(G_XT, nt * d.nch * D2_CHUNK); put(G_HT, nt * 24 * D2_CHUNK); put(G_ZT, nt * D2_ZCH * D2_CHUNK);
    put(G_MASKBITS, V * 4); put(G_OFFS, V * 4); put(G_BSUM, nb * 4); put(G_BOFF, nb * 4); put(G_TOTAL, 4);
    put(G_W1S, 3 * (size_t)d.nk * 32 * 16 * 2); put(G_W1R, 2 * 24 * (size_t)d.NB * 16);
    put(G_W2B, 2 * D2_W2B_HALF); put(G_B2BLK, 128 * 4); put(G_W2R, 2 * D2_W2R_HALF);
    off[G_NCHUNK] = o;
    return o;
}

struct F2View {
    double *stats;
    float *mu, *rstd, *WpT, *WcT, *bgeo, *W1T, *b1e, *W2T, *b2, *WpG, *WcG, *b2blk;
    float4 *XT, *HT, *ZT;
    uint32_t *maskbits, *offs, *bsum, *boff, *total;
    uint8_t *W1S, *W1R, *W2B, *W2R;
};
F2View f2_view(void *ws, const D2Dims &d) {
    size_t off[G_NCHUNK + 1];
    d2_fwd_offsets(d, off);
    char *b = (char *)ws;
    F2View v;
    v.stats = (double *)(b + off[G_STATS]);
    v.mu = (float *)(b + off[G_MU]); v.rstd = (float *)(b + off[G_RSTD]);
    v.WpT = (float *)(b + off[G_WPT]); v.WcT = (float *)(b + off[G_WCT]); v.bgeo = (float *)(b + off[G_BGEO]);
    v.W1T = (float *)(b + off[G_W1T]); v.b1e = (float *)(b + off[G_B1E]);
    v.W2T = (float *)(b + off[G_W2T]); v.b2 = (float *)(b + off[G_B2]);
    v.WpG = (float *)(b + off[G_WPG]); v.WcG = (float *)(b + off[G_WCG]);
    v.XT = (float4 *)(b + off[G_XT]); v.HT = (float4 *)(b + off[G_HT]); v.ZT = (float4 *)(b + off[G_ZT]);
    v.maskbits = (uint32_t *)(b + off[G_MASKBITS]); v.offs = (uint32_t *)(b + off[G_OFFS]);
    v.bsum = (uint32_t *)(b + off[G_BSUM]); v.boff = (uint32_t *)(b + off[G_BOFF]); v.total = (uint32_t *)(b + off[G_TOTAL]);
    v.W1S = (uint8_t *)(b + off[G_W1S]); v.W1R = (uint8_t *)(b + off[G_W1R]);
    v.W2B = (uint8_t *)(b + off[G_W2B]); v.b2blk = (float *)(b + off[G_B2BLK]); v.W2R = (uint8_t *)(b + off[G_W2R]);
    return v;
}

enum B2Chunk { H_DUT, H_DGA, H_PART, H_RED, H_GW2T, H_GB2, H_GW1T, H_GB1, H_S1, H_S0, H_M1, H_M2, H_NCHUNK };
constexpr int D2_MAX_CTAS = 148;

size_t d2_bwd_offsets(const D2Dims &d, size_t off[H_NCHUNK + 1]) {
    size_t o = 0;
    auto put = [&](int c, size_t bytes) { off[c] = o; o += align_up(bytes); };
    put(H_DUT, (size_t)d.ntiles * d.nch * D2_CHUNK); put(H_DGA, (size_t)d.ntiles * 10 * D2_CHUNK);
    put(H_PART, (size_t)D2_MAX_CTAS * D2_PART * 4); put(H_RED, (size_t)D2_PART * 4);
    put(H_GW2T, HD * ZD * 4); put(H_GB2, ZD * 4); put(H_GW1T, XI * HD * 4); put(H_GB1, HD * 4);
    put(H_S1, 32 * (size_t)d.LDX * 4); put(H_S0, 64 * 4); put(H_M1, d.LDX * 4); put(H_M2, d.LDX * 4);
    off[H_NCHUNK] = o;
    return o;
}
struct B2View { float4 *DUT, *DGA; float *part, *red, *gW2T, *gb2, *gW1T, *gb1, *S1, *S0, *m1, *m2; };
B2View b2_view(void *ws, const D2Dims &d) {
    size_t off[H_NCHUNK + 1];
    d2_bwd_offsets(d, off);
    char *b = (char *)ws;
    B2View v;
    v.DUT = (float4 *)(b + off[H_DUT]); v.DGA = (float4 *)(b + off[H_DGA]); v.part = (float *)(b + off[H_PART]);
    v.red = (float *)(b + off[H_RED]);
    v.gW2T = (float *)(b + off[H_GW2T]); v.gb2 = (float *)(b + off[H_GB2]); v.gW1T = (float *)(b + off[H_GW1T]);
    v.gb1 = (float *)(b + off[H_GB1]); v.S1 = (float *)(b + off[H_S1]); v.S0 = (float *)(b + off[H_S0]);
    v.m1 = (float *)(b + off[H_M1]); v.m2 = (float *)(b + off[H_M2]);
    return v;
}

template <int LEVEL, int RC>
int launch_gather2(bool packed, cudaStream_t st, const DecPtrs &p, const D2Dims &d, int V, const int32_t *Vdev, float4 *XT, double *stats) {
    const int grid = Vdev ? d.ntiles : ceil_div(V, D2_ROWS);
    if (packed) dec2_gather_kernel<LEVEL, RC, true><<<grid, D2_ROWS, 0, st>>>(p, V, Vdev, d.LDX, XT, stats);
    else dec2_gather_kernel<LEVEL, RC, false><<<grid, D2_ROWS, 0, st>>>(p, V, Vdev, d.LDX, XT, stats);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}
template <int LEVEL, int RC>
int launch_inputs2(bool packed, cudaStream_t st, const DecPtrs &p, const DecInputGrads &gi, const D2Dims &d, int V, const float4 *XT,
                   const float4 *DUT, const float *mu, const float *rstd, const float *m1, const float *m2) {
    const int grid = ceil_div(V, D2_ROWS);
    if (packed) dec2_bwd_inputs_kernel<LEVEL, RC, true><<<grid, D2_ROWS, 0, st>>>(p, gi, V, XT, DUT, mu, rstd, m1, m2);
    else dec2_bwd_inputs_kernel<LEVEL, RC, false><<<grid, D2_ROWS, 0, st>>>(p, gi, V, XT, DUT, mu, rstd, m1, m2);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}
#define D2_DISPATCH(FN, level, rc, ...)                                                                      \
    [&]() -> int {                                                                                           \
        switch ((level) * 8 + (rc)) {                                                                        \
            case 1: return FN<0, 1>(__VA_ARGS__); case 2: return FN<0, 2>(__VA_ARGS__);                      \
            case 3: return FN<0, 3>(__VA_ARGS__); case 4: return FN<0, 4>(__VA_ARGS__);                      \
            case 5: return FN<0, 5>(__VA_ARGS__);                                                            \
            case 9: return FN<1, 1>(__VA_ARGS__); case 10: return FN<1, 2>(__VA_ARGS__);                     \
            case 11: return FN<1, 3>(__VA_ARGS__); case 12: return FN<1, 4>(__VA_ARGS__);                    \
            case 13: return FN<1, 5>(__VA_ARGS__);                                                           \
            case 17: return FN<2, 1>(__VA_ARGS__); case 18: return FN<2, 2>(__VA_ARGS__);                    \
            case 19: return FN<2, 3>(__VA_ARGS__); case 20: return FN<2, 4>(__VA_ARGS__);                    \
            case 21: return FN<2, 5>(__VA_ARGS__);                                                           \
        }                                                                                                    \
        splatco::set_error("decode v2: unsupported level %d / channels per plane %d", (level), (rc));        \
        return -1;                                                                                           \
    }()

// rows the workspaces are laid out for (splatco_decode_desc::V_layout; 0 = V)
inline int d2_layout_rows(const splatco_decode_desc *d) { return d->V_layout > 0 ? d->V_layout : d->V; }

int v2_decode_fwd(const splatco_decode_desc *d, void *ws, float *neural_opacity, uint8_t *mask, int32_t *M_host, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (d->V == 0) { if (M_host) *M_host = 0; return 0; }
    const int32_t *Vdev = d->V_dev;
    // with the count still on the device the BatchNorm precondition (V >= 2) is the caller's to check once it knows V
    SPLATCO_REQUIRE(Vdev || d->V >= 2, "decode: BatchNorm in train mode needs more than 1 visible anchor (got %d)", d->V);
    SPLATCO_REQUIRE(d->V <= d2_layout_rows(d), "decode_fwd: V = %d exceeds V_layout = %d", d->V, d->V_layout);
    SPLATCO_REQUIRE(!Vdev || !d->noise, "decode_fwd: an explicit noise tensor needs the exact V on the host");
    SPLATCO_REQUIRE(ws && neural_opacity && mask, "decode_fwd: null pointer");
    const D2Dims dd = d2_dims(d2_layout_rows(d), d->rc, d->level);     // layout (and, with V_dev, grid) dimensions
    const int V = d->V;                                                  // exact, or the capacity when V_dev is set
    F2View f = f2_view(ws, dd);
    const DecPtrs p = make_ptrs(d);
    const DecWeights w = make_weights(d);
    SPLATCO_CHECK_CUDA(cudaMemsetAsync(f.stats, 0, 2 * (size_t)dd.LDX * sizeof(double), st));
    if (D2_DISPATCH(launch_gather2, dd.level, dd.rc, d->plane_layout != 0, st, p, dd, V, Vdev, f.XT, f.stats)) return -2;
    dec_fold_kernel<<<FOLD_CTAS, 256, 0, st>>>(w, V, Vdev, dd.rc, dd.level, dd.DP, dd.LDX, f.stats, f.mu, f.rstd, f.WpT, f.WcT,
                                              f.bgeo, f.W1T, f.b1e, f.W2T, f.b2, f.WpG, f.WcG, d->update_running);
    SPLATCO_CHECK_LAUNCH();
    dec2_combine_kernel<<<24, 256, 0, st>>>(dd.DP, dd.nk, dd.NB, f.WpT, f.WcT, f.bgeo, f.W1T, f.b1e, f.W2T, f.b2, f.W1S, f.W1R,
                                            f.W2B, f.b2blk, f.W2R);
    SPLATCO_CHECK_LAUNCH();
    const int nb = ceil_div(V, 256);
    SPLATCO_CHECK_CUDA(cudaMemsetAsync(f.bsum, 0, (size_t)nb * sizeof(uint32_t), st));
    static unsigned char attr_dev[64];
    const int attr_i = current_device() & 63;
    if (!attr_dev[attr_i]) {
        SPLATCO_CHECK_CUDA(cudaFuncSetAttribute(dec2_mlp_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)D2F_SMEM));
        attr_dev[attr_i] = 1;
    }
    D2Fwd a;
    a.V = V; a.Vdev = Vdev; a.nch = dd.nch; a.nk = dd.nk; a.trace = g_decode_profile == 2;
    a.XT = f.XT; a.W1S = f.W1S; a.W2B = f.W2B; a.b2blk = f.b2blk; a.HT = f.HT; a.ZT = f.ZT;
    a.nopac = neural_opacity; a.mask_out = mask; a.maskbits = f.maskbits; a.block_sums = f.bsum;
    prof_record(0, st);
    dec2_mlp_fwd_kernel<<<min(ceil_div(V, D2_ROWS), D2_MAX_CTAS), D2_THREADS, D2F_SMEM, st>>>(a);
    SPLATCO_CHECK_LAUNCH();
    prof_record(1, st);
    scan_block_sums_kernel<<<1, 1024, 0, st>>>(nb, f.bsum, f.boff, f.total);
    SPLATCO_CHECK_LAUNCH();
    dec_offsets_kernel<<<nb, 256, 0, st>>>(V, Vdev, f.maskbits, f.boff, f.offs);
    SPLATCO_CHECK_LAUNCH();
    if (M_host) SPLATCO_CHECK_CUDA(cudaMemcpyAsync(M_host, f.total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return 0;
}

int v2_decode_emit(const splatco_decode_desc *d, const void *ws, int M, float *xyz, float *color, float *opacity,
                   float *scaling, float *rot, void *stream) {
    if (d->V == 0 || M == 0) return 0;
    SPLATCO_REQUIRE(ws && xyz && color && opacity && scaling && rot, "decode_emit: null pointer");
    const D2Dims dd = d2_dims(d2_layout_rows(d), d->rc, d->level);
    F2View f = f2_view(const_cast<void *>(ws), dd);
    dec2_compact_kernel<<<ceil_div(d->V * KO, 256), 256, 0, (cudaStream_t)stream>>>(d->V, d->V_dev, dd.nch, f.XT, f.ZT, f.maskbits, f.offs,
                                                                                 xyz, color, opacity, scaling, rot);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}

}  // namespace

#include "decode2_bwd.cuh"
#include "camgrad.cuh"

namespace splatco {
__global__ void __launch_bounds__(256)
dec2_untile_kernel(int V, int nch, int DP, int LDX, const float4 *__restrict__ XT, float *__restrict__ out) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= V * LDX) return;
    const int v = t / LDX, c = t - v * LDX;
    float val = 0.f;
    if (c < DP + GD) {
        const int uc = c < DP ? D2_UP0 + c : c - DP;
        val = reinterpret_cast<const float *>(XT + ((size_t)(v >> 7) * nch) * D2_ROWS + (v & 127))[d2_tile_idx(uc)];
    }
    out[t] = val;
}

// dL/dcamera_center = -sum over the visible anchors of the direction / distance gradient the input kernels add to
// dL/danchor (dec_bwd_inputs_kernel, dec2_bwd_inputs_kernel; same formula, same operands): one thread per anchor reads
// (dir, dist) and its upstream gradient as two 16-byte cells and leaves one partial per CTA (camgrad.cuh).
//   nch > 0: v2 tile layout (XT / DUT, chunk D2_DIR_CH of a tile of nch chunks);  nch == 0: v1 rows (XIN / DX, columns FD..FD+3)
__global__ void __launch_bounds__(CAM_ROWS)
dec_camera_grad_kernel(int V, int nch, const float4 *__restrict__ X, const float4 *__restrict__ G, float *__restrict__ part) {
    const int v = blockIdx.x * CAM_ROWS + threadIdx.x;
    float cg[CAM_COLS];
#pragma unroll
    for (int c = 0; c < CAM_COLS; ++c) cg[c] = 0.f;
    if (v < V) {
        const size_t cell = nch > 0 ? ((size_t)(v >> 7) * nch + D2_DIR_CH) * D2_ROWS + (v & 127) : ((size_t)v * XI + FD) / 4;
        const float4 dd = __ldg(X + cell), gd = __ldg(G + cell);
        const float dot = dd.x * gd.x + dd.y * gd.y + dd.z * gd.z;
        cg[0] = (gd.x - dd.x * dot) / dd.w + gd.w * dd.x;
        cg[1] = (gd.y - dd.y * dot) / dd.w + gd.w * dd.y;
        cg[2] = (gd.z - dd.z * dot) / dd.w + gd.w * dd.z;
    }
    camera_block_partial(cg, part);
}
}  // namespace splatco

extern "C" int splatco_decode_gathered_rows(const void *ws, int V, int rc, int level, float *out, void *stream) {
    SPLATCO_REQUIRE(ws && out && V > 0 && rc >= 1 && level >= 0 && level <= 2, "decode_gathered_rows: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (use_v2(rc)) {
        const D2Dims dd = d2_dims(V, rc, level);
        dec2_untile_kernel<<<ceil_div(V * dd.LDX, 256), 256, 0, st>>>(V, dd.nch, dd.DP, dd.LDX, f2_view(const_cast<void *>(ws), dd).XT, out);
        SPLATCO_CHECK_LAUNCH();
    } else {
        const DecDims dd = dec_dims(V, rc, level);
        SPLATCO_CHECK_CUDA(cudaMemcpyAsync(out, fwd_view(const_cast<void *>(ws), dd).X, (size_t)V * dd.LDX * sizeof(float),
                                           cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

extern "C" int splatco_decode_set_impl(int impl) {
    SPLATCO_REQUIRE(impl == 1 || impl == 2, "decode_set_impl: 1 (three-stage chain) or 2 (collapsed two-stage pipeline)");
    g_decode_impl = impl;
    return 0;
}
extern "C" int splatco_decode_get_impl(void) { return decode_impl(); }
extern "C" int splatco_decode_profile(int enable) { g_decode_profile = enable; return 0; }
extern "C" int splatco_decode_trace_read(unsigned long long *out128) {
    SPLATCO_REQUIRE(out128, "decode_trace_read: null pointer");
    SPLATCO_CHECK_CUDA(cudaMemcpyFromSymbol(out128, g_d2_trace, sizeof(unsigned long long) * 128));
    return 0;
}
extern "C" int splatco_decode_profile_read(float *fwd_mlp_ms, float *bwd_mlp_ms) {
    const int d = current_device() & 63;
    SPLATCO_REQUIRE(g_prof_have[d], "decode_profile_read: nothing recorded on this device");
    if (fwd_mlp_ms) SPLATCO_CHECK_CUDA(cudaEventElapsedTime(fwd_mlp_ms, g_prof_ev[d][0], g_prof_ev[d][1]));
    if (bwd_mlp_ms) SPLATCO_CHECK_CUDA(cudaEventElapsedTime(bwd_mlp_ms, g_prof_ev[d][2], g_prof_ev[d][3]));
    return 0;
}

// workspaces are sized for whichever implementation is larger, so the choice may change between calls
extern "C" size_t splatco_decode_fwd_ws_bytes(int V, int rc, int level) {
    size_t off[G_NCHUNK + 1];
    const size_t a = v1_decode_fwd_ws_bytes(V, rc, level);
    const size_t b = (rc >= 1 && rc <= 5 && level >= 0 && level <= 2) ? d2_fwd_offsets(d2_dims(V, rc, level), off) : 0;
    return a > b ? a : b;
}
extern "C" size_t splatco_decode_bwd_ws_bytes(int V, int rc, int level) {
    size_t off[H_NCHUNK + 1];
    const size_t a = v1_decode_bwd_ws_bytes(V, rc, level);
    const size_t b = (rc >= 1 && rc <= 5 && level >= 0 && level <= 2) ? d2_bwd_offsets(d2_dims(V, rc, level), off) : 0;
    return a > b ? a : b;
}
extern "C" const int32_t *splatco_decode_count_ptr(const void *ws, int V, int rc, int level) {
    if (!ws) return nullptr;
    if (use_v2(rc)) return reinterpret_cast<const int32_t *>(f2_view(const_cast<void *>(ws), d2_dims(V, rc, level)).total);
    return v1_decode_count_ptr(ws, V, rc, level);
}
extern "C" int splatco_decode_fwd(const splatco_decode_desc *d, void *ws, float *neural_opacity, uint8_t *mask,
                                  int32_t *M_host, void *stream) {
    if (check_desc(d)) return -1;
    SPLATCO_REQUIRE(use_v2(d->rc) || (!d->V_dev && (d->V_layout == 0 || d->V_layout == d->V)),
                    "decode_fwd: V_dev / V_layout need the two-stage implementation (rc <= 5, SPLATCO_DECODE_IMPL != 1)");
    return use_v2(d->rc) ? v2_decode_fwd(d, ws, neural_opacity, mask, M_host, stream)
                         : v1_decode_fwd(d, ws, neural_opacity, mask, M_host, stream);
}
extern "C" int splatco_decode_emit(const splatco_decode_desc *d, const void *ws, int M, float *xyz, float *color,
                                   float *opacity, float *scaling, float *rot, void *stream) {
    if (check_desc(d)) return -1;
    return use_v2(d->rc) ? v2_decode_emit(d, ws, M, xyz, color, opacity, scaling, rot, stream)
                         : v1_decode_emit(d, ws, M, xyz, color, opacity, scaling, rot, stream);
}
extern "C" int splatco_decode_bwd(const splatco_decode_desc *d, const void *fwd_ws, void *bwd_ws, int M,
                                  const float *d_xyz, const float *d_color, const float *d_opacity,
                                  const float *d_scaling, const float *d_rot, const float *d_neural_opacity,
                                  const splatco_decode_grads *g, void *stream) {
    if (check_desc(d)) return -1;
    return use_v2(d->rc) ? v2_decode_bwd(d, fwd_ws, bwd_ws, M, d_xyz, d_color, d_opacity, d_scaling, d_rot, d_neural_opacity, g, stream)
                         : v1_decode_bwd(d, fwd_ws, bwd_ws, M, d_xyz, d_color, d_opacity, d_scaling, d_rot, d_neural_opacity, g, stream);
}

extern "C" int splatco_decode_bwd_camera(const splatco_decode_desc *d, const void *fwd_ws, void *bwd_ws, int M,
                                         const float *d_xyz, const float *d_color, const float *d_opacity,
                                         const float *d_scaling, const float *d_rot, const float *d_neural_opacity,
                                         const splatco_decode_grads *g, void *ws, float *d_cam, void *stream) {
    if (check_desc(d)) return -1;
    SPLATCO_REQUIRE(d_cam && (d->V == 0 || ws), "decode_bwd_camera: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (d->V == 0) {
        SPLATCO_CHECK_CUDA(cudaMemsetAsync(d_cam, 0, 3 * sizeof(float), st));
        return 0;
    }
    const bool v2 = use_v2(d->rc);
    const int rc = v2 ? v2_decode_bwd(d, fwd_ws, bwd_ws, M, d_xyz, d_color, d_opacity, d_scaling, d_rot, d_neural_opacity, g, stream)
                      : v1_decode_bwd(d, fwd_ws, bwd_ws, M, d_xyz, d_color, d_opacity, d_scaling, d_rot, d_neural_opacity, g, stream);
    if (rc) return rc;
    const float4 *X, *G;
    int nch = 0;
    if (v2) {
        const D2Dims dd = d2_dims(d2_layout_rows(d), d->rc, d->level);
        X = f2_view(const_cast<void *>(fwd_ws), dd).XT;
        G = b2_view(bwd_ws, dd).DUT;
        nch = dd.nch;
    } else {
        const DecDims dd = dec_dims(d->V, d->rc, d->level);
        X = reinterpret_cast<const float4 *>(fwd_view(const_cast<void *>(fwd_ws), dd).XIN);
        G = reinterpret_cast<const float4 *>(bwd_view(bwd_ws, dd).DX);
    }
    const int nb = ceil_div(d->V, CAM_ROWS);
    dec_camera_grad_kernel<<<nb, CAM_ROWS, 0, st>>>(d->V, nch, X, G, (float *)ws);
    SPLATCO_CHECK_LAUNCH();
    camera_sum_kernel<<<1, 1024, 0, st>>>(nb, 3, 3, -1.0f, (const float *)ws, d_cam, nullptr);
    SPLATCO_CHECK_LAUNCH();
    return 0;
}
