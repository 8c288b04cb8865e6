// Block-circulant (16 x 16) Bussgang-GMM estimate kernel, FP32 + tensor-core version of qce_circ.cu (QCE_PREC_TC).
//
// Same maths as circ_kernel (C_h,k = F^H diag(c_k) F, F = F_16 (x) F_16, A = I, zero means):
//     rt = F r        l_k = logc_k - sum_i |rt_i|^2 / lambda_k,i        h = F^H [ (sum_k w_k(l) g_k) .* rt ]
// The roofline of this path is HBM (32 N bytes of complex128 I/O per pilot, SURVEY.md section 8d); to get there the side work
// must leave the FP64 pipe:
//   * the two 2-D DFTs run as radix-4 FFTs in FP32 registers (one thread per 16-point transform): the block axis fused into
//     the coalesced global load / store (16 lanes = 256 contiguous bytes), the contiguous axis through a pair-swizzled
//     shared-memory tile (row owners use 128-bit, column owners 64-bit accesses, both bank-conflict free);
//   * the two [N x K] real contractions run on the tensor cores as split-FP16 GEMMs (mma.sync m16n8k16, FP32 accumulation):
//     both operands are computed data, so each is a (hi, lo) FP16 pair and a product is three MMAs (hi*hi + lo*hi + hi*lo,
//     ~22 significant bits).  |rt|^2 is scaled per pilot by a power of two (Parseval bounds it), the parameter matrices by a
//     global power of two fixed at set_params time.  The constant operands are pre-packed in mma fragment order (one 16-byte
//     load per lane per 8 x 16 block, hi and lo together) and stream from L2.
// One CTA = 32 pilots, 256 threads, ~100 KB shared memory -> two CTAs per SM overlap each other's load / compute / store phases.
// Any real-valued pilots are accepted (no grid assumption: Lloyd-Max labels, infinite resolution).
#include <stdlib.h>

#include "qce_common.cuh"
#include "qce_tc_shared.cuh"

namespace qce {

namespace {

constexpr int CT_P = 32;             // pilots per CTA
constexpr int CT_NW = 8;             // warps per CTA (16 warps with 64 registers each measured 7 % slower)
constexpr int CT_N = 256;            // bins (16 x 16)
constexpr int CT_EP = CT_N + 8;      // pitch (halves) of the |rt|^2 operand rows: 528 B = odd multiple of 16 B (ldmatrix conflict-free)
constexpr int CT_R_BYTES = 34816;    // operand region: E hi/lo, later log-probabilities | weight hi/lo
constexpr int CT_XP = CT_N + 8;      // pitch (float2) of one pilot's rt tile: 2112 B = 64 mod 128, so that the float4 updates of
                                     // two pilots (GEMM 2 epilogue) fall into different halves of the 32 banks
#ifndef CT_TWOSUM_EVERY
#define CT_TWOSUM_EVERY 4          // K-steps accumulated in the tensor core before the exact (hi, lo) accumulation.
                                   // Measured at config 3 (rms error of l_k - l_max in nats / worst per-pilot estimate error / ms per
                                   // 2^20 pilots): 1: 0.9e-5 / 5e-6 / 3.08, 2: 1.1e-5 / 6e-6 / 2.95, 4: 1.4e-5 / 7e-6 / 2.82,
                                   // 16: 4.1e-5 / 2.3e-5 / 2.71; plain FP32 accumulation of the full 1 / lambda: 17e-5 / 9e-5 / 2.55.
                                   // Below ~1e-5 nats the FP32 FFT is the floor.
#endif
constexpr float CT_WSCALE = 1024.f;  // weights (<= 1) are scaled into the FP16 normal range

struct CircTcArgs {
    int K;
    int64_t B;
    const uint4* b1;                 // packed 1/lambda fragments  [K/8][16][32]
    const uint4* b2;                 // packed gain fragments      [32][K/16][32]
    const float2* logc2;             // [K] logc - max(logc) as (hi, lo)
    const float* ilbar;              // [N] mean over the components of 1 / lambda: reference quadratic form per pilot
    const float2* tw256;             // plain circulant (one 256-point DFT = 16 x 16 Cooley-Tukey): e^{-2 pi i m / 256}, else null
    double logc_max;
    float inv_s1, inv_s2;            // 2^-s of the packed operands
    const double2* r;
    double2* h_est;
    double* logp_out;
    const double2* h_true;
    double* acc;
    int mode, n_top, flags;
    double rho;
    int prefetch_dist;               // tiles ahead to prefetch into L2 (= resident CTAs), 0 = off
    int* fix_buf;                    // [2 + B] hard selections too close to call in FP32: count, then the pilots -- not answered
    double tie_eps;                  // here but re-evaluated by the complex128 kernel (launch_circ_rows)
};

__device__ __forceinline__ float2 operator+(const float2 a, const float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 operator-(const float2 a, const float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// a * (-i) for the forward transform, a * (+i) for the inverse
template <bool INV>
__device__ __forceinline__ float2 rot90(const float2 a) { return INV ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x); }
// a * (c -+ i s)
template <bool INV>
__device__ __forceinline__ float2 twid(const float2 a, const float c, const float s) {
    return INV ? make_float2(a.x * c - a.y * s, a.y * c + a.x * s) : make_float2(a.x * c + a.y * s, a.y * c - a.x * s);
}
template <bool INV>
__device__ __forceinline__ void dft4(float2& a, float2& b, float2& c, float2& d) {
    const float2 s0 = a + c, s1 = a - c, s2 = b + d, s3 = rot90<INV>(b - d);
    a = s0 + s2; b = s1 + s3; c = s0 - s2; d = s1 - s3;
}
// 16-point DFT in registers (radix 4, decimation in time), scaled by 1/4 (unitary); in and out in natural order
template <bool INV>
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
    constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, C2 = 0.70710678118654752f;
    #pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) dft4<INV>(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);      // over n1: position 4 k1 + n2
    // twiddles W16^(n2 k1)
    v[4 + 1] = twid<INV>(v[4 + 1], C1, S1);   v[4 + 2] = twid<INV>(v[4 + 2], C2, C2);     v[4 + 3] = twid<INV>(v[4 + 3], S1, C1);
    v[8 + 1] = twid<INV>(v[8 + 1], C2, C2);   v[8 + 2] = rot90<INV>(v[8 + 2]);            v[8 + 3] = twid<INV>(v[8 + 3], -C2, C2);
    v[12 + 1] = twid<INV>(v[12 + 1], S1, C1); v[12 + 2] = twid<INV>(v[12 + 2], -C2, C2);  v[12 + 3] = twid<INV>(v[12 + 3], -C1, -S1);
    #pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) dft4<INV>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);   // over n2: X[k1 + 4 k2] at 4 k1 + k2
    float2 o[16];
    #pragma unroll
    for (int k1 = 0; k1 < 4; ++k1)
        #pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) o[k1 + 4 * k2] = v[4 * k1 + k2];
    #pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = make_float2(o[i].x * 0.25f, o[i].y * 0.25f);
}

// KC = K / 64.  CT_NW warps per CTA: GEMM 1 gives each warp KNB = K / (8 CT_NW) blocks of 8 components, GEMM 2 G2NB = 32 / CT_NW
// blocks of 8 bins; the FFT phases run 512 / (32 CT_NW) transforms per thread.
template <int KC>
__global__ void __launch_bounds__(32 * CT_NW, 2) circ_tc_kernel(const CircTcArgs a) {
    constexpr int K = 64 * KC, NT = 32 * CT_NW, NJ = 512 / NT, KNB = K / (8 * CT_NW), G2NB = 32 / CT_NW, SPW = CT_P / CT_NW;
    static_assert(KNB >= 1 && G2NB >= 1 && NJ >= 1 && SPW >= 1, "warp split");
    constexpr int LP = K + 4;                  // pitch (floats) of the log-probability rows
    constexpr int WP = K + 8;                  // pitch (halves) of the weight operand rows
    static_assert(CT_P * LP * 4 + 2 * CT_P * WP * 2 <= CT_R_BYTES, "operand region");
    static_assert(2 * CT_P * CT_EP * 2 <= CT_R_BYTES, "operand region");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* X = reinterpret_cast<float2*>(smem_raw);                               // [32][CT_XP]: 16 x 16 bins per pilot, swizzled
    unsigned char* R = smem_raw + CT_P * CT_XP * sizeof(float2);
    __half* Ehi = reinterpret_cast<__half*>(R);
    __half* Elo = Ehi + CT_P * CT_EP;
    float* lbuf = reinterpret_cast<float*>(R);                                     // aliases E (dead after GEMM 1)
    __half* Whi = reinterpret_cast<__half*>(R + CT_P * LP * 4);
    __half* Wlo = Whi + CT_P * WP;
    float* invsc = reinterpret_cast<float*>(R + CT_R_BYTES);                       // [32] 1 / per-pilot scale of |rt|^2
    float* qref = invsc + CT_P;                                                    // [32] sum_i |rt_i|^2 mean_k(1 / lambda_k,i)
    double* red = reinterpret_cast<double*>(R + CT_R_BYTES + 256);                 // [2]
    int* tief = reinterpret_cast<int*>(R + CT_R_BYTES + 288);                      // [32] pilot handed to the complex128 kernel

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t base = (int64_t)blockIdx.x * CT_P;
    const int nvalid = (int)((a.B - base) < CT_P ? (a.B - base) : CT_P);
    if (tid < 2) red[tid] = 0.0;
    // The reads in flight per SM (two CTAs, each loading for ~1/5 of its life) cover only a third of the HBM bandwidth-delay
    // product: pull the pilots of the tile that will be scheduled one wave of CTAs later into L2 now (one bulk prefetch).
    if (tid == 0) {
        const int64_t pb = base + (int64_t)a.prefetch_dist * CT_P;
        if (pb < a.B) {
            const int64_t np = (a.B - pb) < CT_P ? (a.B - pb) : CT_P;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.r + pb * CT_N), "r"((uint32_t)(np * CT_N * sizeof(double2))) : "memory");
            if (a.acc && a.h_true)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.h_true + pb * CT_N), "r"((uint32_t)(np * CT_N * sizeof(double2))) : "memory");
        }
    }

    // X element (pilot p, block row ar, column b): pairs of columns are XOR-swizzled with the row so that a thread owning a row
    // (128-bit accesses) and a thread owning a column (64-bit accesses) are both bank-conflict free
    auto xidx = [](int p, int ar, int b) { return p * CT_XP + ar * 16 + ((((b >> 1) ^ (ar & 7)) << 1) | (b & 1)); };

    // ---- load (coalesced: the 16 lanes of a pilot read 256 contiguous bytes) + forward FFT along the block axis
    #pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int idx = tid + NT * j, p = idx >> 4, b = idx & 15;
        float2 v[16];
        if (p < nvalid) {
            const double2* src = a.r + ((base + p) * CT_N + b);
            #pragma unroll
            for (int ar = 0; ar < 16; ++ar) { const double2 d = __ldcs(src + ar * 16); v[ar] = make_float2((float)d.x, (float)d.y); }
        } else {
            #pragma unroll
            for (int ar = 0; ar < 16; ++ar) v[ar] = make_float2(0.f, 0.f);
        }
        fft16<false>(v);
        if (a.tw256) {                         // plain circulant: twiddle W_256^(n2 k1) between the two radix-16 stages
            #pragma unroll
            for (int ar = 1; ar < 16; ++ar) {
                const float2 w = __ldg(a.tw256 + ((b * ar) & 255));
                v[ar] = make_float2(v[ar].x * w.x - v[ar].y * w.y, v[ar].x * w.y + v[ar].y * w.x);
            }
        }
        #pragma unroll
        for (int ar = 0; ar < 16; ++ar) X[xidx(p, ar, b)] = v[ar];
    }
    __syncwarp();                              // pilot p is written and read by the same 16 lanes (idx >> 4 in both phases)

    // ---- forward FFT along the contiguous axis (thread = one row), |rt|^2 as per-pilot scaled FP16 (hi, lo)
    #pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int idx = tid + NT * j, p = idx >> 4, ar = idx & 15;
        float2 v[16];
        float4* row = reinterpret_cast<float4*>(X + p * CT_XP + ar * 16);
        #pragma unroll
        for (int c = 0; c < 8; ++c) { const float4 q = row[c ^ (ar & 7)]; v[2 * c] = make_float2(q.x, q.y); v[2 * c + 1] = make_float2(q.z, q.w); }
        fft16<false>(v);
        float e[16], psum = 0.f;
        #pragma unroll
        for (int c = 0; c < 8; ++c) row[c ^ (ar & 7)] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
        // The log-probabilities are ~ -N +- tens of nats: rounding them to FP32 would cost 3e-5 nats each.  Only their differences
        // matter, so everything is kept relative to a per-pilot reference quadratic form q_ref (the mean 1 / lambda over the
        // components) and to max_k logc_k; the export adds both back in FP64.
        float qr = 0.f;
        #pragma unroll
        for (int b = 0; b < 16; ++b) { e[b] = v[b].x * v[b].x + v[b].y * v[b].y; psum += e[b]; qr = fmaf(e[b], __ldg(a.ilbar + ar * 16 + b), qr); }
        #pragma unroll
        for (int off = 8; off > 0; off >>= 1) {                                                     // the 16 rows of pilot p
            psum += __shfl_xor_sync(0xffffffffu, psum, off);
            qr += __shfl_xor_sync(0xffffffffu, qr, off);
        }
        if (ar == 0) qref[p] = qr;
        int ex = 0;
        float sc = 1.f;
        if (psum > 0.f && psum < 3.0e38f) { frexpf(psum, &ex); sc = ldexpf(1.f, 14 - ex); }         // every e * sc < 2^14
        if (ar == 0) invsc[p] = 1.f / sc;
        uint32_t hi2[8], lo2[8];
        #pragma unroll
        for (int c = 0; c < 8; ++c) {
            __half h0, l0, h1, l1;
            split_half(e[2 * c] * sc, h0, l0);
            split_half(e[2 * c + 1] * sc, h1, l1);
            hi2[c] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
            lo2[c] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
        }
        uint4* eh = reinterpret_cast<uint4*>(Ehi + p * CT_EP + ar * 16);
        uint4* el = reinterpret_cast<uint4*>(Elo + p * CT_EP + ar * 16);
        eh[0] = make_uint4(hi2[0], hi2[1], hi2[2], hi2[3]); eh[1] = make_uint4(hi2[4], hi2[5], hi2[6], hi2[7]);
        el[0] = make_uint4(lo2[0], lo2[1], lo2[2], lo2[3]); el[1] = make_uint4(lo2[4], lo2[5], lo2[6], lo2[7]);
    }
    __syncthreads();

    // ---- GEMM 1: q'[p][k] = sum_i E[p][i] (1 / lambda[k][i] - ilbar[i])   (warp: 32 pilots x KNB blocks of 8 components)
    // The constant fragments stream from L2: they are fetched PF k-steps ahead of their MMAs.
    // Precision: q is ~N nats and the combination weights need it to ~1e-5 nats, which an FP32 tensor-core accumulator cannot
    // hold over 48 accumulations (measured 2e-4 nats rms).  So (a) the operand is the DEVIATION of 1 / lambda from its mean over
    // the components (the common part cancels in the softmax and is evaluated once per pilot, q_ref), and (b) every group of
    // CT_TWOSUM_EVERY K-steps starts from a zero accumulator and is added to a running (hi, lo) FP32 pair with an exact TwoSum.
    const int g = lane >> 2, t4 = lane & 3;
    {
        float sum_hi[2][KNB][4], sum_lo[2][KNB][4];
        #pragma unroll
        for (int m = 0; m < 2; ++m)
            #pragma unroll
            for (int n = 0; n < KNB; ++n)
                #pragma unroll
                for (int c = 0; c < 4; ++c) { sum_hi[m][n][c] = 0.f; sum_lo[m][n][c] = 0.f; }
        const uint4* bp = a.b1 + ((size_t)(warp * KNB) * 16) * 32 + lane;
        constexpr int KS = CT_N / 16, PF = 4, TS_EVERY = CT_TWOSUM_EVERY;
        uint4 bq[PF][KNB];
        float acc[2][KNB][4];
        #pragma unroll
        for (int f = 0; f < PF; ++f)
            #pragma unroll
            for (int n = 0; n < KNB; ++n) bq[f][n] = __ldg(bp + ((size_t)n * 16 + f) * 32);
        #pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            uint32_t ah[2][4], al[2][4];
            #pragma unroll
            for (int m = 0; m < 2; ++m) {
                const int off = (m * 16 + (lane & 15)) * CT_EP + ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(ah[m], Ehi + off);
                ldmatrix_x4(al[m], Elo + off);
            }
            uint4 bv[KNB];
            #pragma unroll
            for (int n = 0; n < KNB; ++n) {
                bv[n] = bq[ks % PF][n];
                if (ks + PF < KS) bq[ks % PF][n] = __ldg(bp + ((size_t)n * 16 + ks + PF) * 32);
            }
            if (ks % TS_EVERY == 0) {
                #pragma unroll
                for (int m = 0; m < 2; ++m)
                    #pragma unroll
                    for (int n = 0; n < KNB; ++n)
                        #pragma unroll
                        for (int c = 0; c < 4; ++c) acc[m][n][c] = 0.f;
            }
            // pass-major order: consecutive MMAs hit different accumulators
            #pragma unroll
            for (int pass = 0; pass < 3; ++pass)
                #pragma unroll
                for (int n = 0; n < KNB; ++n)
                    #pragma unroll
                    for (int m = 0; m < 2; ++m)
                        mma16816(acc[m][n], pass == 1 ? al[m] : ah[m], pass == 2 ? bv[n].z : bv[n].x, pass == 2 ? bv[n].w : bv[n].y);
            if (ks % TS_EVERY == TS_EVERY - 1)
            #pragma unroll
            for (int m = 0; m < 2; ++m)
                #pragma unroll
                for (int n = 0; n < KNB; ++n)
                    #pragma unroll
                    for (int c = 0; c < 4; ++c) {        // (sum_hi, sum_lo) += acc without losing the rounding error (Knuth TwoSum)
                        const float x = sum_hi[m][n][c], y = acc[m][n][c];
                        const float t = x + y, bb = t - x;
                        sum_lo[m][n][c] += (x - (t - bb)) + (y - bb);
                        sum_hi[m][n][c] = t;
                    }
        }
        __syncthreads();                       // every warp is done with E: its space becomes the log-probability rows
        #pragma unroll
        for (int m = 0; m < 2; ++m)
            #pragma unroll
            for (int n = 0; n < KNB; ++n) {
                const int k = (warp * KNB + n) * 8 + 2 * t4;
                const float2 lc0 = __ldg(a.logc2 + k), lc1 = __ldg(a.logc2 + k + 1);
                #pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int p = m * 16 + g + 8 * hh;
                    const float s = invsc[p] * a.inv_s1;                               // a power of two: the products are exact
                    const float l0 = (lc0.x - sum_hi[m][n][2 * hh] * s) + (lc0.y - sum_lo[m][n][2 * hh] * s);
                    const float l1 = (lc1.x - sum_hi[m][n][2 * hh + 1] * s) + (lc1.y - sum_lo[m][n][2 * hh + 1] * s);
                    *reinterpret_cast<float2*>(lbuf + p * LP + k) = make_float2(l0, l1);
                }
            }
    }
    __syncthreads();

    // ---- combination weights per pilot
    if (a.logp_out) {
        for (int o = tid; o < nvalid * K; o += NT) a.logp_out[base * K + o] = tc_logp_export((double)lbuf[(o / K) * LP + (o % K)] + (a.logc_max - (double)qref[o / K]));
        __syncthreads();
    }
    if (a.mode == QCE_MODE_ALL) {
        #pragma unroll
        for (int pp = 0; pp < SPW; ++pp) {
            const int p = warp * SPW + pp;
            float v[K / 32], mx = -INFINITY;
            #pragma unroll
            for (int j = 0; j < K / 32; ++j) { v[j] = lbuf[p * LP + lane + 32 * j]; mx = fmaxf(mx, v[j]); }
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            float sum = 0.f;
            #pragma unroll
            for (int j = 0; j < K / 32; ++j) { v[j] = __expf(v[j] - mx); sum += v[j]; }
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
            const float inv = CT_WSCALE / sum;
            #pragma unroll
            for (int j = 0; j < K / 32; ++j) {
                __half hi, lo;
                split_half(v[j] * inv, hi, lo);
                Whi[p * WP + lane + 32 * j] = hi;
                Wlo[p * WP + lane + 32 * j] = lo;
            }
        }
    } else {
        if (tid < CT_P) {
            bool tie = false;
            weights_from_logp(lbuf + tid * LP, K, a.mode, a.n_top, a.rho, a.flags, &tie, a.tie_eps);
            tie = tie && tid < nvalid;
            tief[tid] = tie;
            if (tie) a.fix_buf[2 + atomicAdd(a.fix_buf, 1)] = (int)(base + tid);
        }
        __syncthreads();
        for (int o = tid; o < CT_P * K; o += NT) {
            const int p = o / K, k = o % K;
            __half hi, lo;
            split_half(lbuf[p * LP + k] * CT_WSCALE, hi, lo);
            Whi[p * WP + k] = hi;
            Wlo[p * WP + k] = lo;
        }
    }
    __syncthreads();

    // ---- GEMM 2: G[p][i] = sum_k w[p][k] g[k][i]   (warp: 32 pilots x G2NB blocks of 8 bins), rt <- G .* rt
    if (a.h_est || a.acc) {
        float acc[2][G2NB][4];
        #pragma unroll
        for (int m = 0; m < 2; ++m)
            #pragma unroll
            for (int n = 0; n < G2NB; ++n)
                #pragma unroll
                for (int c = 0; c < 4; ++c) acc[m][n][c] = 0.f;
        const uint4* bp = a.b2 + ((size_t)(warp * G2NB) * (K / 16)) * 32 + lane;
        constexpr int KS = K / 16, PF = 2;
        uint4 bq[PF][G2NB];
        #pragma unroll
        for (int f = 0; f < PF; ++f)
            #pragma unroll
            for (int n = 0; n < G2NB; ++n) bq[f][n] = __ldg(bp + ((size_t)n * KS + f) * 32);
        #pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            uint32_t ah[2][4], al[2][4];
            #pragma unroll
            for (int m = 0; m < 2; ++m) {
                const int off = (m * 16 + (lane & 15)) * WP + ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(ah[m], Whi + off);
                ldmatrix_x4(al[m], Wlo + off);
            }
            uint4 bv[G2NB];
            #pragma unroll
            for (int n = 0; n < G2NB; ++n) {
                bv[n] = bq[ks % PF][n];
                if (ks + PF < KS) bq[ks % PF][n] = __ldg(bp + ((size_t)n * KS + ks + PF) * 32);
            }
            #pragma unroll
            for (int pass = 0; pass < 3; ++pass)
                #pragma unroll
                for (int n = 0; n < G2NB; ++n)
                    #pragma unroll
                    for (int m = 0; m < 2; ++m)
                        mma16816(acc[m][n], pass == 1 ? al[m] : ah[m], pass == 2 ? bv[n].z : bv[n].x, pass == 2 ? bv[n].w : bv[n].y);
        }
        const float gs = a.inv_s2 / CT_WSCALE;
        #pragma unroll
        for (int m = 0; m < 2; ++m)
            #pragma unroll
            for (int n = 0; n < G2NB; ++n) {
                const int bin = (warp * G2NB + n) * 8 + 2 * t4, ar = bin >> 4, b = bin & 15;      // bins (b, b + 1): one swizzled pair
                #pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int p = m * 16 + g + 8 * hh;
                    float4* x = reinterpret_cast<float4*>(X + xidx(p, ar, b));
                    const float g0 = acc[m][n][2 * hh] * gs, g1 = acc[m][n][2 * hh + 1] * gs;
                    const float4 q = *x;
                    *x = make_float4(q.x * g0, q.y * g0, q.z * g1, q.w * g1);
                }
            }
        __syncthreads();

        // ---- inverse FFT along the contiguous axis (thread = one row)
        #pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int idx = tid + NT * j, p = idx >> 4, ar = idx & 15;
            float2 v[16];
            float4* row = reinterpret_cast<float4*>(X + p * CT_XP + ar * 16);
            #pragma unroll
            for (int c = 0; c < 8; ++c) { const float4 q = row[c ^ (ar & 7)]; v[2 * c] = make_float2(q.x, q.y); v[2 * c + 1] = make_float2(q.z, q.w); }
            fft16<true>(v);
            #pragma unroll
            for (int c = 0; c < 8; ++c) row[c ^ (ar & 7)] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
        }
        __syncwarp();                          // same 16 lanes per pilot again

        // ---- inverse FFT along the block axis fused into the (coalesced) store, NMSE accumulators
        float errf = 0.f, pwf = 0.f;
        #pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int idx = tid + NT * j, p = idx >> 4, b = idx & 15;
            float2 v[16];
            #pragma unroll
            for (int ar = 0; ar < 16; ++ar) v[ar] = X[xidx(p, ar, b)];
            if (a.tw256) {
                #pragma unroll
                for (int ar = 1; ar < 16; ++ar) {
                    const float2 w = __ldg(a.tw256 + ((b * ar) & 255));
                    v[ar] = make_float2(v[ar].x * w.x + v[ar].y * w.y, v[ar].y * w.x - v[ar].x * w.y);
                }
            }
            fft16<true>(v);
            if (p < nvalid && !(a.mode != QCE_MODE_ALL && tief[p])) {
                const size_t o = (size_t)(base + p) * CT_N + b;
                if (a.h_est) {
                    #pragma unroll
                    for (int ar = 0; ar < 16; ++ar) __stcs(a.h_est + o + ar * 16, make_double2((double)v[ar].x, (double)v[ar].y));
                }
                if (a.acc && a.h_true) {
                    #pragma unroll
                    for (int ar = 0; ar < 16; ++ar) {
                        const double2 h = __ldcs(a.h_true + o + ar * 16);
                        const float hx = (float)h.x, hy = (float)h.y, dx = v[ar].x - hx, dy = v[ar].y - hy;
                        errf = fmaf(dx, dx, fmaf(dy, dy, errf));
                        pwf = fmaf(hx, hx, fmaf(hy, hy, pwf));
                    }
                }
            }
        }
        if (a.acc) {
            double err = (double)errf, pw = (double)pwf;
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                err += __shfl_xor_sync(0xffffffffu, err, off);
                pw += __shfl_xor_sync(0xffffffffu, pw, off);
            }
            if (lane == 0) { atomicAdd(&red[0], err); atomicAdd(&red[1], pw); }
            __syncthreads();
            if (tid == 0) {
                int cnt = nvalid;
                if (a.mode != QCE_MODE_ALL) for (int p = 0; p < nvalid; ++p) cnt -= tief[p];
                atomicAdd(a.acc + 0, red[0]); atomicAdd(a.acc + 1, red[1]); atomicAdd(a.acc + 2, (double)cnt);
            }
        }
    }
}

// Constant operands in mma.m16n8k16 B-fragment order.  Thread (g = lane / 4, t = lane % 4) of block (nb, ks) holds
// b0 = {B[16 ks + 2t][8 nb + g], B[16 ks + 2t + 1][.]}, b1 = the same 8 rows further; stored as uint4 {b0 hi, b1 hi, b0 lo, b1 lo}.
// which = 0: B[i][k] = 1 / lambda (source inv_lambda_t [N][K]),  which = 1: B[k][i] = gain (source gain [K][N]).
// sub != nullptr: sub[row] is subtracted first (the 1 / lambda operand is packed as its deviation from the mean over the components).
// one_d: the bin axis (rows of 1 / lambda, columns of the gains) is stored in the order the two-stage 256-point FFT leaves it:
// position s = 16 k1 + k2 holds frequency k1 + 16 k2.
__device__ __forceinline__ int circ_bin_of(int s, int one_d) { return one_d ? (s >> 4) + 16 * (s & 15) : s; }

__global__ void circ_tc_pack_kernel(const double* __restrict__ src, const float* __restrict__ sub, int rows, int cols, double scale,
                                    uint4* __restrict__ out, int perm_rows, int perm_cols) {
    const int nks = rows / 16, nnb = cols / 8;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nnb * nks * 32) return;
    const int lane = idx & 31, ks = (idx >> 5) % nks, nb = (idx >> 5) / nks;
    const int g = lane >> 2, t = lane & 3, col = nb * 8 + g;
    __half hi[4], lo[4];
    #pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int row = ks * 16 + 2 * t + (e & 1) + 8 * (e >> 1);
        const double x = (src[(size_t)circ_bin_of(row, perm_rows) * cols + circ_bin_of(col, perm_cols)] - (sub ? (double)sub[row] : 0.0)) * scale;
        hi[e] = __double2half(x);
        lo[e] = __double2half(x - (double)__half2float(hi[e]));
    }
    auto pack = [](__half a0, __half a1) { return (uint32_t)__half_as_ushort(a0) | ((uint32_t)__half_as_ushort(a1) << 16); };
    out[idx] = make_uint4(pack(hi[0], hi[1]), pack(hi[2], hi[3]), pack(lo[0], lo[1]), pack(lo[2], lo[3]));
}

__global__ void circ_tc_logc_kernel(const double* __restrict__ logc, int K, double logc_max, float2* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < K) out[k] = tc_logc_pair(logc[k] - logc_max);
}

__global__ void circ_tc_ilbar_kernel(const double* __restrict__ inv_lambda_t, int N, int K, int one_d, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;       // storage position
    if (i >= N) return;
    double sum = 0.0;
    for (int k = 0; k < K; ++k) sum += inv_lambda_t[(size_t)circ_bin_of(i, one_d) * K + k];
    out[i] = (float)(sum / K);
}

__global__ void circ_tc_twiddle_kernel(float2* __restrict__ out) {
    const int m = threadIdx.x;
    double sn, cs;
    sincospi(-2.0 * m / 256.0, &sn, &cs);
    out[m] = make_float2((float)cs, (float)sn);
}

double pow2_scale_for(const double* dev, size_t n, cudaStream_t s, qce_status* st) {
    // power of two that puts the largest magnitude into [2^12, 2^13)
    double* host = (double*)malloc(n * sizeof(double));
    *st = QCE_OK;
    if (!host || cudaMemcpyAsync(host, dev, n * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
        free(host);
        set_error("circulant tensor-core pack: device read failed");
        *st = QCE_ERR_CUDA;
        return 1.0;
    }
    double mx = 0.0;
    bool finite = true;
    for (size_t i = 0; i < n; ++i) { const double v = fabs(host[i]); if (!(v < 1e300)) finite = false; if (v > mx) mx = v; }
    free(host);
    if (!finite || !(mx > 0.0)) return 0.0;
    int ex = 0;
    frexp(mx, &ex);
    return ldexp(1.0, 13 - ex);
}

}  // namespace

bool circ_tc_shape_ok(const qce_circ_model* m) {     // block-circulant 16 x 16, or plain circulant of length 256 (one two-stage FFT)
    return ((m->n1 == 16 && m->n2 == 16) || (m->n1 == 1 && m->n2 == 256)) && (m->n_comp == 64 || m->n_comp == 128);
}

void circ_tc_free(qce_circ_model* m) {
    cudaFree(m->tc_b1); cudaFree(m->tc_b2); cudaFree(m->tc_logc2); cudaFree(m->tc_ilbar); cudaFree(m->tc_tw);
    m->tc_b1 = m->tc_b2 = m->tc_logc2 = m->tc_ilbar = m->tc_tw = nullptr;
    m->tc_ready = false;
}

qce_status circ_tc_pack(qce_circ_model* m, cudaStream_t s) {
    m->tc_ready = false;
    if (!circ_tc_shape_ok(m)) return QCE_OK;
    const size_t N = m->n_ant, K = m->n_comp;
    qce_status st = QCE_OK;
    const double s1 = pow2_scale_for(m->inv_lambda_t, N * K, s, &st);
    if (st) return st;
    const double s2 = pow2_scale_for(m->gain, N * K, s, &st);
    if (st) return st;
    if (!(s1 > 0.0) || !(s2 > 0.0)) return QCE_OK;                      // degenerate parameters: complex128 kernel only
    const size_t frag_bytes = (N * K / 4) * sizeof(uint4);              // 4 values per lane entry, hi and lo: 16 B
    if (!m->tc_b1) {
        QCE_CUDA_TRY(cudaMalloc(&m->tc_b1, frag_bytes));
        QCE_CUDA_TRY(cudaMalloc(&m->tc_b2, frag_bytes));
        QCE_CUDA_TRY(cudaMalloc(&m->tc_logc2, K * sizeof(float2)));
        QCE_CUDA_TRY(cudaMalloc(&m->tc_ilbar, N * sizeof(float)));
    }
    const int one_d = m->n1 == 1;
    if (one_d && !m->tc_tw) {
        QCE_CUDA_TRY(cudaMalloc(&m->tc_tw, 256 * sizeof(float2)));
        circ_tc_twiddle_kernel<<<1, 256, 0, s>>>((float2*)m->tc_tw);
        QCE_CHECK_LAUNCH("circ_tc_twiddle_kernel");
    }
    const int total = (int)(N * K / 4);
    circ_tc_ilbar_kernel<<<(unsigned)((N + 127) / 128), 128, 0, s>>>(m->inv_lambda_t, (int)N, (int)K, one_d, (float*)m->tc_ilbar);
    QCE_CHECK_LAUNCH("circ_tc_ilbar_kernel");
    circ_tc_pack_kernel<<<(total + 255) / 256, 256, 0, s>>>(m->inv_lambda_t, (const float*)m->tc_ilbar, (int)N, (int)K, s1, (uint4*)m->tc_b1, one_d, 0);
    QCE_CHECK_LAUNCH("circ_tc_pack_kernel");
    circ_tc_pack_kernel<<<(total + 255) / 256, 256, 0, s>>>(m->gain, nullptr, (int)K, (int)N, s2, (uint4*)m->tc_b2, 0, one_d);
    QCE_CHECK_LAUNCH("circ_tc_pack_kernel");
    {
        double* h_logc = (double*)malloc(K * sizeof(double));
        if (!h_logc || cudaMemcpyAsync(h_logc, m->logc, K * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
            cudaStreamSynchronize(s) != cudaSuccess) {
            free(h_logc);
            set_error("circulant tensor-core pack: device read failed");
            return QCE_ERR_CUDA;
        }
        double mx = h_logc[0];
        for (size_t k = 1; k < K; ++k) mx = h_logc[k] > mx ? h_logc[k] : mx;
        free(h_logc);
        m->tc_logc_max = mx;
    }
    circ_tc_logc_kernel<<<(unsigned)((K + 127) / 128), 128, 0, s>>>(m->logc, (int)K, m->tc_logc_max, (float2*)m->tc_logc2);
    QCE_CHECK_LAUNCH("circ_tc_logc_kernel");
    m->tc_inv_s1 = (float)(1.0 / s1);
    m->tc_inv_s2 = (float)(1.0 / s2);
    m->tc_ready = true;
    return QCE_OK;
}

// fix list of a launch, in the stream's scratch; the count is reset in stream order
static qce_status circ_fix_list(cudaStream_t s, int64_t rows, int** out) {
    StreamScratch* sc = scratch_for(s);
    qce_status st = grow(sc->circ_fix, ((size_t)rows + 2) * sizeof(int));     // [0] count, [1] unused here (layout of qce_last_fix_count), then the list
    if (st) return st;
    QCE_CUDA_TRY(cudaMemsetAsync(sc->circ_fix.p, 0, 2 * sizeof(int), s));
    sc->last_fix = *out = (int*)sc->circ_fix.p;
    return QCE_OK;
}

template <int KC>
static qce_status launch_circ_tc_k(const CircTcArgs& a, cudaStream_t s) {
    constexpr size_t SMEM = CT_P * CT_XP * sizeof(float2) + CT_R_BYTES + 512;
    static PerDeviceOnce once;
    if (once.first(current_device())) QCE_CUDA_TRY(cudaFuncSetAttribute(circ_tc_kernel<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    circ_tc_kernel<KC><<<(unsigned)((a.B + CT_P - 1) / CT_P), 32 * CT_NW, SMEM, s>>>(a);
    QCE_CHECK_LAUNCH("circ_tc_kernel");
    return QCE_OK;
}

qce_status launch_circ_tc(const qce_circ_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                          double* h_est, double* logp_out, const double* h_true, double* acc) {
    if (!m->tc_ready) { set_error("circulant tensor-core kernel: n1=%d n2=%d K=%d not supported", m->n1, m->n2, m->n_comp); return QCE_ERR_UNSUPPORTED; }
    if (B == 0) return QCE_OK;
    CircTcArgs a;
    a.K = m->n_comp; a.B = B;
    a.b1 = (const uint4*)m->tc_b1; a.b2 = (const uint4*)m->tc_b2; a.logc2 = (const float2*)m->tc_logc2;
    a.ilbar = (const float*)m->tc_ilbar; a.logc_max = m->tc_logc_max;
    a.tw256 = (m->n1 == 1) ? (const float2*)m->tc_tw : nullptr;
    a.inv_s1 = m->tc_inv_s1; a.inv_s2 = m->tc_inv_s2;
    a.r = (const double2*)r; a.h_est = (double2*)h_est; a.logp_out = logp_out; a.h_true = (const double2*)h_true; a.acc = acc;
    a.mode = mode; a.n_top = n_top; a.flags = m->flags; a.rho = rho;
    {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const int pf_env = getenv("QCE_CIRC_PREFETCH") ? atoi(getenv("QCE_CIRC_PREFETCH")) : -1;
        a.prefetch_dist = pf_env >= 0 ? pf_env : sms;     // measured: 0 -> 396, sms/2 .. sms -> 412, 2 sms -> 354 M est/s at config 3
    }
    // hard selections: pilots whose selection the FP32 log-likelihoods (~1.4e-5 nats rms, profiles/r02_flip_rate.json) cannot
    // decide go on a fix list and are answered by the complex128 kernel.  QCE_TC_TIE_EPS overrides the gap (0: no re-evaluation).
    // 'all' lists nothing, but its list is still reset: qce_last_fix_count reports this call's 0, not an earlier call's count
    a.fix_buf = nullptr;
    a.tie_eps = getenv("QCE_TC_TIE_EPS") ? atof(getenv("QCE_TC_TIE_EPS")) : 5e-4;
    {
        int* list = nullptr;
        qce_status st = circ_fix_list(s, mode == QCE_MODE_ALL ? 0 : B, &list);
        if (st) return st;
        if (mode != QCE_MODE_ALL) a.fix_buf = list;
    }
    const qce_status st = m->n_comp == 64 ? launch_circ_tc_k<1>(a, s) : launch_circ_tc_k<2>(a, s);
    if (st || mode == QCE_MODE_ALL || !(h_est || acc)) return st;
    return launch_circ_rows(m, s, r, a.fix_buf + 2, a.fix_buf, B, mode, n_top, rho, h_est, h_true, acc);
}

}  // namespace qce
