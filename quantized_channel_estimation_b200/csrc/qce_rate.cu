// Accumulators of the scripts' statistical lower bound on the achievable rate (Bussgang_GMM.py:291-309, Bussgang_MFA.py:154-172;
// utils.rate_lower_bound is the complex128 torch form over a materialised estimate array).  Per pilot row b:
//     g_b     = h_est_b / max(|h_est_b|^2, 0.1)           (the scripts divide by the SQUARED norm)
//     inner_b = g_b^H B h_b                               B = diagonal Bussgang matrix of the global model
//     q_b     = Re g_b^H C_q g_b                          C_q = C_r - B C B^H, dense N x N
// and acc[0..4] += { sum Re inner, sum Im inner, sum |inner|^2, sum q, rows }.  The bound is a function of these five sums only
// (utils.rate_from_accumulators), and they add across chunks and ranks like the NMSE accumulators.
//   * norm, g and inner: FP64 (O(N) per pilot).  The variance is S2/n - |S1/n|^2, a difference of large sums: the per-pilot inner
//     products must not carry FP32 rounding into it.
//   * q: a [pilots x 2N] . [2N x 2N] product on the tensor cores (mma.sync m16n8k16, FP32 accumulation) with the real embedding
//     E[2i+a][2j+b] = {Re, -Im; Im, Re} of the Hermitian part (C_q + C_q^H) / 2 (same Re g^H C_q g, and E is symmetric), then a
//     row-wise dot with g in the epilogue.  Both operands are computed data, so each is an FP16 (hi, lo) pair and a product is
//     three MMAs (hi*hi + lo*hi + hi*lo, ~22 significant bits), as in circ_tc_kernel.  g is scaled per pilot by a power of two
//     that puts max |Re g|, |Im g| into [2^12, 2^13), E by one global power of two fixed at set_params time; both are undone
//     exactly before the FP64 sum.  The E fragments are pre-packed in mma B-fragment order and stream from L2.
// Any 1 <= N <= 256: the model is zero-padded to Np = next multiple of 16 (zero g entries, zero E rows / columns: exact).
// One CTA = 64 pilots, 8 warps.  Per pilot the kernel reads 16 N bytes of estimates and 8 N or 16 N of channels; the
// quadratic form is 3 (2 Np)^2 MACs, so at N = 64 the kernel is bound by those reads.
#include <math.h>
#include <stdlib.h>

#include "qce_common.cuh"
#include "qce_tc_shared.cuh"

namespace qce {

namespace {

constexpr int RT_P = 64;               // pilots per CTA
constexpr int RT_NW = 8;               // warps per CTA
constexpr int RT_MT = RT_P / 16;       // m16 tiles per CTA

struct RateArgs {
    const double2* h_est;              // [B][N]
    const void* h_true;                // [B][N] c64 / c128
    int h_true_c64;
    const double2* buss;               // [N] diagonal of B
    const uint4* frag;                 // [Np / 4 n-blocks][Np / 8 k-steps][32 lanes] {b0 hi, b1 hi, b0 lo, b1 lo}
    double inv_se;                     // 2^-s of the packed E
    int N, Np;
    int64_t B;
    double* acc;                       // [5]
    int prefetch_dist;                 // tiles ahead whose inputs are pulled into L2 (one per SM: half a wave of CTAs)
};

__device__ __forceinline__ void prefetch_l2(const void* p, uint64_t bytes) {
    bytes &= ~(uint64_t)15;                                           // a hint: 16-byte granules only
    if (bytes && ((uintptr_t)p & 15) == 0)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"((uint32_t)bytes) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// NJ = ceil(Np / 32): entries of a row per lane in the FP64 phase
template <int NJ>
__global__ void __launch_bounds__(32 * RT_NW, 2) rate_tc_kernel(const RateArgs a) {
    const int pitch = 2 * a.Np + 8;    // halves: (4 Np + 16) bytes = odd multiple of 16 B (Np % 16 == 0): ldmatrix conflict-free
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __half* Ghi = reinterpret_cast<__half*>(smem_raw);                   // [P][pitch] scaled g, real-interleaved, FP16 hi
    __half* Glo = Ghi + RT_P * pitch;                                    // ... and lo
    float* qpart = reinterpret_cast<float*>(Glo + RT_P * pitch);         // [NW][P] per-warp partial quadratic forms
    double* unsc = reinterpret_cast<double*>(qpart + RT_NW * RT_P);      // [P] 1 / (scale^2 s_E)
    double* red = unsc + RT_P;                                           // [NW][4]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t base = (int64_t)blockIdx.x * RT_P;
    const int nvalid = (int)((a.B - base) < RT_P ? (a.B - base) : RT_P);
    // the loads of the FP64 phase are the kernel's HBM traffic, and a CTA has none in flight during its tensor-core phase: pull
    // the rows of the tile scheduled half a wave later into L2 now
    if (tid == 0) {
        const int64_t pb = base + (int64_t)a.prefetch_dist * RT_P;
        if (pb < a.B) {
            const int64_t np = (a.B - pb) < RT_P ? (a.B - pb) : RT_P;
            const int hs = a.h_true_c64 ? 8 : 16;
            prefetch_l2(a.h_est + pb * a.N, (uint64_t)np * a.N * 16);
            prefetch_l2(reinterpret_cast<const char*>(a.h_true) + pb * a.N * hs, (uint64_t)np * a.N * hs);
        }
    }

    // ---- FP64 phase: one warp per row (RPI rows with their loads in flight together), lane owns entries lane + 32 j
    double s_re = 0.0, s_im = 0.0, s_sq = 0.0;
    constexpr int RPI = NJ >= 4 ? 1 : 4 / NJ;
    for (int p0 = warp * RPI; p0 < RT_P; p0 += RT_NW * RPI) {
        double2 he[RPI][NJ], ht[RPI][NJ];
        #pragma unroll
        for (int r = 0; r < RPI; ++r)
            #pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int i = lane + 32 * j;
                he[r][j] = make_double2(0.0, 0.0);
                ht[r][j] = make_double2(0.0, 0.0);
                if (p0 + r < nvalid && i < a.N) {
                    const size_t o = (size_t)(base + p0 + r) * a.N + i;
                    he[r][j] = __ldcs(a.h_est + o);
                    if (a.h_true_c64) {
                        const float2 f = __ldcs(reinterpret_cast<const float2*>(a.h_true) + o);
                        ht[r][j] = make_double2((double)f.x, (double)f.y);
                    } else {
                        ht[r][j] = __ldcs(reinterpret_cast<const double2*>(a.h_true) + o);
                    }
                }
            }
        #pragma unroll
        for (int r = 0; r < RPI; ++r) {
            const int p = p0 + r;
            double nrm = 0.0, ir = 0.0, ii = 0.0, mx = 0.0;
            #pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int i = lane + 32 * j;
                if (i < a.N) {
                    const double2 e = he[r][j], h = ht[r][j], b = __ldg(a.buss + i);
                    const double bx = b.x * h.x - b.y * h.y, by = b.x * h.y + b.y * h.x;      // (B h)_i
                    nrm += e.x * e.x + e.y * e.y;
                    ir += e.x * bx + e.y * by;                                                // conj(e) (B h)_i
                    ii += e.x * by - e.y * bx;
                    mx = fmax(mx, fmax(fabs(e.x), fabs(e.y)));
                }
            }
            nrm = warp_sum(nrm); ir = warp_sum(ir); ii = warp_sum(ii);
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            const double nf = nrm < 0.1 ? 0.1 : nrm;                  // np.clip(|h_est|^2, 1e-1, inf)
            if (p < nvalid) {
                const double inr = ir / nf, ini = ii / nf;
                s_re += inr; s_im += ini; s_sq += inr * inr + ini * ini;
            }
            const double gmax = mx / nf;
            double sc = 1.0;
            if (gmax > 0.0 && gmax < 1e300) { int ex = 0; frexp(gmax, &ex); sc = ldexp(1.0, 13 - ex); }
            if (lane == 0) unsc[p] = a.inv_se / sc / sc;                 // exact: powers of two, no overflow of sc^2
            const double f = sc / nf;
            #pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int i = lane + 32 * j;
                if (i < a.Np) {                                       // entries N <= i < Np are the zero padding
                    __half hx, lx, hy, ly;
                    split_half((float)(he[r][j].x * f), hx, lx);
                    split_half((float)(he[r][j].y * f), hy, ly);
                    *reinterpret_cast<__half2*>(Ghi + p * pitch + 2 * i) = __halves2half2(hx, hy);
                    *reinterpret_cast<__half2*>(Glo + p * pitch + 2 * i) = __halves2half2(lx, ly);
                }
            }
        }
    }
    if (lane == 0) { red[warp * 4 + 0] = s_re; red[warp * 4 + 1] = s_im; red[warp * 4 + 2] = s_sq; red[warp * 4 + 3] = 0.0; }
    __syncthreads();

    // ---- tensor-core phase: Y = G E (warp: all P pilots x pairs of 8-column blocks), q_b += sum_c G[b][c] Y[b][c]
    const int g = lane >> 2, t4 = lane & 3;
    const int KS = a.Np / 8;                                          // k-steps of 16 over 2 Np = pairs of n-blocks of 8
    float qp[RT_MT][2];
    #pragma unroll
    for (int m = 0; m < RT_MT; ++m) { qp[m][0] = 0.f; qp[m][1] = 0.f; }
    for (int pr = warp; pr < KS; pr += RT_NW) {
        float acc[RT_MT][2][4];
        #pragma unroll
        for (int m = 0; m < RT_MT; ++m)
            #pragma unroll
            for (int n = 0; n < 2; ++n)
                #pragma unroll
                for (int c = 0; c < 4; ++c) acc[m][n][c] = 0.f;
        const uint4* bp0 = a.frag + (size_t)(2 * pr) * KS * 32 + lane;
        const uint4* bp1 = bp0 + (size_t)KS * 32;
        // the fragments stream from L2 two k-steps ahead of their MMAs (KS >= 2)
        uint4 nx0 = __ldg(bp0), nx1 = __ldg(bp1), ny0 = __ldg(bp0 + 32), ny1 = __ldg(bp1 + 32);
        for (int ks = 0; ks < KS; ++ks) {
            const uint4 b0 = nx0, b1 = nx1;
            nx0 = ny0; nx1 = ny1;
            if (ks + 2 < KS) { ny0 = __ldg(bp0 + (size_t)(ks + 2) * 32); ny1 = __ldg(bp1 + (size_t)(ks + 2) * 32); }
            #pragma unroll
            for (int m = 0; m < RT_MT; ++m) {
                uint32_t ah[4], al[4];
                const int off = (m * 16 + (lane & 15)) * pitch + ks * 16 + (lane >> 4) * 8;
                ldmatrix_x4(ah, Ghi + off);
                ldmatrix_x4(al, Glo + off);
                mma16816(acc[m][0], ah, b0.x, b0.y);
                mma16816(acc[m][1], ah, b1.x, b1.y);
                mma16816(acc[m][0], al, b0.x, b0.y);
                mma16816(acc[m][1], al, b1.x, b1.y);
                mma16816(acc[m][0], ah, b0.z, b0.w);
                mma16816(acc[m][1], ah, b1.z, b1.w);
            }
        }
        #pragma unroll
        for (int m = 0; m < RT_MT; ++m)
            #pragma unroll
            for (int n = 0; n < 2; ++n)
                #pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int row = m * 16 + g + 8 * hh, col = (2 * pr + n) * 8 + 2 * t4;
                    const float2 gh = __half22float2(*reinterpret_cast<const __half2*>(Ghi + row * pitch + col));
                    const float2 gl = __half22float2(*reinterpret_cast<const __half2*>(Glo + row * pitch + col));
                    qp[m][hh] = fmaf(acc[m][n][2 * hh], gh.x + gl.x, fmaf(acc[m][n][2 * hh + 1], gh.y + gl.y, qp[m][hh]));
                }
    }
    #pragma unroll
    for (int m = 0; m < RT_MT; ++m)
        #pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            float v = qp[m][hh];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (t4 == 0) qpart[warp * RT_P + m * 16 + g + 8 * hh] = v;
        }
    __syncthreads();
    if (tid < RT_P) {                                                 // warps 0 and 1: one pilot per thread
        double q = 0.0;
        #pragma unroll
        for (int w = 0; w < RT_NW; ++w) q += (double)qpart[w * RT_P + tid];
        q = warp_sum(q * unsc[tid]);                                  // padding rows are zero
        if (lane == 0) red[warp * 4 + 3] = q;
    }
    __syncthreads();
    if (tid == 0) {
        double v[4] = {0.0, 0.0, 0.0, 0.0};
        for (int w = 0; w < RT_NW; ++w)
            #pragma unroll
            for (int c = 0; c < 4; ++c) v[c] += red[w * 4 + c];
        #pragma unroll
        for (int c = 0; c < 4; ++c) atomicAdd(a.acc + c, v[c]);
        atomicAdd(a.acc + 4, (double)nvalid);
    }
}

// E element (row k, column n) of the real embedding of (C_q + C_q^H) / 2, zero in the padding
__device__ __forceinline__ double rate_embed(const double2* __restrict__ cq, int N, int k, int n) {
    const int i = k >> 1, j = n >> 1;
    if (i >= N || j >= N) return 0.0;
    const double2 cij = cq[(size_t)i * N + j], cji = cq[(size_t)j * N + i];
    const double re = 0.5 * (cij.x + cji.x), im = 0.5 * (cij.y - cji.y);
    return ((k ^ n) & 1) == 0 ? re : ((k & 1) ? im : -im);
}

// E * se in mma.m16n8k16 B-fragment order: thread (g, t) of block (nb, ks) holds b0 = {E[16 ks + 2t][8 nb + g], E[16 ks + 2t + 1][.]},
// b1 = the same 8 rows further, stored as {b0 hi, b1 hi, b0 lo, b1 lo}
__global__ void rate_pack_kernel(const double2* __restrict__ cq, int N, int Np, double se, uint4* __restrict__ out) {
    const int KS = Np / 8, NB = Np / 4;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= NB * KS * 32) return;
    const int lane = idx & 31, ks = (idx >> 5) % KS, nb = (idx >> 5) / KS;
    const int col = nb * 8 + (lane >> 2), t = lane & 3;
    __half hi[4], lo[4];
    #pragma unroll
    for (int e = 0; e < 4; ++e) {
        const double x = rate_embed(cq, N, ks * 16 + 2 * t + (e & 1) + 8 * (e >> 1), col) * se;
        hi[e] = __double2half(x);
        lo[e] = __double2half(x - (double)__half2float(hi[e]));
    }
    auto pack = [](__half a0, __half a1) { return (uint32_t)__half_as_ushort(a0) | ((uint32_t)__half_as_ushort(a1) << 16); };
    out[idx] = make_uint4(pack(hi[0], hi[1]), pack(hi[2], hi[3]), pack(lo[0], lo[1]), pack(lo[2], lo[3]));
}

constexpr size_t rate_smem(int Np) {
    return (size_t)2 * RT_P * (2 * Np + 8) * sizeof(__half) + RT_NW * RT_P * sizeof(float) + RT_P * sizeof(double) + RT_NW * 4 * sizeof(double);
}

template <int NJ>
qce_status launch_rate_k(const RateArgs& a, cudaStream_t s) {
    static PerDeviceOnce once;
    if (once.first(current_device()))
        QCE_CUDA_TRY(cudaFuncSetAttribute(rate_tc_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rate_smem(32 * NJ)));
    rate_tc_kernel<NJ><<<(unsigned)((a.B + RT_P - 1) / RT_P), 32 * RT_NW, rate_smem(a.Np), s>>>(a);
    QCE_CHECK_LAUNCH("rate_tc_kernel");
    return QCE_OK;
}

}  // namespace

qce_status rate_pack(qce_rate_model* m, cudaStream_t s, const double* cq) {
    // E's power of two: the largest |entry| of the Hermitian part goes into [2^12, 2^13)
    const size_t N = m->n_ant;
    double* host = (double*)malloc(N * N * 2 * sizeof(double));
    if (!host || cudaMemcpyAsync(host, cq, N * N * 2 * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
        free(host);
        set_error("qce_rate_model_set_params: device read of C_q failed");
        return QCE_ERR_CUDA;
    }
    double mx = 0.0;
    bool finite = true;
    for (size_t i = 0; i < N; ++i)
        for (size_t j = 0; j < N; ++j) {
            const double re = 0.5 * (host[2 * (i * N + j)] + host[2 * (j * N + i)]);
            const double im = 0.5 * (host[2 * (i * N + j) + 1] - host[2 * (j * N + i) + 1]);
            if (!(fabs(re) < 1e300) || !(fabs(im) < 1e300)) finite = false;
            mx = fmax(mx, fmax(fabs(re), fabs(im)));
        }
    free(host);
    if (!finite) { set_error("qce_rate_model_set_params: C_q has non-finite entries"); return QCE_ERR_INVALID; }
    double se = 1.0;
    if (mx > 0.0) { int ex = 0; frexp(mx, &ex); se = ldexp(1.0, 13 - ex); }
    const int total = (m->n_pad / 4) * (m->n_pad / 8) * 32;
    rate_pack_kernel<<<(total + 255) / 256, 256, 0, s>>>((const double2*)cq, m->n_ant, m->n_pad, se, (uint4*)m->frag);
    QCE_CHECK_LAUNCH("rate_pack_kernel");
    m->inv_se = 1.0 / se;
    return QCE_OK;
}

qce_status launch_rate(const qce_rate_model* m, cudaStream_t s, const double* h_est, const void* h_true, int h_true_c64, int64_t B,
                       double* acc) {
    RateArgs a;
    a.h_true = h_true; a.h_true_c64 = h_true_c64;
    a.buss = (const double2*)m->buss; a.frag = (const uint4*)m->frag; a.inv_se = m->inv_se;
    a.N = m->n_ant; a.Np = m->n_pad; a.acc = acc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    a.prefetch_dist = sms;
    const int64_t chunk = (int64_t)1 << 30;                            // keeps the grid below 2^31 CTAs
    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
        a.B = (B - b0) < chunk ? (B - b0) : chunk;
        a.h_est = (const double2*)h_est + (size_t)b0 * m->n_ant;
        a.h_true = (const char*)h_true + (size_t)b0 * m->n_ant * (h_true_c64 ? 8 : 16);
        const int nj = (m->n_pad + 31) / 32;
        const qce_status st = nj == 1 ? launch_rate_k<1>(a, s) : nj == 2 ? launch_rate_k<2>(a, s) : nj <= 4 ? launch_rate_k<4>(a, s)
                                                                                                         : launch_rate_k<8>(a, s);
        if (st) return st;
    }
    return QCE_OK;
}

}  // namespace qce
