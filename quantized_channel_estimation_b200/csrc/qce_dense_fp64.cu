// Complex128 SIMT estimate kernel: the validation-grade path (QCE_PREC_FP64).
//
// Per sample it evaluates exactly what Gmm_nbit.estimate_from_y (modules/gmm_cplx_bussgang.py:196-243)
// and Mofa.estimate_from_y (modules/mofa_cplx_bussgang.py:124-159) evaluate after
// _prepare_for_prediction, in IEEE double:
//   phase 1   l_k = logc_k - |Linv_k r - zoff_k|^2                 (gmm:380-386, 413-417, 435)
//   phase 1.5 weights from l per combination mode                   (gmm:197-242 / mofa:125-158)
//   phase 2   h = sum_k w_k (W_k r + hoff_k)                        (gmm:331-332 / mofa:215-216)
// One CTA owns a tile of TS samples; the tile (transposed) and the [TS][K] log-probabilities live in
// shared memory, so per-component estimates never touch HBM.  Parameters stream from L2.
// Any n_obs / n_ant / K that fits shared memory is supported.
#include "qce_common.cuh"

namespace qce {

struct Fp64Args {
    int No, N, K;
    int64_t B;
    const double2* Linv;
    const double2* W;
    const double2* zoff;
    const double2* hoff;
    const double* logc;
    const double2* r;
    double2* h_est;
    double* logp_out;
    const void* h_true;
    int h_true_c64;
    double* acc;
    int mode, n_top, flags;
    double rho;
    // re-evaluation of listed rows (null: the rows are 0 .. B-1 in order): tile entry i is row rows[i], i < *n_rows_dev.  A listed
    // row >= B (the list of a formatted image longer than the batch, qce_estimate_formatted) is skipped: not staged, written or counted
    const int* rows;
    const int* n_rows_dev;
    // r == null: the pilots are observed + quantised on the fly (A = I), bit-exact to quantize_kernel
    const void* obs_h;
    const double2* obs_noise;
    double obs_noise_scale;
    int obs_h_c64;
    QuantTables qt;
};

__device__ __forceinline__ void cfma(double2& acc, const double2 a, const double2 b) {
    acc.x = fma(a.x, b.x, acc.x);
    acc.x = fma(-a.y, b.y, acc.x);
    acc.y = fma(a.x, b.y, acc.y);
    acc.y = fma(a.y, b.x, acc.y);
}

template <int TS>
__global__ void __launch_bounds__(256) dense_fp64_kernel(Fp64Args a) {
    constexpr int SP = TS / 2;          // sample pairs
    constexpr int RG = 256 / SP;        // row groups
    constexpr int RM = 4;               // rows per thread per chunk in phase 2
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* rT = reinterpret_cast<double2*>(smem_raw);                       // [No][TS]
    double* lp = reinterpret_cast<double*>(rT + (size_t)a.No * TS);           // [TS][K]
    double* part = lp + (size_t)TS * a.K;                                      // [8][TS]
    __shared__ double red[3];
    __shared__ int64_t s_row[TS];       // batch row of every tile entry
    __shared__ bool s_ok[TS];           // the entry is a row of the batch (< B)

    const int t = threadIdx.x;
    const int sp = t % SP, rg = t / SP;
    const int warp = t >> 5;
    const int No = a.No, N = a.N, K = a.K;
    const int64_t n_rows = a.n_rows_dev ? (int64_t)__ldg(a.n_rows_dev) : a.B;
    for (int64_t base = (int64_t)blockIdx.x * TS; base < n_rows; base += (int64_t)gridDim.x * TS) {
    const int nvalid = (int)((n_rows - base) < TS ? (n_rows - base) : TS);
    bool ok = false;
    if (t < TS) {
        const int64_t row = (t < nvalid) ? (a.rows ? (int64_t)a.rows[base + t] : base + t) : 0;
        ok = t < nvalid && row >= 0 && row < a.B;
        s_row[t] = ok ? row : 0;
        s_ok[t] = ok;
    }
    if (t < 3) red[t] = 0.0;
    const int n_ok = __syncthreads_count(ok);      // rows this tile writes and counts

    // stage the tile transposed: rT[j][s]
    for (int idx = t; idx < TS * No; idx += 256) {
        int s = idx / No, j = idx % No;
        double2 v = make_double2(0.0, 0.0);
        if (s_ok[s]) {
            const int64_t e = s_row[s] * No + j;
            if (a.r) {
                v = a.r[e];
            } else {      // get_observation_nbit with A = I (utils.py:241-251): two roundings, then the quantiser
                double2 h;
                if (a.obs_h_c64) { const float2 hf = reinterpret_cast<const float2*>(a.obs_h)[e]; h = make_double2((double)hf.x, (double)hf.y); }
                else h = reinterpret_cast<const double2*>(a.obs_h)[e];
                const double2 w = a.obs_noise[e];
                const double2 y = make_double2(__dadd_rn(h.x, __dmul_rn(a.obs_noise_scale, w.x)), __dadd_rn(h.y, __dmul_rn(a.obs_noise_scale, w.y)));
                v = quantize_value(a.qt.n_bits, a.qt.n_thr, a.qt.thr, a.qt.labels, y, nullptr);
            }
        }
        rT[(size_t)j * TS + s] = v;
    }
    __syncthreads();

    // ---- phase 1: weighted log-probabilities
    for (int k = 0; k < K; ++k) {
        double q0 = 0.0, q1 = 0.0;
        for (int i = rg; i < No; i += RG) {
            const double2 zo = a.zoff[(size_t)k * No + i];
            double2 z0 = make_double2(-zo.x, -zo.y), z1 = z0;
            const double2* __restrict__ Lrow = a.Linv + ((size_t)k * No + i) * No;
            #pragma unroll 4
            for (int j = 0; j < No; ++j) {
                const double2 l = __ldg(Lrow + j);
                const double2 r0 = rT[(size_t)j * TS + 2 * sp];
                const double2 r1 = rT[(size_t)j * TS + 2 * sp + 1];
                cfma(z0, l, r0);
                cfma(z1, l, r1);
            }
            q0 += z0.x * z0.x + z0.y * z0.y;
            q1 += z1.x * z1.x + z1.y * z1.y;
        }
        // deterministic reduction over row groups: shuffles inside the warp, fixed order across warps
        #pragma unroll
        for (int off = SP; off < 32; off <<= 1) {
            q0 += __shfl_xor_sync(0xffffffffu, q0, off);
            q1 += __shfl_xor_sync(0xffffffffu, q1, off);
        }
        if ((t & 31) < SP) {
            part[warp * TS + 2 * sp] = q0;
            part[warp * TS + 2 * sp + 1] = q1;
        }
        __syncthreads();
        if (t < TS) {
            double q = 0.0;
            #pragma unroll
            for (int w = 0; w < 8; ++w) q += part[w * TS + t];
            lp[(size_t)t * K + k] = a.logc[k] - q;
        }
        __syncthreads();
    }

    // ---- phase 1.5: per-sample weights
    if (a.logp_out) {
        for (int idx = t; idx < nvalid * K; idx += 256)
            if (s_ok[idx / K]) a.logp_out[s_row[idx / K] * K + (idx % K)] = lp[idx];
        __syncthreads();
    }
    if (t < TS) weights_from_logp(lp + (size_t)t * K, K, a.mode, a.n_top, a.rho, a.flags);
    __syncthreads();

    // ---- phase 2: weighted LMMSE combination
    double err = 0.0, pw = 0.0;
    const bool want = (a.h_est != nullptr) || (a.acc != nullptr);
    if (want) {
        for (int rb = 0; rb < N; rb += RG * RM) {
            double2 acc0[RM], acc1[RM];
            #pragma unroll
            for (int m = 0; m < RM; ++m) acc0[m] = acc1[m] = make_double2(0.0, 0.0);
            for (int k = 0; k < K; ++k) {
                const double w0 = lp[(size_t)(2 * sp) * K + k], w1 = lp[(size_t)(2 * sp + 1) * K + k];
                if (w0 == 0.0 && w1 == 0.0) continue;
                #pragma unroll
                for (int m = 0; m < RM; ++m) {
                    const int i = rb + rg + RG * m;
                    if (i >= N) break;
                    const double2 ho = a.hoff[(size_t)k * N + i];
                    double2 e0 = ho, e1 = ho;
                    const double2* __restrict__ Wrow = a.W + ((size_t)k * N + i) * No;
                    #pragma unroll 4
                    for (int j = 0; j < No; ++j) {
                        const double2 w = __ldg(Wrow + j);
                        cfma(e0, w, rT[(size_t)j * TS + 2 * sp]);
                        cfma(e1, w, rT[(size_t)j * TS + 2 * sp + 1]);
                    }
                    acc0[m].x += w0 * e0.x; acc0[m].y += w0 * e0.y;     // h_est += p_k * h_k  (gmm:224-228)
                    acc1[m].x += w1 * e1.x; acc1[m].y += w1 * e1.y;
                }
            }
            #pragma unroll
            for (int m = 0; m < RM; ++m) {
                const int i = rb + rg + RG * m;
                if (i >= N) break;
                #pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int s = 2 * sp + u;
                    if (!s_ok[s]) continue;
                    const double2 v = u ? acc1[m] : acc0[m];
                    const int64_t o = s_row[s] * N + i;
                    if (a.h_est) a.h_est[o] = v;
                    if (a.acc && a.h_true) {
                        double2 h;
                        if (a.h_true_c64) {
                            float2 hf = reinterpret_cast<const float2*>(a.h_true)[o];
                            h = make_double2((double)hf.x, (double)hf.y);
                        } else {
                            h = reinterpret_cast<const double2*>(a.h_true)[o];
                        }
                        const double dx = v.x - h.x, dy = v.y - h.y;
                        err += dx * dx + dy * dy;
                        pw += h.x * h.x + h.y * h.y;
                    }
                }
            }
        }
    }
    if (a.acc) {
        #pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            err += __shfl_xor_sync(0xffffffffu, err, off);
            pw += __shfl_xor_sync(0xffffffffu, pw, off);
        }
        if ((t & 31) == 0) { atomicAdd(&red[0], err); atomicAdd(&red[1], pw); }
        __syncthreads();
        if (t == 0) {
            atomicAdd(a.acc + 0, red[0]);
            atomicAdd(a.acc + 1, red[1]);
            atomicAdd(a.acc + 2, (double)n_ok);
        }
    }
    __syncthreads();      // red[], s_row[], the tile and lp are rewritten by the next tile of this CTA
    }
}

template <int TS>
static qce_status launch_ts(const Fp64Args& a, cudaStream_t s, size_t smem, int64_t grid_cap = 0) {
    static PerDeviceOnce once;
    if (once.first(current_device()))
        QCE_CUDA_TRY(cudaFuncSetAttribute(dense_fp64_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    int64_t grid = (a.B + TS - 1) / TS;
    if (grid_cap > 0 && grid > grid_cap) grid = grid_cap;
    dense_fp64_kernel<TS><<<(unsigned)grid, 256, smem, s>>>(a);
    QCE_CHECK_LAUNCH("dense_fp64_kernel");
    return QCE_OK;
}

qce_status launch_dense_fp64_raw(const qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top,
                                 double rho, double* h_est, double* logp_out, const void* h_true, int h_true_c64,
                                 double* acc) {
    if (B == 0) return QCE_OK;
    Fp64Args a;
    a.No = m->n_obs; a.N = m->n_ant; a.K = m->n_comp; a.B = B;
    a.Linv = (const double2*)m->Linv; a.W = (const double2*)m->W;
    a.zoff = (const double2*)m->zoff; a.hoff = (const double2*)m->hoff; a.logc = m->logc;
    a.r = (const double2*)r; a.h_est = (double2*)h_est; a.logp_out = logp_out;
    a.h_true = h_true; a.h_true_c64 = h_true_c64; a.acc = acc;
    a.mode = mode; a.n_top = n_top; a.flags = m->flags; a.rho = rho;
    a.rows = nullptr; a.n_rows_dev = nullptr; a.obs_h = nullptr; a.obs_noise = nullptr; a.obs_noise_scale = 0.0; a.obs_h_c64 = 0; a.qt = QuantTables{};
    auto need = [&](int ts) {
        return (size_t)a.No * ts * sizeof(double2) + (size_t)ts * a.K * sizeof(double) + (size_t)8 * ts * sizeof(double);
    };
    const size_t cap = 220 * 1024;
    if (B > (int64_t)2147483647 * 8) { set_error("batch too large for one launch"); return QCE_ERR_INVALID; }
    if (need(32) <= cap && B >= 32 * 148) return launch_ts<32>(a, s, need(32));
    if (need(16) <= cap && B >= 16 * 64) return launch_ts<16>(a, s, need(16));
    if (need(8) <= cap) return launch_ts<8>(a, s, need(8));
    set_error("fp64 kernel: n_obs=%d, K=%d do not fit shared memory", a.No, a.K);
    return QCE_ERR_UNSUPPORTED;
}

// The listed rows are few (near-ties of a hard selection, pilots off the tensor-core grid): small tiles for parallelism, and a grid
// that does not depend on the (device-side) length of the list -- CTAs without a tile exit at once, long lists are walked grid-stride.
qce_status launch_dense_fp64_rows(const qce_model* m, cudaStream_t s, const RowSource& src, const int* rows, const int* n_rows_dev,
                                  int64_t max_rows, int mode, int n_top, double rho, double* h_est, double* logp_out,
                                  const void* h_true, int h_true_c64, double* acc) {
    if (max_rows == 0) return QCE_OK;
    Fp64Args a;
    a.No = m->n_obs; a.N = m->n_ant; a.K = m->n_comp; a.B = max_rows;
    a.Linv = (const double2*)m->Linv; a.W = (const double2*)m->W;
    a.zoff = (const double2*)m->zoff; a.hoff = (const double2*)m->hoff; a.logc = m->logc;
    a.r = (const double2*)src.r; a.h_est = (double2*)h_est; a.logp_out = logp_out;
    a.h_true = h_true; a.h_true_c64 = h_true_c64; a.acc = acc;
    a.mode = mode; a.n_top = n_top; a.flags = m->flags; a.rho = rho;
    a.rows = rows; a.n_rows_dev = n_rows_dev;
    a.obs_h = src.obs_h; a.obs_noise = (const double2*)src.obs_noise; a.obs_noise_scale = src.obs_noise_scale; a.obs_h_c64 = src.obs_h_c64; a.qt = src.qt;
    if (!a.r && !(a.obs_h && a.obs_noise)) { set_error("re-evaluation of flagged rows: the source pilots are not available"); return QCE_ERR_INVALID; }
    const size_t need = (size_t)a.No * 8 * sizeof(double2) + (size_t)8 * a.K * sizeof(double) + (size_t)8 * 8 * sizeof(double);
    if (need > (size_t)220 * 1024) { set_error("fp64 kernel: n_obs=%d, K=%d do not fit shared memory", a.No, a.K); return QCE_ERR_UNSUPPORTED; }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, current_device());
    return launch_ts<8>(a, s, need, 2 * (int64_t)sms);
}

qce_status launch_dense_fp64(const qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top,
                             double rho, double* h_est, double* logp_out, const double* h_true, double* acc) {
    return launch_dense_fp64_raw(m, s, r, B, mode, n_top, rho, h_est, logp_out, h_true, 0, acc);
}

}  // namespace qce
