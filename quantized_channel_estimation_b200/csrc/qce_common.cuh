// Shared declarations of the qce_b200 library (internal; the public ABI is include/qce_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>

#include "qce_b200.h"

namespace qce {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launch_count;          // calls may come from several host threads (one per stream / device)
inline void count_launch(int n = 1) { g_launch_count.fetch_add(n, std::memory_order_relaxed); }

#define QCE_CUDA_TRY(expr)                                                                      \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            qce::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,    \
                           __LINE__);                                                           \
            return QCE_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define QCE_CHECK_LAUNCH(name)                                                                  \
    do {                                                                                        \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess) {                                                                \
            qce::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));            \
            return QCE_ERR_CUDA;                                                                \
        }                                                                                       \
        qce::count_launch();                                                                    \
    } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: one flag per (kernel instantiation, device)
struct PerDeviceOnce {
    bool done[64] = {};
    bool first(int dev) { if (dev < 0 || dev >= 64) return true; if (done[dev]) return false; done[dev] = true; return true; }
};
inline int current_device() { int d = 0; cudaGetDevice(&d); return d; }

// Grow-on-demand buffer: device memory, or page-locked host memory when `pinned`.  A plain struct: a copy aliases the buffer, and
// only free_buf releases it.
struct ScratchBuf {
    void* p = nullptr;
    size_t bytes = 0;
    bool pinned = false;
};

// Grows only, never shrinks: a larger need frees the buffer and allocates the new size (zeroed when zero_fill).  cudaFree
// synchronises the device, so a steady state of equal-sized calls must never get here.
inline qce_status grow(ScratchBuf& b, size_t bytes, bool zero_fill = false) {
    if (bytes <= b.bytes) return QCE_OK;
    if (b.p) QCE_CUDA_TRY(b.pinned ? cudaFreeHost(b.p) : cudaFree(b.p));
    b.p = nullptr; b.bytes = 0;
    QCE_CUDA_TRY(b.pinned ? cudaMallocHost(&b.p, bytes) : cudaMalloc(&b.p, bytes));
    if (zero_fill) QCE_CUDA_TRY(cudaMemset(b.p, 0, bytes));
    b.bytes = bytes;
    return QCE_OK;
}

inline void free_buf(ScratchBuf& b) {
    if (b.p) { if (b.pinned) cudaFreeHost(b.p); else cudaFree(b.p); }
    b.p = nullptr; b.bytes = 0;
}

struct QuantTables {            // device-resident quantiser tables
    int n_bits;
    int n_thr;                  // 2^b - 1
    const double* thr;          // device [n_thr]
    const double* labels;       // device [n_thr + 1]
};

}  // namespace qce

struct qce_quantizer {
    qce::QuantTables t;
    double* dev_buf;            // thr followed by labels
};

// Tensor-core parameter image of one model (see qce_dense_tc.cu)
struct TcParams {
    void* image = nullptr;      // packed FP16 hi/lo operand images, device
    size_t image_bytes = 0;
    void* image2 = nullptr;     // per-CTA half images of the SM-pair (cta_group::2) kernel
    size_t image2_bytes = 0;
    float* zoff = nullptr;      // [K][2*n_obs] whitened offsets (fp32)
    float* hoff = nullptr;      // [K][2*n_ant]
    float* zscale = nullptr;    // [K] power-of-two scale folded out of the Linv_k image
    float* hscale = nullptr;    // [K]
    void* logc2 = nullptr;      // [K] float2: logc_k as an FP32 (hi, lo) pair
    int* flags = nullptr;       // device scratch: [0] offsets non-zero, [1] some Linv_k not lower triangular
    bool has_offsets = false;
    bool triangular = false;
    bool ready = false;
    // pilots off the integer grid (data_scale = 0: Lloyd-Max labels, unquantised data): staged as FP16 (hi, lo) tile pairs of
    // r / eff_scale, three tensor passes
    bool split_a = false;
    double eff_scale = 0.0;     // data_scale, or 2^-8 when split_a
    // split path (n_obs or n_ant above 64): a whitening-only image and up to four LMMSE row-block images (n_ant = 256: four blocks
    // of 128 columns); the estimate runs as log-probability launch -> selection -> one launch per row block
    bool split = false;
    void* image_z = nullptr;
    void* image_h[4] = {nullptr, nullptr, nullptr, nullptr};
    int h_parts = 0;            // number of row-block launches
    int part_cols = 0;          // real columns (of the 2 n_ant) per row block
};

// host-buffer entry points: the staging sets (private streams, pinned slots) are pooled per device (qce_api.cu); every model carries an
// event recorded after its last parameter upload, which the staging streams wait on

struct qce_circ_model {
    int n1, n2, n_ant, n_comp, flags;
    int device = 0;
    cudaEvent_t params_ready = nullptr;
    double* inv_lambda_t = nullptr;   // [N][K]  1 / eigenvalues of C_r,k, transposed for coalesced access
    double* gain = nullptr;           // [K][N]  b_k c_k / lambda_k
    double* logc = nullptr;           // [K]
    bool params_set = false;
    // FP32 / tensor-core kernel (qce_circ_tc.cu): the two parameter matrices as FP16 (hi, lo) mma fragments
    void* tc_b1 = nullptr;
    void* tc_b2 = nullptr;
    void* tc_logc2 = nullptr;
    void* tc_ilbar = nullptr;         // [N] float: mean over the components of 1 / lambda
    void* tc_tw = nullptr;            // [256] float2 twiddles of the plain-circulant (one-dimensional) variant
    double tc_logc_max = 0.0;
    float tc_inv_s1 = 0.f, tc_inv_s2 = 0.f;
    bool tc_ready = false;
};

struct qce_mfa_model {
    int n_ant, latent, n_comp, flags;
    int device = 0;
    cudaEvent_t params_ready = nullptr;
    double* inv_delta = nullptr;      // [K][N]
    double* evec = nullptr;           // [K][N]
    double* D = nullptr;              // c128 [K][2M][N]
    double* Y = nullptr;              // c128 [K][N][2M]
    double* m_r = nullptr;            // c128 [K][N]
    double* mu = nullptr;             // c128 [K][N]
    double* logc = nullptr;           // [K]
    bool params_set = false;
};

// rate lower-bound accumulators (qce_rate.cu)
struct qce_rate_model {
    int n_ant = 0, n_pad = 0;         // N, and N rounded up to a multiple of 16
    int device = 0;
    double* buss = nullptr;           // c128 [N] diagonal of the Bussgang matrix
    void* frag = nullptr;             // [n_pad / 4][n_pad / 8][32] uint4: E (real embedding of C_q) as FP16 (hi, lo) mma fragments
    double inv_se = 1.0;              // 2^-s of the packed E
    bool params_set = false;
};

struct qce_model {
    int n_obs, n_ant, n_comp, flags;
    int device = 0;
    cudaEvent_t params_ready = nullptr;
    // fp64 parameter copies (device)
    double* Linv = nullptr;     // c128 [K][No][No]
    double* W = nullptr;        // c128 [K][N][No]
    double* zoff = nullptr;     // c128 [K][No]
    double* hoff = nullptr;     // c128 [K][N]
    double* logc = nullptr;     // f64  [K]
    double data_scale = 0.0;
    bool params_set = false;
    TcParams tc;
};

#ifdef __CUDACC__
namespace qce {
// ---- the quantiser's scalar arithmetic (modules/utils.py:189-203), shared by quantize_kernel and the complex128 re-evaluation path
// 1/np.sqrt(2) = 0x3FE6A09E667F3BCC (NOT sqrt(0.5) = ...BCD), SURVEY.md section 7 "bit-exact quantiser"
__device__ __forceinline__ double inv_sqrt2() { return __longlong_as_double(0x3FE6A09E667F3BCCLL); }

__device__ __forceinline__ double sign_np(double x) {   // np.sign: -1, 0, +1, NaN
    return (x > 0.0) ? 1.0 : ((x < 0.0) ? -1.0 : ((x == 0.0) ? 0.0 : x));
}

__device__ __forceinline__ int digitize(double x, const double* __restrict__ thr, int n_thr) {
    // np.digitize(x, thr) with right=False on ascending thr: #{thr <= x}; NaN sorts last.
    if (x != x) return n_thr;
    int lo = 0, hi = n_thr;                // first index with thr[idx] > x
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (thr[mid] <= x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// r = Q(y) for one complex sample (tables anywhere the pointer reaches: shared or global memory)
__device__ __forceinline__ double2 quantize_value(int n_bits, int n_thr, const double* __restrict__ thr, const double* __restrict__ lab,
                                                  const double2 y, uchar2* code_out) {
    double2 r;
    uchar2 code;
    if (n_bits == 1) {
        const double sr = sign_np(y.x), si = sign_np(y.y);
        code.x = (sr != sr) ? 3 : (unsigned char)((int)sr + 1);
        code.y = (si != si) ? 3 : (unsigned char)((int)si + 1);
        if (sr != sr || si != si) {        // numpy's complex product spreads a NaN to both parts
            r.x = r.y = __longlong_as_double(0x7FF8000000000000LL);
        } else {
            r.x = __dmul_rn(inv_sqrt2(), sr) + 0.0;  // + 0.0: -0 -> +0 like numpy's (c*a - 0*b)
            r.y = __dmul_rn(inv_sqrt2(), si) + 0.0;
        }
    } else {
        const int ir = digitize(y.x, thr, n_thr), ii = digitize(y.y, thr, n_thr);
        code.x = (unsigned char)ir;
        code.y = (unsigned char)ii;
        r.x = lab[ir];
        r.y = lab[ii];
    }
    if (code_out) *code_out = code;
    return r;
}

// Per-sample weights from weighted log-probabilities, in place (lp[k] -> w[k]); T = double, or float for the FP32 kernels.
// tie != null (FP32 kernels): *tie is set when the hard selection is too close to call with log-likelihoods that carry an error of
// up to ~tie_eps nats -- the deciding gap (maximum vs runner-up, last selected vs first left out) or a prefix sum vs rho -- so that
// the caller can hand the pilot to the complex128 kernel.
template <typename T>
__device__ inline void weights_from_logp(T* lp, int K, int mode, int n_top, double rho, int flags, bool* tie = nullptr, double tie_eps = 0.0) {
    double mx = lp[0], mx2 = -INFINITY;
    int amax = 0;
    bool close = false;
    for (int k = 1; k < K; ++k) {
        if (lp[k] > mx) { mx2 = mx; mx = lp[k]; amax = k; }
        else if ((double)lp[k] > mx2) mx2 = lp[k];
    }
    if (mode == QCE_MODE_TOP1) {
        // gmm:349 argmax of the weighted log-prob; mofa:359-366 argmax of exp(.) -> 0 when all underflow
        if (tie) *tie = !(mx - mx2 > tie_eps) || ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && fabs(mx + 745.1332) < 0.01);
        if ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && exp(mx) == 0.0) amax = 0;
        for (int k = 0; k < K; ++k) lp[k] = (k == amax) ? (T)1.0 : (T)0.0;
        return;
    }
    double sum = 0.0;
    for (int k = 0; k < K; ++k) sum += exp((double)lp[k] - mx);
    const double lse = mx + log(sum);               // scipy.special.logsumexp (gmm:652) / _log_sum (mofa:394-400)
    for (int k = 0; k < K; ++k) lp[k] = (T)exp((double)lp[k] - lse);
    if (tie) *tie = !(mx == mx);
    if (mode == QCE_MODE_ALL) return;
    // descending selection (np.argsort(p)[::-1], gmm:210 / :233); selected entries are marked by the sign bit
    const int limit = (mode == QCE_MODE_TOPN) ? (n_top < K ? n_top : K) : K;
    double cum = 0.0, last = -1.0;
    bool done = false;
    for (int it = 0; it <= limit; ++it) {
        int best = -1;
        double bv = -1.0;
        for (int k = 0; k < K; ++k)
            if (!signbit(lp[k]) && (double)lp[k] > bv) { bv = (double)lp[k]; best = k; }
        if (best < 0) break;
        if (done || it == limit) {                  // first candidate left out: a near-tie with the last selected one could swap them
            if (bv > last * (1.0 - tie_eps)) close = true;
            break;
        }
        lp[best] = (T)(-bv);
        cum += bv;
        last = bv;
        // searchsorted(cumsum, rho) + 1 (gmm:234): stop after the first prefix with cumsum >= rho
        if (mode == QCE_MODE_CUMPROB) {
            if (fabs(cum - rho) < tie_eps) close = true;
            if (cum >= rho) { if (!tie) break; done = true; }
        }
        if (!tie && it + 1 == limit) break;
    }
    if (tie && close) *tie = true;
    for (int k = 0; k < K; ++k) lp[k] = signbit(lp[k]) ? (T)((double)(-lp[k]) / cum) : (T)0.0;
}

}  // namespace qce
#endif

namespace qce {
// qce_quantize.cu
qce_status launch_quantize(const QuantTables* t, cudaStream_t s, const double* y, int64_t n_complex, double* r_out,
                           uint8_t* codes_out);
qce_status launch_observe_quantize(const QuantTables* t, cudaStream_t s, const void* h, int h_is_c64,
                                   const double* noise, double noise_scale, int64_t n_complex, double* y_out,
                                   double* r_out, uint8_t* codes_out);
qce_status launch_decode_codes(const QuantTables* t, cudaStream_t s, const uint8_t* codes, int64_t n_complex, double* r_out);
qce_status launch_c128_to_c64(cudaStream_t s, const double* in, int64_t n_complex, float* out);
// qce_dense_fp64.cu
qce_status launch_dense_fp64(const qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top,
                             double rho, double* h_est, double* logp_out, const double* h_true, double* acc);
qce_status launch_dense_fp64_raw(const qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top,
                                 double rho, double* h_est, double* logp_out, const void* h_true, int h_true_c64,
                                 double* acc);
// complex128 re-evaluation of a device-side list of rows (rows[0 .. *n_rows_dev)) of a batch: the pilots are read from r, or
// (r == null) observed + quantised on the fly from (obs_h, obs_noise) exactly like quantize_kernel; results are written to the
// listed rows of h_est / logp_out and added to acc
struct RowSource {
    const double* r = nullptr;          // c128 [B][n_obs] quantised pilots, or null
    const void* obs_h = nullptr;        // c64 / c128 [B][n_obs] channels (A = I)
    const double* obs_noise = nullptr;  // c128 [B][n_obs]
    double obs_noise_scale = 0.0;
    int obs_h_c64 = 0;
    QuantTables qt{};
};

// Pilot tiles of the dense tensor-core path (qce_dense_tc.cu), shared by all models
struct TileScratch {
    ScratchBuf img, bad;                   // zeroed on allocation: the last work unit reads up to 4 tiles past the batch
    ScratchBuf lp2;                        // [rows][K] float2 log-probabilities (modes other than fused 'all')
    ScratchBuf wts;                        // [rows][K] float weights
    ScratchBuf img2;                       // bucketed top-1: pilot tiles regrouped by selected component
    ScratchBuf bidx;                       // int32: top[rows] | perm[slots] | unit_comp[units] | cnt[K] off[K] cursor[K] n_units
    const qce_model* owner = nullptr;      // model whose pilots are currently formatted here
    int64_t rows = 0;
    // fix list: rows of the formatted batch that are re-evaluated by the complex128 kernel after the tensor-core launches
    // ([0] is the length, [1] counts the near-ties re-selected so far, the indices follow), and where their pilots come from
    ScratchBuf fix;
    RowSource src;
    // tie list of the chunk in flight ([0] = count, then chunk rows): hard selections too close to call in FP32, re-selected in
    // complex128 (tc_refine_kernel) before the combine launch
    ScratchBuf tie;
    ScratchBuf tmp_est;                    // pair mode: [chunk rows][2N] FP32 rows the (pilot, component) launches add into
    int* fix_list() const { return (int*)fix.p; }
    int* tie_list() const { return (int*)tie.p; }
};

// Every grow-on-demand buffer of the library, one entry per (device, stream) (qce_api.cu): calls on different streams may be in
// flight at once (host threads on streams of their own, the private streams of the host-buffer path), so no buffer is shared
// between streams.  An entry is used only by the calls that enqueue work on its stream; the store's mutex guards the map.
struct StreamScratch {
    TileScratch tc;
    ScratchBuf circ_fix;                   // circulant tensor-core fix list: [0] count, [1] unused, then the rows
    ScratchBuf pipe_r;                     // qce_pipeline, complex128 path: quantised pilots of one chunk
    ScratchBuf host_in, host_out;          // device slot of a host-buffer call (private staging streams only)
    ScratchBuf host_mid_in, host_mid_out;  // its device-only intermediates (decoded pilots, complex128 estimates)
    const int* last_fix = nullptr;         // tc.fix or circ_fix, whichever the latest tensor-core call used: qce_last_fix_count
};
StreamScratch* scratch_for(cudaStream_t s);        // creates the stream's entry if it has none
StreamScratch* scratch_find(cudaStream_t s);       // null if it has none
void scratch_release(cudaStream_t s);              // frees the entry's buffers and erases it (the stream is about to be destroyed)

qce_status launch_dense_fp64_rows(const qce_model* m, cudaStream_t s, const RowSource& src, const int* rows, const int* n_rows_dev,
                                  int64_t max_rows, int mode, int n_top, double rho, double* h_est, double* logp_out,
                                  const void* h_true, int h_true_c64, double* acc);
// qce_dense_tc.cu
qce_status tc_pack_params(qce_model* m, cudaStream_t s);
void tc_free(qce_model* m);
qce_status launch_dense_tc(qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top,
                           double rho, double* h_est, double* logp_out, const void* h_true, int h_true_c64,
                           double* acc);
qce_status tc_format(qce_model* m, cudaStream_t s, const double* r, int64_t B);
qce_status tc_estimate_formatted(qce_model* m, cudaStream_t s, int64_t B, double* h_est, const void* h_true, int h_true_c64,
                                 double* acc);
qce_status launch_pipeline_tc(qce_model* m, const QuantTables* qt, cudaStream_t s, const void* h, int h_is_c64,
                              const double* noise, double noise_scale, int64_t B, int mode, int n_top, double rho, double* h_est,
                              double* acc);
bool tc_supported(const qce_model* m, int mode);
const char* tc_unsupported_reason(const qce_model* m);      // "" or ": <why>", appended to the error message
// qce_mfa.cu
qce_status launch_mfa(const qce_mfa_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                      double* h_est, double* logp_out, const double* h_true, double* acc);
// qce_circ_tc.cu
bool circ_tc_shape_ok(const qce_circ_model* m);
qce_status circ_tc_pack(qce_circ_model* m, cudaStream_t s);
void circ_tc_free(qce_circ_model* m);
qce_status launch_circ_tc(const qce_circ_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                          double* h_est, double* logp_out, const double* h_true, double* acc);
// qce_circ.cu
qce_status launch_circ(const qce_circ_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                       double* h_est, double* logp_out, const double* h_true, double* acc);
qce_status launch_circ_rows(const qce_circ_model* m, cudaStream_t s, const double* r, const int* rows, const int* n_rows_dev, int64_t max_rows,
                            int mode, int n_top, double rho, double* h_est, const double* h_true, double* acc);
// qce_rate.cu
qce_status rate_pack(qce_rate_model* m, cudaStream_t s, const double* cq);
qce_status launch_rate(const qce_rate_model* m, cudaStream_t s, const double* h_est, const void* h_true, int h_true_c64, int64_t B,
                       double* acc);
}  // namespace qce
