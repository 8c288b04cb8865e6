/*
 * qce_b200.h -- C ABI of the B200-native Bussgang-GMM / Bussgang-MFA inference path.
 *
 * The reference (benediktfesl/Quantized_Channel_Estimation) is pure Python and has no FFI of
 * its own; its boundary for this path is the Python method surface
 *     Gmm_nbit.estimate_from_y          modules/gmm_cplx_bussgang.py:166-243
 *     Mofa.estimate_from_y              modules/mofa_cplx_bussgang.py:117-159
 *     utils.quant                       modules/utils.py:189-203
 *     utils.get_observation_nbit        modules/utils.py:241-251
 * Each entry point below names the reference code whose per-sample arithmetic it replaces.
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; complex arrays are interleaved (re, im) doubles ("c128") or floats ("c64"),
 *     row-major, exactly numpy's / torch's memory layout;
 *   - "dev" pointers are CUDA device pointers owned by the caller, "host" pointers are host memory;
 *     device arrays need the alignment of their element type (16 bytes for c128, 8 for c64); estimate and
 *     true-channel arrays that are 32-byte aligned (every cudaMalloc / torch allocation is) are moved with
 *     256-bit accesses by the tensor-core path, others with 128-bit ones -- same results;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all device work is
 *     enqueued on it and the call returns without synchronising unless stated otherwise;
 *   - every function returns QCE_OK (0) or a negative qce_status; qce_last_error_string() gives
 *     the message of the last failure on the calling thread.  Nothing throws, nothing falls back
 *     to the CPU.
 */
#ifndef QCE_B200_H
#define QCE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QCE_ABI_VERSION 1

typedef int qce_status;
enum {
    QCE_OK = 0,
    QCE_ERR_INVALID = -1,      /* bad argument (shape, mode, null pointer)                          */
    QCE_ERR_CUDA = -2,         /* a CUDA runtime call or kernel launch failed                       */
    QCE_ERR_UNSUPPORTED = -3,  /* shape / mode not supported by the requested kernel                */
    QCE_ERR_NO_DEVICE = -4     /* no sm_100 device                                                  */
};

/* combination modes of estimate_from_y's `n_summands_or_proba` (gmm:197-242, mofa:125-158) */
enum {
    QCE_MODE_ALL = 0,      /* 'all'   : sum_k p_k h_k (not renormalised)                             */
    QCE_MODE_TOP1 = 1,     /* int 1   : hard decision argmax_k                                       */
    QCE_MODE_TOPN = 2,     /* int n>1 : n largest p_k, renormalised                                  */
    QCE_MODE_CUMPROB = 3   /* float   : smallest descending prefix with cumsum >= rho, renormalised  */
};

/* arithmetic of the estimate kernel */
enum {
    QCE_PREC_FP64 = 0,     /* complex128 SIMT kernel (validation / arbitrary shapes)                  */
    QCE_PREC_TC = 1        /* tcgen05 tensor-core kernel, FP16 hi/lo split operands, FP32 accumulate  */
};

/* flags for qce_model_create */
enum {
    QCE_FLAG_TOP1_EXP_ARGMAX = 1  /* Mofa.predict_proba_max quirk: argmax of exp(log p) (mofa:359-366):
                                     if every exp underflows the label is 0                          */
};

typedef struct qce_model qce_model;
typedef struct qce_quantizer qce_quantizer;
typedef struct qce_circ_model qce_circ_model;
typedef struct qce_mfa_model qce_mfa_model;

int qce_abi_version(void);
const char* qce_last_error_string(void);
/* number of CUDA kernels this library has launched so far in this process (bench.py's gpu_launches) */
int64_t qce_launch_count(void);
/* 1 if a CUDA device of compute capability 10.x is visible */
int qce_device_ok(void);
/* Rows of the most recent QCE_PREC_TC estimate enqueued on `stream` (current device) that the tensor-core path handed to the
 * complex128 kernel: pilots off the quantiser grid and hard selections (top-1 / top-n / cumulative) whose deciding log-likelihood
 * gap is below what FP32 accumulation resolves.  Synchronises the stream.  -1 if no such call has been made on the stream. */
int64_t qce_last_fix_count(void* stream);

/* ---- quantiser (modules/utils.py:189-203; tables from utils.py:531-590) ----------------------- */

/* n_bits == 1: thresholds/labels ignored (may be NULL).  Otherwise thresholds_host[2^b-1] ascending,
 * labels_host[2^b].  The tables are copied to the device here, once. */
qce_status qce_quantizer_create(int n_bits, const double* thresholds_host, const double* labels_host,
                                qce_quantizer** out);
void qce_quantizer_destroy(qce_quantizer* q);

/* r = Q(y) per real dimension, bit-exact to utils.quant:
 *   1 bit : 1/sqrt(2) * (sign(re) + j sign(im))   (sign(+-0) = 0, sign(NaN) = NaN)
 *   b bit : labels[#{thresholds <= x}]            (np.digitize right=False; NaN -> last bin)
 * y_dev: c128 [n_complex].  r_out_dev (c128 [n_complex]) and codes_out_dev (uint8 [n_complex][2], the
 * level index; 1 bit: 0 neg / 1 zero / 2 pos / 3 NaN) may each be NULL. */
qce_status qce_quantize(const qce_quantizer* q, void* stream, const void* y_dev, int64_t n_complex,
                        void* r_out_dev, uint8_t* codes_out_dev);

/* get_observation_nbit with A = I (utils.py:241-251): y = h + noise_scale * noise (two roundings, no
 * FMA), then quantise.  h_dev is c64 (h_is_c64 = 1, SCMMulti's dtype) or c128; noise_dev c128.
 * q == NULL means n_bits = inf (only y is produced).  y_out_dev / r_out_dev / codes_out_dev may be NULL. */
qce_status qce_observe_quantize(const qce_quantizer* q, void* stream, const void* h_dev, int h_is_c64,
                                const void* noise_dev, double noise_scale, int64_t n_complex,
                                void* y_out_dev, void* r_out_dev, uint8_t* codes_out_dev);

/* ---- per-SNR model: host-precomputed component parameters ------------------------------------- */

/* n_obs = rows of the pilot matrix A (length of r), n_ant = channel length N, n_comp = K. */
qce_status qce_model_create(int n_obs, int n_ant, int n_comp, int flags, qce_model** out);
void qce_model_destroy(qce_model* m);

/* Parameters of one (snr, n_bits, quantiser) setting -- the quantities Gmm_nbit._prepare_for_prediction
 * (gmm:246-328) / Mofa._prepare_for_prediction (mofa:162-212) derive, folded so that per sample
 *     z_k   = Linv_k r - zoff_k                 (whitened residual,   gmm:413-417)
 *     l_k   = logc_k - |z_k|^2                  (weighted log-lik.,   gmm:380-386, :435 / mofa:346-381)
 *     h_k   = W_k r + hoff_k                    (component LMMSE,     gmm:331-332 / mofa:215-216)
 * with Linv_k = L_k^-1 (C_r,k = L_k L_k^H), zoff_k = Linv_k m_r,k, W_k = C_h,k A_eff,k^H C_r,k^-1,
 * hoff_k = mu_k - W_k m_r,k, logc_k = ln w_k - n_obs ln(pi) - ln|C_r,k|.
 * All arrays are device c128 / f64, row-major: Linv [K][n_obs][n_obs], W [K][n_ant][n_obs],
 * zoff [K][n_obs], hoff [K][n_ant], logc [K].  The model copies / repacks them (caller may free).
 * data_scale > 0 declares that every real and imaginary part of every r the caller will pass is an
 * integer multiple m * data_scale with |m| <= 2048 (true for 1-bit and uniform quantisers); the
 * tensor-core kernel then needs two instead of three FP16 passes.  Pass 0 for arbitrary data. */
qce_status qce_model_set_params(qce_model* m, void* stream, const double* Linv_dev, const double* W_dev,
                                const double* zoff_dev, const double* hoff_dev, const double* logc_dev,
                                double data_scale);

/* ---- the hot path ------------------------------------------------------------------------------ */

/* estimate_from_y after _prepare_for_prediction (gmm:196-243 / mofa:124-159) for a batch.
 *   r_dev      c128 [B][n_obs]  quantised pilots
 *   h_est_dev  c128 [B][n_ant]  output (may be NULL when only the accumulators are wanted)
 *   logp_out_dev  f64 [B][K] weighted log-probabilities l_k (may be NULL)
 *   h_true_dev c128 [B][n_ant] and acc_dev f64[3] (may both be NULL): acc += { sum|h_est-h|^2, sum|h|^2, B }
 *   mode / n_top / rho: see QCE_MODE_*; precision: QCE_PREC_* */
qce_status qce_estimate(qce_model* m, void* stream, const void* r_dev, int64_t B, int mode, int n_top,
                        double rho, int precision, void* h_est_dev, double* logp_out_dev,
                        const void* h_true_dev, double* acc_dev);

/* Fused pipeline on device-resident channels: observe (A = I) -> quantise -> estimate -> NMSE
 * accumulators, i.e. one Monte-Carlo step of Bussgang_GMM.py:284-289 for one SNR.
 * h_dev c64/c128 [B][N], noise_dev c128 [B][N]; h_est_dev may be NULL; acc_dev f64[3] may be NULL. */
qce_status qce_pipeline(qce_model* m, const qce_quantizer* q, void* stream, const void* h_dev, int h_is_c64,
                        const void* noise_dev, double noise_scale, int64_t B, int mode, int n_top, double rho,
                        int precision, void* h_est_dev, double* acc_dev);

/* Two-step form of the tensor-core path (QCE_PREC_TC, QCE_MODE_ALL).  qce_format_pilots converts r (c128 [B][n_obs],
 * values on the quantiser grid declared by data_scale) into the FP16 tile image the estimate kernel stages with bulk
 * copies, and keeps it in the library's per-stream scratch.  qce_estimate_formatted then runs the estimate kernel alone on the
 * first B pilots of that image (same model, same stream); outputs as in qce_estimate.  bench.py uses the pair to time the dominant kernel in
 * isolation; qce_estimate with QCE_PREC_TC is exactly format + estimate. */
qce_status qce_format_pilots(qce_model* m, void* stream, const void* r_dev, int64_t B);
qce_status qce_estimate_formatted(qce_model* m, void* stream, int64_t B, void* h_est_dev, const void* h_true_dev,
                                  double* acc_dev);

/* ---- circulant / block-circulant covariances (new algorithm; the reference only has the dense path, into which it
 * converts every covariance type, gmm:110-136).  C_h,k = F^H diag(c_k) F with F = F_n1 (x) F_n2 unitary (n1 = 1: plain
 * circulant), A = I, zero means.  Host-precomputed per (snr, bits): inv_lambda_t [N][K] = 1 / eigenvalues of C_r,k
 * (transposed), gain [K][N] = b_k c_k / lambda_k, logc [K] = ln w_k - N ln(pi) - sum_i ln lambda_k,i; all device f64.
 * qce_circ_estimate has the semantics of qce_estimate (complex128 arithmetic, all four modes). */
qce_status qce_circ_model_create(int n1, int n2, int n_comp, int flags, qce_circ_model** out);
void qce_circ_model_destroy(qce_circ_model* m);
qce_status qce_circ_model_set_params(qce_circ_model* m, void* stream, const double* inv_lambda_t_dev, const double* gain_dev,
                                     const double* logc_dev);
qce_status qce_circ_estimate(qce_circ_model* m, void* stream, const void* r_dev, int64_t B, int mode, int n_top, double rho,
                             void* h_est_dev, double* logp_out_dev, const void* h_true_dev, double* acc_dev);
/* The same with a precision selector.  QCE_PREC_FP64: the complex128 kernel above.  QCE_PREC_TC: FP32 radix-4 FFTs and
 * split-FP16 tensor-core contractions (16 x 16 blocks or plain circulant of length 256, K = 64 or 128; any real-valued pilots; estimates within ~1e-6 of the
 * complex128 path), QCE_ERR_UNSUPPORTED for other shapes. */
qce_status qce_circ_estimate_prec(qce_circ_model* m, void* stream, const void* r_dev, int64_t B, int mode, int n_top, double rho,
                                  int precision, void* h_est_dev, double* logp_out_dev, const void* h_true_dev, double* acc_dev);

/* ---- mixture of factor analysers in Woodbury form (A = I, n_bits > 1 or infinite resolution): C_r,k = U U^H + Delta_k is
 * never formed (the reference builds it densely and pinvh's it, mofa:199-207).  Host-precomputed per (snr, bits), all
 * device arrays: inv_delta [K][N] f64 = 1/Delta; evec [K][N] f64 = psi b / Delta; D c128 [K][2M][N] (rows 0..M-1: V1,
 * rows M..2M-1: T = L_S^-1 U^H Delta^-1); Y c128 [K][N][2M] = [Lambda | -(e .* U) L_S^-H]; m_r c128 [K][N];
 * mu c128 [K][N]; logc [K] = ln amps_k - N ln(pi) - sum ln Delta - ln det S.  Per pilot:
 *   x = r - m_r,k;  l_k = logc_k - (sum_i |x_i|^2 inv_delta_i - |T x|^2);  h_k = mu_k + e .* x + Y [V1 x; T x].
 * qce_mfa_estimate has the semantics of qce_estimate (complex128 arithmetic, all four modes, flags as qce_model_create). */
qce_status qce_mfa_model_create(int n_ant, int latent_dim, int n_comp, int flags, qce_mfa_model** out);
void qce_mfa_model_destroy(qce_mfa_model* m);
qce_status qce_mfa_model_set_params(qce_mfa_model* m, void* stream, const double* inv_delta_dev, const double* evec_dev,
                                    const double* D_dev, const double* Y_dev, const double* m_r_dev, const double* mu_dev,
                                    const double* logc_dev);
qce_status qce_mfa_estimate(qce_mfa_model* m, void* stream, const void* r_dev, int64_t B, int mode, int n_top, double rho,
                            void* h_est_dev, double* logp_out_dev, const void* h_true_dev, double* acc_dev);

/* ---- achievable-rate lower bound (Bussgang_GMM.py:291-309, Bussgang_MFA.py:154-172) in summable form.  Per estimate row
 * g = h_est / max(|h_est|^2, 0.1), inner = g^H B h with B the diagonal Bussgang matrix of the global model, q = Re g^H C_q g.
 * The bound is log2(1 + |m|^2 / (v + Q / n)) with m = S1 / n, v = S2 / n - |m|^2, where S1 = sum inner, S2 = sum |inner|^2,
 * Q = sum q: five sums that add across batches and ranks like the NMSE accumulators.  inner in FP64, q on the tensor cores
 * (split FP16 operands, FP32 accumulation).  1 <= n_ant <= 256 (QCE_ERR_UNSUPPORTED above).  Calls from a thread whose current
 * device is not the model's return QCE_ERR_INVALID. */
typedef struct qce_rate_model qce_rate_model;
qce_status qce_rate_model_create(int n_ant, qce_rate_model** out);
void       qce_rate_model_destroy(qce_rate_model* m);
/* buss_diag_dev c128 [N] (the diagonal of B), cq_dev c128 [N][N]; the model symmetrises, scales, splits and packs a copy
 * (synchronises the stream once to read the range of C_q) */
qce_status qce_rate_model_set_params(qce_rate_model* m, void* stream, const double* buss_diag_dev, const double* cq_dev);
/* acc_dev f64[5] += { sum Re inner, sum Im inner, sum |inner|^2, sum Re g^H C_q g, B }; h_est_dev c128 [B][N]; h_true_dev
 * c64 (h_true_c64 = 1) or c128 [B][N].  B = 0 enqueues nothing. */
qce_status qce_rate_accumulate(qce_rate_model* m, void* stream, const void* h_est_dev, const void* h_true_dev,
                               int h_true_c64, int64_t B, double* acc_dev);

/* Host-buffer form of qce_estimate: r_host c128 [B][n_obs] -> h_est_host c128 [B][n_ant].  Copies are chunked (32 MiB, four chunks
 * in flight) and overlapped with the kernels on private streams.  The streams and staging slots come from a per-device pool: a call
 * takes a free set (or creates one) and returns it at the end, so concurrent calls -- on one model or several -- never share buffers
 * and never wait for each other; the private streams wait on an event recorded after the model's last parameter upload -- no global
 * lock, no device-wide synchronisation.  Page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are copied directly, pageable
 * ones through the pinned slots.  Returns after the last chunk has landed in h_est_host (synchronous).  The calling thread's current
 * device must be the one the model was created on (QCE_ERR_INVALID otherwise). */
qce_status qce_estimate_host(qce_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho,
                             int precision, void* h_est_host);
/* Frees the pooled staging sets (pinned host memory, device slots, streams) that are not in use by a call in flight. */
void qce_host_staging_release(void);
/* Compact transfer formats of the same call (the estimate itself is unchanged: the codes are expanded to the quantised pilots on the
 * device, the estimates narrowed there).  codes_host: uint8 [B][n_obs][2], per real dimension the level index that qce_quantize /
 * qce_observe_quantize write (1 bit: 0 neg / 1 zero / 2 pos / 3 NaN; b bit: 0 .. 2^b - 1); q supplies the labels.  out_c64 != 0:
 * h_est_host is complex64 [B][n_ant] (the tensor-core estimates carry FP32 accuracy anyway), else complex128.  At n_obs = n_ant =
 * 64: 128 B in + 512 B out per pilot instead of 1 KiB + 1 KiB. */
qce_status qce_estimate_host_codes(qce_model* m, const qce_quantizer* q, const uint8_t* codes_host, int64_t B, int mode, int n_top,
                                   double rho, int precision, void* h_est_host, int out_c64);
/* The same for the circulant / block-circulant and the Woodbury-MFA models (r_host and h_est_host c128 [B][n_ant]). */
qce_status qce_circ_estimate_host(qce_circ_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho,
                                  int precision, void* h_est_host);
qce_status qce_mfa_estimate_host(qce_mfa_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho,
                                 void* h_est_host);

#ifdef __cplusplus
}
#endif
#endif /* QCE_B200_H */
