// C-ABI entry points of libqce_b200.so (declared in include/qce_b200.h).
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "qce_common.cuh"

namespace qce {
static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launch_count{0};

// keyed by (device, stream): stream handles are only unique per device (the default stream is 0 everywhere)
static std::mutex g_scratch_mu;
static std::map<std::pair<int, cudaStream_t>, StreamScratch> g_scratch;
StreamScratch* scratch_for(cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_scratch_mu);
    return &g_scratch[std::make_pair(current_device(), s)];
}
StreamScratch* scratch_find(cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_scratch_mu);
    auto it = g_scratch.find(std::make_pair(current_device(), s));
    return it == g_scratch.end() ? nullptr : &it->second;
}
void scratch_release(cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_scratch_mu);
    auto it = g_scratch.find(std::make_pair(current_device(), s));
    if (it == g_scratch.end()) return;
    StreamScratch& e = it->second;
    TileScratch& t = e.tc;
    for (ScratchBuf* b : {&t.img, &t.bad, &t.lp2, &t.wts, &t.img2, &t.bidx, &t.fix, &t.tie, &t.tmp_est, &e.circ_fix, &e.pipe_r,
                          &e.host_in, &e.host_out, &e.host_mid_in, &e.host_mid_out})
        free_buf(*b);
    g_scratch.erase(it);
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace qce

using namespace qce;

struct HostCtx {                // staging of ONE host-buffer call at a time: pinned slots and private streams (the device slots
                                // are in the streams' scratch)
    static constexpr int NSLOT = 4;  // chunks in flight: keeps the H2D and the D2H copy engines busy back to back
    int device = -1;
    cudaStream_t streams[NSLOT] = {};
    cudaEvent_t done[NSLOT] = {};
    ScratchBuf pin_in[NSLOT], pin_out[NSLOT];
    HostCtx() { for (int i = 0; i < NSLOT; ++i) pin_in[i].pinned = pin_out[i].pinned = true; }
};

void host_ctx_free(HostCtx* c) {
    if (!c) return;
    for (int i = 0; i < HostCtx::NSLOT; ++i) {
        if (c->streams[i]) { cudaStreamSynchronize(c->streams[i]); scratch_release(c->streams[i]); cudaStreamDestroy(c->streams[i]); }
        if (c->done[i]) cudaEventDestroy(c->done[i]);
        free_buf(c->pin_in[i]);
        free_buf(c->pin_out[i]);
    }
    delete c;
}

namespace {
// Staging sets are pooled per device: a host-buffer call takes a free set (or creates one) and returns it when it is done, so
// concurrent calls -- on one model or on several -- never share buffers or streams and never wait for each other, and the memory
// is bounded by the number of calls that were ever in flight at once (not by the number of models).
std::mutex g_host_pool_mu;
std::vector<HostCtx*> g_host_pool[64];
HostCtx* host_ctx_acquire(int device) {
    std::lock_guard<std::mutex> lock(g_host_pool_mu);
    auto& pool = g_host_pool[device & 63];
    if (!pool.empty()) { HostCtx* c = pool.back(); pool.pop_back(); return c; }
    HostCtx* c = new HostCtx();
    c->device = device;
    return c;
}
void host_ctx_release(HostCtx* c) {
    std::lock_guard<std::mutex> lock(g_host_pool_mu);
    g_host_pool[c->device & 63].push_back(c);
}
struct HostCtxLease {
    HostCtx* c;
    explicit HostCtxLease(int device) : c(host_ctx_acquire(device)) {}
    ~HostCtxLease() { host_ctx_release(c); }
};

// Pageable caller buffers are staged through pinned memory by the calling thread; one memcpy stream moves ~8 GB/s, far below
// PCIe, so large copies are split over a few threads.
void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    const unsigned hw = std::thread::hardware_concurrency();
    size_t nt = bytes >> 22;                                  // one thread per 4 MiB
    const size_t cap = hw >= 16 ? 8 : (hw >= 4 ? hw / 2 : 1);
    if (nt > cap) nt = cap;
    if (nt <= 1) { memcpy(dst, src, bytes); return; }
    const size_t piece = ((bytes / nt) + 4095) & ~(size_t)4095;
    std::vector<std::thread> th;
    for (size_t i = 1; i < nt; ++i) {
        const size_t off = i * piece;
        if (off >= bytes) break;
        const size_t len = (off + piece < bytes) ? piece : bytes - off;
        th.emplace_back([=] { memcpy((char*)dst + off, (const char*)src + off, len); });
    }
    memcpy(dst, src, piece < bytes ? piece : bytes);
    for (auto& t : th) t.join();
}
}  // namespace

extern "C" {

int qce_abi_version(void) { return QCE_ABI_VERSION; }

void qce_host_staging_release(void) {
    std::vector<HostCtx*> all;
    {
        std::lock_guard<std::mutex> lock(g_host_pool_mu);
        for (auto& pool : g_host_pool) { all.insert(all.end(), pool.begin(), pool.end()); pool.clear(); }
    }
    int cur = 0;
    cudaGetDevice(&cur);
    for (HostCtx* c : all) { cudaSetDevice(c->device); host_ctx_free(c); }
    cudaSetDevice(cur);
}

int64_t qce_last_fix_count(void* stream) {
    const StreamScratch* sc = scratch_find((cudaStream_t)stream);
    const int* p = sc ? sc->last_fix : nullptr;
    if (!p) return -1;
    int n[2] = {0, 0};      // rows answered completely in complex128, near-ties re-selected in complex128
    if (cudaMemcpyAsync(n, p, sizeof(n), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess ||
        cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) { cudaGetLastError(); return -1; }
    return (int64_t)n[0] + n[1];
}
const char* qce_last_error_string(void) { return g_err; }
int64_t qce_launch_count(void) { return g_launch_count.load(std::memory_order_relaxed); }

int qce_device_ok(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return 0; }
    int dev = 0, major = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    return major == 10;
}

static qce_status require_device() {
    if (!qce_device_ok()) {
        set_error("no sm_100 CUDA device visible: this library has no CPU fallback");
        return QCE_ERR_NO_DEVICE;
    }
    return QCE_OK;
}

// ---------------------------------------------------------------------------------------- quantiser

qce_status qce_quantizer_create(int n_bits, const double* thr, const double* labels, qce_quantizer** out) {
    if (!out || n_bits < 1 || n_bits > 8) { set_error("qce_quantizer_create: n_bits must be in 1..8"); return QCE_ERR_INVALID; }
    if (n_bits > 1 && (!thr || !labels)) { set_error("qce_quantizer_create: tables required for n_bits > 1"); return QCE_ERR_INVALID; }
    qce_status st = require_device();
    if (st) return st;
    qce_quantizer* q = new qce_quantizer();
    q->t.n_bits = n_bits;
    q->t.n_thr = (1 << n_bits) - 1;
    q->t.thr = q->t.labels = nullptr;
    q->dev_buf = nullptr;
    if (n_bits > 1) {
        const int nt = q->t.n_thr;
        for (int i = 1; i < nt; ++i)
            if (!(thr[i] >= thr[i - 1])) { delete q; set_error("qce_quantizer_create: thresholds must ascend"); return QCE_ERR_INVALID; }
        cudaError_t e = cudaMalloc(&q->dev_buf, sizeof(double) * (2 * nt + 1));
        if (e == cudaSuccess) e = cudaMemcpy(q->dev_buf, thr, sizeof(double) * nt, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(q->dev_buf + nt, labels, sizeof(double) * (nt + 1), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            set_error("qce_quantizer_create: %s", cudaGetErrorString(e));
            if (q->dev_buf) cudaFree(q->dev_buf);
            delete q;
            return QCE_ERR_CUDA;
        }
        q->t.thr = q->dev_buf;
        q->t.labels = q->dev_buf + nt;
    }
    *out = q;
    return QCE_OK;
}

void qce_quantizer_destroy(qce_quantizer* q) {
    if (!q) return;
    if (q->dev_buf) cudaFree(q->dev_buf);
    delete q;
}

qce_status qce_quantize(const qce_quantizer* q, void* stream, const void* y, int64_t n, void* r_out, uint8_t* codes_out) {
    if (!q || n < 0 || (n > 0 && !y)) { set_error("qce_quantize: invalid argument"); return QCE_ERR_INVALID; }
    return launch_quantize(&q->t, (cudaStream_t)stream, (const double*)y, n, (double*)r_out, codes_out);
}

qce_status qce_observe_quantize(const qce_quantizer* q, void* stream, const void* h, int h_is_c64, const void* noise,
                                double noise_scale, int64_t n, void* y_out, void* r_out, uint8_t* codes_out) {
    if (n < 0 || (n > 0 && (!h || !noise))) { set_error("qce_observe_quantize: invalid argument"); return QCE_ERR_INVALID; }
    if (!q && (r_out || codes_out)) { set_error("qce_observe_quantize: r/codes requested without a quantiser"); return QCE_ERR_INVALID; }
    return launch_observe_quantize(q ? &q->t : nullptr, (cudaStream_t)stream, h, h_is_c64, (const double*)noise,
                                   noise_scale, n, (double*)y_out, (double*)r_out, codes_out);
}

// -------------------------------------------------------------------------------------------- model

qce_status qce_model_create(int n_obs, int n_ant, int n_comp, int flags, qce_model** out) {
    if (!out || n_obs < 1 || n_ant < 1 || n_comp < 1) { set_error("qce_model_create: invalid shape"); return QCE_ERR_INVALID; }
    qce_status st = require_device();
    if (st) return st;
    qce_model* m = new qce_model();
    m->n_obs = n_obs; m->n_ant = n_ant; m->n_comp = n_comp; m->flags = flags;
    m->device = current_device();
    cudaEventCreateWithFlags(&m->params_ready, cudaEventDisableTiming);
    const size_t K = n_comp, No = n_obs, N = n_ant;
    cudaError_t e = cudaMalloc(&m->Linv, K * No * No * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->W, K * N * No * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->zoff, K * No * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->hoff, K * N * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->logc, K * 8);
    if (e != cudaSuccess) {
        set_error("qce_model_create: %s", cudaGetErrorString(e));
        qce_model_destroy(m);
        return QCE_ERR_CUDA;
    }
    *out = m;
    return QCE_OK;
}

void qce_model_destroy(qce_model* m) {
    if (!m) return;
    if (m->params_ready) cudaEventDestroy(m->params_ready);
    tc_free(m);
    cudaFree(m->Linv); cudaFree(m->W); cudaFree(m->zoff); cudaFree(m->hoff); cudaFree(m->logc);
    delete m;
}

qce_status qce_model_set_params(qce_model* m, void* stream, const double* Linv, const double* W, const double* zoff,
                                const double* hoff, const double* logc, double data_scale) {
    if (!m || !Linv || !W || !zoff || !hoff || !logc || data_scale < 0) { set_error("qce_model_set_params: invalid argument"); return QCE_ERR_INVALID; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t K = m->n_comp, No = m->n_obs, N = m->n_ant;
    QCE_CUDA_TRY(cudaMemcpyAsync(m->Linv, Linv, K * No * No * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->W, W, K * N * No * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->zoff, zoff, K * No * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->hoff, hoff, K * N * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->logc, logc, K * 8, cudaMemcpyDeviceToDevice, s));
    m->data_scale = data_scale;
    m->params_set = true;
    m->tc.ready = false;
    if (tc_supported(m, QCE_MODE_ALL)) {
        qce_status st = tc_pack_params(m, s);
        if (st) return st;
    }
    QCE_CUDA_TRY(cudaEventRecord(m->params_ready, s));
    return QCE_OK;
}

// ---------------------------------------------------------------------------------------- estimate

static qce_status check_mode(int mode, int n_top, double rho, int K) {
    switch (mode) {
        case QCE_MODE_ALL: case QCE_MODE_TOP1: return QCE_OK;
        case QCE_MODE_TOPN:
            if (n_top < 1) { set_error("n_top must be >= 1"); return QCE_ERR_INVALID; }
            return QCE_OK;
        case QCE_MODE_CUMPROB:
            if (!(rho == rho)) { set_error("rho is NaN"); return QCE_ERR_INVALID; }
            return QCE_OK;
        default: set_error("unknown mode %d", mode); return QCE_ERR_INVALID;
    }
    (void)K;
}

// the tensor-core kernels of `mode` for this model, or QCE_ERR_UNSUPPORTED and why not
static qce_status tc_require(const qce_model* m, int mode, const char* fn) {
    if (tc_supported(m, mode) && m->tc.ready) return QCE_OK;
    set_error("%s: tensor-core kernel does not support n_obs=%d n_ant=%d K=%d mode=%d%s", fn, m->n_obs, m->n_ant, m->n_comp, mode,
              tc_unsupported_reason(m));
    return QCE_ERR_UNSUPPORTED;
}

static qce_status estimate_impl(qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                                int precision, double* h_est, double* logp_out, const void* h_true, int h_true_c64,
                                double* acc) {
    if (!m || !m->params_set) { set_error("qce_estimate: model has no parameters"); return QCE_ERR_INVALID; }
    if (B < 0 || (B > 0 && !r)) { set_error("qce_estimate: invalid batch"); return QCE_ERR_INVALID; }
    qce_status st = check_mode(mode, n_top, rho, m->n_comp);
    if (st) return st;
    if (precision == QCE_PREC_FP64)
        return launch_dense_fp64_raw(m, s, r, B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
    if (precision == QCE_PREC_TC) {
        st = tc_require(m, mode, "qce_estimate");
        if (st) return st;
        return launch_dense_tc(m, s, r, B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
    }
    set_error("unknown precision %d", precision);
    return QCE_ERR_INVALID;
}

qce_status qce_estimate(qce_model* m, void* stream, const void* r, int64_t B, int mode, int n_top, double rho, int precision,
                        void* h_est, double* logp_out, const void* h_true, double* acc) {
    return estimate_impl(m, (cudaStream_t)stream, (const double*)r, B, mode, n_top, rho, precision, (double*)h_est, logp_out,
                         h_true, 0, acc);
}

qce_status qce_pipeline(qce_model* m, const qce_quantizer* q, void* stream, const void* h, int h_is_c64, const void* noise,
                        double noise_scale, int64_t B, int mode, int n_top, double rho, int precision, void* h_est,
                        double* acc) {
    if (!m || !q || B < 0 || (B > 0 && (!h || !noise))) { set_error("qce_pipeline: invalid argument"); return QCE_ERR_INVALID; }
    if (m->n_obs != m->n_ant) { set_error("qce_pipeline: A = I requires n_obs == n_ant"); return QCE_ERR_INVALID; }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t N = m->n_ant;
    if (!m->params_set) { set_error("qce_pipeline: model has no parameters"); return QCE_ERR_INVALID; }
    {
        qce_status stm = check_mode(mode, n_top, rho, m->n_comp);
        if (stm) return stm;
    }
    if (precision == QCE_PREC_TC) {
        qce_status st = tc_require(m, mode, "qce_pipeline");
        if (st) return st;
        // one formatter launch (observe + quantise + FP16 tiles) and one estimate launch per 2^22 pilots
        const int64_t chunk = (int64_t)1 << 22;
        const size_t hs = h_is_c64 ? 8 : 16;
        for (int64_t b0 = 0; b0 < B; b0 += chunk) {
            const int64_t nb = (B - b0) < chunk ? (B - b0) : chunk;
            const char* hp = (const char*)h + (size_t)b0 * N * hs;
            qce_status st = launch_pipeline_tc(m, &q->t, s, hp, h_is_c64, (const double*)noise + (size_t)b0 * N * 2, noise_scale, nb, mode, n_top, rho,
                                               h_est ? (double*)h_est + (size_t)b0 * N * 2 : nullptr, acc);
            if (st) return st;
        }
        return QCE_OK;
    }
    // quantised pilots of one chunk live in the stream's scratch (grown on first use, then reused)
    const int64_t chunk_max = (int64_t)1 << 20;
    const int64_t chunk = B < chunk_max ? B : chunk_max;
    ScratchBuf& pipe_r = scratch_for(s)->pipe_r;
    qce_status st = grow(pipe_r, (size_t)chunk * N * 16);
    if (st) return st;
    const size_t hstride = h_is_c64 ? 8 : 16;
    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
        const int64_t nb = (B - b0) < chunk ? (B - b0) : chunk;
        const char* hp = (const char*)h + (size_t)b0 * N * hstride;
        st = launch_observe_quantize(&q->t, s, hp, h_is_c64, (const double*)noise + (size_t)b0 * N * 2, noise_scale,
                                     nb * N, nullptr, (double*)pipe_r.p, nullptr);
        if (st) return st;
        st = estimate_impl(m, s, (const double*)pipe_r.p, nb, mode, n_top, rho, precision,
                           h_est ? (double*)h_est + (size_t)b0 * N * 2 : nullptr, nullptr, hp, h_is_c64, acc);
        if (st) return st;
    }
    return QCE_OK;
}

qce_status qce_circ_model_create(int n1, int n2, int n_comp, int flags, qce_circ_model** out) {
    if (!out || n1 < 1 || n2 < 1 || n_comp < 1 || n1 > 256 || n2 > 256 || n_comp > 4096) { set_error("qce_circ_model_create: invalid shape"); return QCE_ERR_INVALID; }
    qce_status st = require_device();
    if (st) return st;
    qce_circ_model* m = new qce_circ_model();
    m->n1 = n1; m->n2 = n2; m->n_ant = n1 * n2; m->n_comp = n_comp; m->flags = flags;
    m->device = current_device();
    cudaEventCreateWithFlags(&m->params_ready, cudaEventDisableTiming);
    const size_t N = m->n_ant, K = n_comp;
    cudaError_t e = cudaMalloc(&m->inv_lambda_t, N * K * 8);
    if (e == cudaSuccess) e = cudaMalloc(&m->gain, N * K * 8);
    if (e == cudaSuccess) e = cudaMalloc(&m->logc, K * 8);
    if (e != cudaSuccess) { set_error("qce_circ_model_create: %s", cudaGetErrorString(e)); qce_circ_model_destroy(m); return QCE_ERR_CUDA; }
    *out = m;
    return QCE_OK;
}

void qce_circ_model_destroy(qce_circ_model* m) {
    if (!m) return;
    if (m->params_ready) cudaEventDestroy(m->params_ready);
    circ_tc_free(m);
    cudaFree(m->inv_lambda_t); cudaFree(m->gain); cudaFree(m->logc);
    delete m;
}

qce_status qce_circ_model_set_params(qce_circ_model* m, void* stream, const double* inv_lambda_t, const double* gain, const double* logc) {
    if (!m || !inv_lambda_t || !gain || !logc) { set_error("qce_circ_model_set_params: invalid argument"); return QCE_ERR_INVALID; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = m->n_ant, K = m->n_comp;
    QCE_CUDA_TRY(cudaMemcpyAsync(m->inv_lambda_t, inv_lambda_t, N * K * 8, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->gain, gain, N * K * 8, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->logc, logc, K * 8, cudaMemcpyDeviceToDevice, s));
    m->params_set = true;
    qce_status st = circ_tc_pack(m, s);
    if (st) return st;
    QCE_CUDA_TRY(cudaEventRecord(m->params_ready, s));
    return QCE_OK;
}

qce_status qce_circ_estimate_prec(qce_circ_model* m, void* stream, const void* r, int64_t B, int mode, int n_top, double rho, int precision,
                                  void* h_est, double* logp_out, const void* h_true, double* acc) {
    if (!m || !m->params_set || B < 0 || (B > 0 && !r)) { set_error("qce_circ_estimate: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = check_mode(mode, n_top, rho, m->n_comp);
    if (st) return st;
    if (precision == QCE_PREC_TC)
        return launch_circ_tc(m, (cudaStream_t)stream, (const double*)r, B, mode, n_top, rho, (double*)h_est, logp_out, (const double*)h_true, acc);
    if (precision != QCE_PREC_FP64) { set_error("unknown precision %d", precision); return QCE_ERR_INVALID; }
    return launch_circ(m, (cudaStream_t)stream, (const double*)r, B, mode, n_top, rho, (double*)h_est, logp_out, (const double*)h_true, acc);
}

qce_status qce_circ_estimate(qce_circ_model* m, void* stream, const void* r, int64_t B, int mode, int n_top, double rho, void* h_est,
                             double* logp_out, const void* h_true, double* acc) {
    return qce_circ_estimate_prec(m, stream, r, B, mode, n_top, rho, QCE_PREC_FP64, h_est, logp_out, h_true, acc);
}

qce_status qce_mfa_model_create(int n_ant, int latent, int n_comp, int flags, qce_mfa_model** out) {
    if (!out || n_ant < 1 || latent < 1 || n_comp < 1) { set_error("qce_mfa_model_create: invalid shape"); return QCE_ERR_INVALID; }
    qce_status st = require_device();
    if (st) return st;
    qce_mfa_model* m = new qce_mfa_model();
    m->n_ant = n_ant; m->latent = latent; m->n_comp = n_comp; m->flags = flags;
    m->device = current_device();
    cudaEventCreateWithFlags(&m->params_ready, cudaEventDisableTiming);
    const size_t N = n_ant, M2 = 2 * (size_t)latent, K = n_comp;
    cudaError_t e = cudaMalloc(&m->inv_delta, K * N * 8);
    if (e == cudaSuccess) e = cudaMalloc(&m->evec, K * N * 8);
    if (e == cudaSuccess) e = cudaMalloc(&m->D, K * M2 * N * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->Y, K * N * M2 * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->m_r, K * N * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->mu, K * N * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->logc, K * 8);
    if (e != cudaSuccess) { set_error("qce_mfa_model_create: %s", cudaGetErrorString(e)); qce_mfa_model_destroy(m); return QCE_ERR_CUDA; }
    *out = m;
    return QCE_OK;
}

void qce_mfa_model_destroy(qce_mfa_model* m) {
    if (!m) return;
    if (m->params_ready) cudaEventDestroy(m->params_ready);
    cudaFree(m->inv_delta); cudaFree(m->evec); cudaFree(m->D); cudaFree(m->Y); cudaFree(m->m_r); cudaFree(m->mu); cudaFree(m->logc);
    delete m;
}

qce_status qce_mfa_model_set_params(qce_mfa_model* m, void* stream, const double* inv_delta, const double* evec, const double* D,
                                    const double* Y, const double* m_r, const double* mu, const double* logc) {
    if (!m || !inv_delta || !evec || !D || !Y || !m_r || !mu || !logc) { set_error("qce_mfa_model_set_params: invalid argument"); return QCE_ERR_INVALID; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = m->n_ant, M2 = 2 * (size_t)m->latent, K = m->n_comp;
    QCE_CUDA_TRY(cudaMemcpyAsync(m->inv_delta, inv_delta, K * N * 8, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->evec, evec, K * N * 8, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->D, D, K * M2 * N * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->Y, Y, K * N * M2 * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->m_r, m_r, K * N * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->mu, mu, K * N * 16, cudaMemcpyDeviceToDevice, s));
    QCE_CUDA_TRY(cudaMemcpyAsync(m->logc, logc, K * 8, cudaMemcpyDeviceToDevice, s));
    m->params_set = true;
    QCE_CUDA_TRY(cudaEventRecord(m->params_ready, s));
    return QCE_OK;
}

qce_status qce_mfa_estimate(qce_mfa_model* m, void* stream, const void* r, int64_t B, int mode, int n_top, double rho, void* h_est,
                            double* logp_out, const void* h_true, double* acc) {
    if (!m || !m->params_set || B < 0 || (B > 0 && !r)) { set_error("qce_mfa_estimate: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = check_mode(mode, n_top, rho, m->n_comp);
    if (st) return st;
    return launch_mfa(m, (cudaStream_t)stream, (const double*)r, B, mode, n_top, rho, (double*)h_est, logp_out, (const double*)h_true, acc);
}

qce_status qce_rate_model_create(int n_ant, qce_rate_model** out) {
    if (!out || n_ant < 1) { set_error("qce_rate_model_create: invalid shape"); return QCE_ERR_INVALID; }
    if (n_ant > 256) { set_error("qce_rate_model_create: n_ant=%d not supported (at most 256)", n_ant); return QCE_ERR_UNSUPPORTED; }
    qce_status st = require_device();
    if (st) return st;
    qce_rate_model* m = new qce_rate_model();
    m->n_ant = n_ant;
    m->n_pad = (n_ant + 15) & ~15;
    m->device = current_device();
    cudaError_t e = cudaMalloc(&m->buss, (size_t)n_ant * 16);
    if (e == cudaSuccess) e = cudaMalloc(&m->frag, (size_t)m->n_pad * m->n_pad * 16);     // (2 Np)^2 halves, hi and lo
    if (e != cudaSuccess) { set_error("qce_rate_model_create: %s", cudaGetErrorString(e)); qce_rate_model_destroy(m); return QCE_ERR_CUDA; }
    *out = m;
    return QCE_OK;
}

void qce_rate_model_destroy(qce_rate_model* m) {
    if (!m) return;
    cudaFree(m->buss); cudaFree(m->frag);
    delete m;
}

static qce_status rate_device_check(const qce_rate_model* m, const char* fn) {
    if (current_device() != m->device) {
        set_error("%s: the model lives on device %d, the calling thread's current device is %d", fn, m->device, current_device());
        return QCE_ERR_INVALID;
    }
    return QCE_OK;
}

qce_status qce_rate_model_set_params(qce_rate_model* m, void* stream, const double* buss_diag, const double* cq) {
    if (!m || !buss_diag || !cq) { set_error("qce_rate_model_set_params: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = rate_device_check(m, "qce_rate_model_set_params");
    if (st) return st;
    cudaStream_t s = (cudaStream_t)stream;
    m->params_set = false;
    QCE_CUDA_TRY(cudaMemcpyAsync(m->buss, buss_diag, (size_t)m->n_ant * 16, cudaMemcpyDeviceToDevice, s));
    st = rate_pack(m, s, cq);
    if (st) return st;
    m->params_set = true;
    return QCE_OK;
}

qce_status qce_rate_accumulate(qce_rate_model* m, void* stream, const void* h_est, const void* h_true, int h_true_c64, int64_t B,
                               double* acc) {
    if (!m || !m->params_set || B < 0 || (B > 0 && (!h_est || !h_true || !acc))) { set_error("qce_rate_accumulate: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = rate_device_check(m, "qce_rate_accumulate");
    if (st) return st;
    if (B == 0) return QCE_OK;
    return launch_rate(m, (cudaStream_t)stream, (const double*)h_est, h_true, h_true_c64 ? 1 : 0, B, acc);
}

qce_status qce_format_pilots(qce_model* m, void* stream, const void* r, int64_t B) {
    if (!m || !m->params_set || B < 0 || (B > 0 && !r)) { set_error("qce_format_pilots: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = tc_require(m, QCE_MODE_ALL, "qce_format_pilots");
    if (st) return st;
    return tc_format(m, (cudaStream_t)stream, (const double*)r, B);
}

qce_status qce_estimate_formatted(qce_model* m, void* stream, int64_t B, void* h_est, const void* h_true, double* acc) {
    if (!m || !m->params_set || B < 0) { set_error("qce_estimate_formatted: invalid argument"); return QCE_ERR_INVALID; }
    qce_status st = tc_require(m, QCE_MODE_ALL, "qce_estimate_formatted");
    if (st) return st;
    return tc_estimate_formatted(m, (cudaStream_t)stream, B, (double*)h_est, h_true, 0, acc);
}

}  // extern "C"

// Host-buffer estimate, shared by the dense / circulant / MFA entry points: r_host c128 [B][n_in] -> h_est_host c128 [B][n_out].
// NSLOT chunks are in flight: H2D copy, kernel(s) and D2H copy of a chunk run on the slot's own stream, so that both copy engines
// stay busy back to back.  Page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are copied directly;
// pageable ones go through the pinned staging slots.  `run(stream, dev_in, rows, dev_out)` enqueues the estimate of one chunk.
template <typename Run>
static qce_status estimate_host_impl(int model_device, cudaEvent_t params_ready, size_t in_row, size_t out_row,
                                     size_t mid_in_row, size_t mid_out_row, const void* r_host, int64_t B, void* h_est_host, Run run) {
    // in_row / out_row: bytes per pilot that cross PCIe; mid_*_row: bytes per pilot of device-only intermediates (0: none)
    if (current_device() != model_device) {
        set_error("host-buffer estimate: the model lives on device %d, the calling thread's current device is %d", model_device, current_device());
        return QCE_ERR_INVALID;
    }
    HostCtxLease lease(model_device);
    HostCtx* hs = lease.c;
    const size_t slot_bytes = (size_t)32 << 20;
    constexpr int NSLOT = HostCtx::NSLOT;
    size_t max_row = in_row > out_row ? in_row : out_row;
    if (mid_in_row > max_row) max_row = mid_in_row;
    if (mid_out_row > max_row) max_row = mid_out_row;
    int64_t chunk = (int64_t)(slot_bytes / max_row);
    if (chunk < 128) chunk = 128;
    StreamScratch* dev[NSLOT];         // device slots: in the scratch of the slot's stream
    for (int i = 0; i < NSLOT; ++i) {
        if (!hs->streams[i]) {
            QCE_CUDA_TRY(cudaStreamCreateWithFlags(&hs->streams[i], cudaStreamNonBlocking));
            QCE_CUDA_TRY(cudaEventCreateWithFlags(&hs->done[i], cudaEventDisableTiming));
        }
        dev[i] = scratch_for(hs->streams[i]);
        qce_status st = grow(dev[i]->host_in, (size_t)chunk * in_row);
        if (!st) st = grow(dev[i]->host_out, (size_t)chunk * out_row);
        if (!st) st = grow(dev[i]->host_mid_in, (size_t)chunk * mid_in_row);
        if (!st) st = grow(dev[i]->host_mid_out, (size_t)chunk * mid_out_row);
        if (st) return st;
    }
    // parameters were uploaded / packed on the caller's stream: the private streams wait for that upload (an event, not a device-wide
    // synchronisation: other streams of the process are left alone)
    for (int i = 0; i < NSLOT; ++i) QCE_CUDA_TRY(cudaStreamWaitEvent(hs->streams[i], params_ready, 0));
    const int64_t nchunks = (B + chunk - 1) / chunk;
    auto is_pinned = [](const void* p) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return at.type == cudaMemoryTypeHost;
    };
    const bool in_pinned = is_pinned(r_host), out_pinned = is_pinned(h_est_host);
    // pinned staging slots only where the caller's buffer is pageable (page-locked buffers are copied directly)
    for (int i = 0; i < NSLOT; ++i) {
        qce_status st = grow(hs->pin_in[i], in_pinned ? 0 : (size_t)chunk * in_row);
        if (!st) st = grow(hs->pin_out[i], out_pinned ? 0 : (size_t)chunk * out_row);
        if (st) return st;
    }
    int64_t pending_b0[NSLOT], pending_nb[NSLOT];
    for (int i = 0; i < NSLOT; ++i) { pending_b0[i] = -1; pending_nb[i] = 0; }
    auto drain = [&](int slot) -> qce_status {
        if (pending_b0[slot] < 0) return QCE_OK;
        QCE_CUDA_TRY(cudaEventSynchronize(hs->done[slot]));
        if (!out_pinned)
            parallel_memcpy((char*)h_est_host + (size_t)pending_b0[slot] * out_row, hs->pin_out[slot].p, (size_t)pending_nb[slot] * out_row);
        pending_b0[slot] = -1;
        return QCE_OK;
    };
    for (int64_t c = 0; c < nchunks; ++c) {
        const int slot = (int)(c % NSLOT);
        qce_status st = drain(slot);
        if (st) return st;
        const int64_t b0 = c * chunk, nb = (B - b0) < chunk ? (B - b0) : chunk;
        const char* src = (const char*)r_host + (size_t)b0 * in_row;
        if (!in_pinned) { parallel_memcpy(hs->pin_in[slot].p, src, (size_t)nb * in_row); src = (const char*)hs->pin_in[slot].p; }
        cudaStream_t s = hs->streams[slot];
        const StreamScratch* d = dev[slot];
        QCE_CUDA_TRY(cudaMemcpyAsync(d->host_in.p, src, (size_t)nb * in_row, cudaMemcpyHostToDevice, s));
        st = run(s, (const double*)d->host_in.p, nb, (double*)d->host_out.p, d->host_mid_in.p, d->host_mid_out.p);
        if (st) return st;
        void* dst = out_pinned ? (void*)((char*)h_est_host + (size_t)b0 * out_row) : hs->pin_out[slot].p;
        QCE_CUDA_TRY(cudaMemcpyAsync(dst, d->host_out.p, (size_t)nb * out_row, cudaMemcpyDeviceToHost, s));
        QCE_CUDA_TRY(cudaEventRecord(hs->done[slot], s));
        pending_b0[slot] = b0; pending_nb[slot] = nb;
    }
    for (int slot = 0; slot < NSLOT; ++slot) {
        qce_status st = drain(slot);
        if (st) return st;
    }
    return QCE_OK;
}

extern "C" {

qce_status qce_estimate_host(qce_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho, int precision,
                             void* h_est_host) {
    if (!m || !m->params_set || B < 0 || (B > 0 && (!r_host || !h_est_host))) { set_error("qce_estimate_host: invalid argument"); return QCE_ERR_INVALID; }
    return estimate_host_impl(m->device, m->params_ready, (size_t)m->n_obs * 16, (size_t)m->n_ant * 16, 0, 0, r_host, B, h_est_host,
                              [&](cudaStream_t s, const double* din, int64_t nb, double* dout, void*, void*) {
                                  return estimate_impl(m, s, din, nb, mode, n_top, rho, precision, dout, nullptr, nullptr, 0, nullptr);
                              });
}

qce_status qce_estimate_host_codes(qce_model* m, const qce_quantizer* q, const uint8_t* codes_host, int64_t B, int mode, int n_top, double rho,
                                   int precision, void* h_est_host, int out_c64) {
    if (!m || !q || !m->params_set || B < 0 || (B > 0 && (!codes_host || !h_est_host))) { set_error("qce_estimate_host_codes: invalid argument"); return QCE_ERR_INVALID; }
    const size_t No = m->n_obs, N = m->n_ant;
    return estimate_host_impl(m->device, m->params_ready, No * 2, N * (out_c64 ? 8 : 16), No * 16, out_c64 ? N * 16 : 0, codes_host, B, h_est_host,
                              [&](cudaStream_t s, const double* din, int64_t nb, double* dout, void* mid_in, void* mid_out) {
                                  qce_status st = launch_decode_codes(&q->t, s, (const uint8_t*)din, nb * (int64_t)No, (double*)mid_in);
                                  if (st) return st;
                                  double* est = out_c64 ? (double*)mid_out : dout;
                                  st = estimate_impl(m, s, (const double*)mid_in, nb, mode, n_top, rho, precision, est, nullptr, nullptr, 0, nullptr);
                                  if (st || !out_c64) return st;
                                  return launch_c128_to_c64(s, est, nb * (int64_t)N, (float*)dout);
                              });
}

qce_status qce_circ_estimate_host(qce_circ_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho, int precision,
                                  void* h_est_host) {
    if (!m || !m->params_set || B < 0 || (B > 0 && (!r_host || !h_est_host))) { set_error("qce_circ_estimate_host: invalid argument"); return QCE_ERR_INVALID; }
    return estimate_host_impl(m->device, m->params_ready, (size_t)m->n_ant * 16, (size_t)m->n_ant * 16, 0, 0, r_host, B, h_est_host,
                              [&](cudaStream_t s, const double* din, int64_t nb, double* dout, void*, void*) {
                                  return qce_circ_estimate_prec(m, (void*)s, din, nb, mode, n_top, rho, precision, dout, nullptr, nullptr, nullptr);
                              });
}

qce_status qce_mfa_estimate_host(qce_mfa_model* m, const void* r_host, int64_t B, int mode, int n_top, double rho, void* h_est_host) {
    if (!m || !m->params_set || B < 0 || (B > 0 && (!r_host || !h_est_host))) { set_error("qce_mfa_estimate_host: invalid argument"); return QCE_ERR_INVALID; }
    return estimate_host_impl(m->device, m->params_ready, (size_t)m->n_ant * 16, (size_t)m->n_ant * 16, 0, 0, r_host, B, h_est_host,
                              [&](cudaStream_t s, const double* din, int64_t nb, double* dout, void*, void*) {
                                  return qce_mfa_estimate(m, (void*)s, din, nb, mode, n_top, rho, dout, nullptr, nullptr, nullptr);
                              });
}

}  // extern "C"
