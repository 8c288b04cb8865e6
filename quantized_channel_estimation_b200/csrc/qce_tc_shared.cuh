// Shared pieces of the tensor-core kernels: kernel arguments and mbarrier / bulk-copy / tcgen05 PTX wrappers of qce_dense_tc.cu;
// the mma.sync split-FP16 helpers of qce_circ_tc.cu and qce_rate.cu.
#pragma once
#include <math.h>
#include <stdlib.h>

#include "qce_common.cuh"

namespace qce {

// per-role cycle counters (QCE_TC_PROF=1 prints them) cost issue slots in the single-thread MMA loop: compile them in only
// with -DQCE_TC_PROFILE
#ifdef QCE_TC_PROFILE
#define QCE_CLK() clock64()
#else
#define QCE_CLK() 0LL
#endif

constexpr int TILE_M = 128;
constexpr int TILES = 2;
constexpr int NUM_THREADS = 384;
constexpr int SMEM_LIMIT = 227 * 1024;

// A component of weight 0 has logc = -inf; the reference gives it responsibility 0.  The FP32 (hi, lo) pairs of the tensor-core
// kernels cannot hold -inf: the lo part of the split and the pair subtraction l = logc - q would both be -inf - (-inf) = NaN, which
// spreads through the softmax to every estimate of the pilot.  So the pair of such a component is the finite (TC_LOGC_ZERO_WEIGHT,
// 0): its l_k stays at -2^100 (a quadratic form would have to reach 2^76, half an ulp there, to move it), exp(l_k - l_max) is 0,
// and it is the maximum only if every component is.  The FP64 logc keeps -inf, and the log-probability exports map anything below
// TC_LOGP_ZERO_WEIGHT back to -inf.
constexpr float TC_LOGC_ZERO_WEIGHT = -0x1p100f;
constexpr double TC_LOGP_ZERO_WEIGHT = -0x1p99;

__device__ __forceinline__ float2 tc_logc_pair(double l) {
    if (l == -INFINITY) return make_float2(TC_LOGC_ZERO_WEIGHT, 0.f);
    const float hi = (float)l;
    return make_float2(hi, (float)(l - (double)hi));
}

__device__ __forceinline__ double tc_logp_export(double l) { return l < TC_LOGP_ZERO_WEIGHT ? -INFINITY : l; }

struct TcArgs {
    const __half* image;       // CG=1: [K][hi | lo] stacked [E(Linv); E(W)] images, canonical K-major core-matrix order
    const unsigned char* image2;  // CG=2: [K][rank][hi K0 | hi K1 | lo K0 | lo K1] per-CTA half images (see tc2_pack_kernel)
    const float* zscale;       // [K] 2^-e of the Linv image
    const float* hscale;       // [K]
    const float* zoff;         // [K][2No] fp32 (only if OFFS)
    const float* hoff;         // [K][2N]
    const float2* logc2;       // [K] logc_k as an unevaluated FP32 pair (hi, lo)
    const __half* a_img;       // [n_tiles][128 x 2No] pilots as exact FP16 integers, canonical K-major core-matrix tiles
    const unsigned char* bad;  // [n_tiles * 128] rows the tensor-core path cannot answer (data not on the quantiser grid): their
                               // estimates are neither written nor accumulated here; they are on the fix list and re-evaluated
                               // completely by the complex128 kernel after the tensor-core launches
    int* tie_buf;              // EPI=1 label mode: [0] count, then the rows of this launch whose top-1 selection is too close to
    float tie_eps, inv_nobs;   // call (deciding log-likelihood gap below tie_eps nats, times q / n_obs of the best component when
                               // that exceeds one): tc_refine_kernel + the exact selection re-select them
    double2* h_est;            // [B][N] or null
    float2* lp_out;            // EPI=1: [B][K] weighted log-probabilities as FP32 (hi, lo) pairs
    const float* w_in;         // EPI=2: [B][K] combination weights
    const void* h_true;        // [B][N] c64/c128 or null
    int h_true_c64;
    double* acc;               // [3] or null
    int64_t B;
    int K, No, N;
    long long* prof;           // optional per-role cycle counters of block 0 (QCE_TC_PROF=1), else null
    int tri;                   // Linv_k lower triangular (Cholesky whitening): skip the structurally zero columns
    // H-part launches of the split path (64 < N <= 128): this launch produces the real columns [h_col0, h_col0 + NH) of the
    // 2N-column estimate row
    int h_stride;              // floats per component in hoff (2N)
    int h_col0;
    int count_rows;            // add the number of rows to acc[2] (only one of the H-part launches does)
    int wide_io;               // h_est and h_true are 32-byte aligned: rows are written / read with 256-bit accesses
    // bucketed top-1 combination (EPI=2, all three null otherwise): the pilots were regrouped by their selected component, work
    // unit u holds pilots of component unit_comp[u] only and runs that ONE component; slot -> pilot through perm (-1 = padding)
    const int* unit_comp;      // [*n_units_dev]
    const int* perm;           // [B] (B = slot capacity of the launch)
    const int* n_units_dev;    // number of work units actually filled (device-side: the bucket sizes are data)
    // pair mode of the bucketed combination (top-n / cumulative / sparse 'all'): a slot is one (pilot, component) pair with the
    // combination weight slot_w[slot]; a pilot has several slots in different units, so the weighted LMMSE rows are ADDED to the
    // pilot's (zero-initialised) FP32 row with vector reductions; tc_pair_finish_kernel turns the rows into estimates + NMSE sums
    const float* slot_w;       // [slots] or null
    float* pair_acc;           // [rows][2N] FP32 rows the pair launches add into (vector reductions)
    // launches that are enqueued unconditionally but only one of which has work (bucketed pairs vs the dense weighted launch: the
    // number of pairs is data): the kernel returns at once unless *run_flag == run_flag_want
    const int* run_flag;
    int run_flag_want;
    // EPI=1 with top_out != null: running argmax of l_k in the epilogue thread instead of the log-probability export (top-1 label
    // with tc_select_kernel's semantics: first index among equal maxima; QCE_FLAG_TOP1_EXP_ARGMAX in top_flags: label 0 on underflow)
    int* top_out;              // [B]
    int top_flags;
};

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        if (clock64() - t0 > 8000000000LL) {      // ~4 s: a protocol bug must not hang the GPU
            printf("qce dense_tc: mbarrier timeout (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, bar, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}
// arrive on the barrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
    uint32_t raddr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(bar), "r"(rank));
    // default semantics (release at CTA scope, like cutlass::arch::ClusterBarrier::arrive): a cluster-scope release costs a
    // full fence + L1 invalidate per arrival; the data handed over here lives in TMEM / async-proxy smem, not in generic memory
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one lane of a converged warp (the warp runs the issuing loop with uniform control flow so that descriptors stay in
// uniform registers; only the tcgen05 instructions themselves are predicated on the elected lane)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_commit2(uint32_t bar) {      // cta_group::2: arrive on the barrier at this offset in both CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// shared-memory matrix descriptors are passed as (low word, common high word): the low word is a 32-bit base plus an
// immediate in the issuing loop, the high word (SBO | version) is a constant
__device__ __forceinline__ void umma2_f16(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accum) : "memory");
}
// K-major, no-swizzle canonical layout: 8x16B core matrices; LBO = byte step between the two K-adjacent core
// matrices of one MMA, SBO = byte step between M/N-adjacent core matrices (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;        // descriptor version 1 (Blackwell)
    return d;                      // base_offset 0, lbo_mode 0, layout_type 0 = SWIZZLE_NONE
}
__device__ __forceinline__ constexpr uint32_t make_idesc(int n_cols) {
    // c_format F32 (bit 4), a/b format F16 (0), a/b K-major (0), N>>3 at bit 17, M>>4 at bit 24
    return (1u << 4) | ((uint32_t)(n_cols >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t* u = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
          "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
          "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- mma.sync helpers of the split-FP16 kernels (qce_circ_tc.cu, qce_rate.cu): an operand x is carried as hi + lo with
// hi = fp16(x), lo = fp16(x - hi), and a product is three MMAs (hi*hi + lo*hi + hi*lo, ~22 significant bits)
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_ptr) {
    const uint32_t addr = (uint32_t)__cvta_generic_to_shared(smem_ptr);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t b0, const uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split_half(const float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}

}  // namespace qce
