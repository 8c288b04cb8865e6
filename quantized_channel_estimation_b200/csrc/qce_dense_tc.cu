// Tensor-core estimate kernel (QCE_PREC_TC): tcgen05.mma + TMEM accumulators + bulk-TMA operand staging.
//
// Maths (mode 'all', reference modules/gmm_cplx_bussgang.py:220-228 after _prepare_for_prediction):
//     l_k = logc_k - |Linv_k r - zoff_k|^2,   h = sum_k softmax(l)_k (W_k r + hoff_k)
// Formulation as real GEMMs.  A complex matrix-vector product is the real product with the 2x2-block
// embedding E[2i+a][2j+b] = {Re, -Im; Im, Re}, vectors interleaved (re, im).  One sample tile is 128
// pilots (the MMA M dimension, one TMEM lane per pilot); for component k the tensor core computes
//     Z = R * E(Linv_k)^T   [128 x 2No]      H = R * E(W_k)^T   [128 x 2N]
// with FP32 accumulators in TMEM.  Precision: the quantised pilots are small integers times a known
// scale (1 bit: +-1; uniform b bit: odd integers), i.e. EXACT in FP16, so only the parameter operand is
// split, P = P_hi + P_lo (two FP16 terms, ~22 significant bits after a per-matrix power-of-two scale),
// and every GEMM is two kind::f16 passes accumulating into the same TMEM tile.
//
// CTA organisation (persistent, one CTA per SM, 384 threads):
//   warp 0      bulk-TMA producer: streams the pre-formatted operand image of component k = 0..K-1 -- the stacked
//               matrix [E(Linv_k); E(W_k)] (so one MMA of N = 2No + 2N columns yields Z|H at once), hi then lo
//               term, each in two K-halves -- through a ring of shared-memory stages (cp.async.bulk + mbarrier tx)
//   warp 1      MMA issuer (one elected thread): each staged chunk is used for BOTH resident sample tiles
//               (256 pilots per CTA share one operand fetch), tile-major so the tiles' accumulators complete half
//               a component apart; Linv_k is lower triangular, so K-step ks only feeds columns >= 16 ks and the
//               MMA is issued with the shrunken N; tcgen05.commit releases stages / publishes accumulators
//   warp 2      TMEM allocator
//   warps 4-7   epilogue warpgroup of tile 0, warps 8-11 of tile 1: one thread per pilot; tcgen05.ld the
//               whitened row -> |z|^2 -> l_k -> lazily rescaled online softmax -> FMA of the LMMSE row into
//               128 register accumulators.  Per-component estimates never leave the SM.
// CG = 2 (default): two CTAs of a cluster form an SM pair; the leader issues tcgen05.mma.cta_group::2 with M = 256 (each
// CTA's 128-pilot tile in its own TMEM) and each CTA stages only HALF of every operand chunk (its N'/2 rows), which
// halves the shared-memory operand traffic per SM -- the measured limit of cta_group::1 SS-mode MMAs (172 clk for
// M128 x N256 x K16 instead of 128) -- and the L2->smem traffic.  Cross-CTA signalling: multicast tcgen05.commit for
// "stage free" / "accumulator ready", remote mbarrier arrives (mapa) for "peer chunk landed" / "accumulator drained".
// The two tiles ping-pong: while the epilogue warpgroup of tile 0 drains Z|H(k), the tensor core produces
// Z|H(k) of tile 1, and so on.
#include "qce_tc_shared.cuh"

namespace qce {

// CG=2 per-CTA operand images.  K-step ks (16 reduction elements) needs the stacked rows [skip, NT), skip = 16 ks for a
// triangular Linv (else 0): N' = NT - skip rows, of which rank 0 holds the first N'/2 and rank 1 the rest.  A chunk is the
// concatenation over the K-steps of one K-half of the sub-blocks [2 k-cores][N'/16 n-cores][128 B].
__host__ __device__ constexpr int tc2_nprime(int nt, int tri16, int ks) { return nt - tri16 * ks; }
__host__ __device__ constexpr int tc2_sub_off(int nt, int tri16, int ksps, int half, int s2) {     // byte offset of sub-block s2 in its chunk
    return 16 * (s2 * nt - tri16 * (s2 * half * ksps + s2 * (s2 - 1) / 2));
}
__host__ __device__ constexpr int tc2_chunk_bytes(int nt, int tri16, int ksps, int half) { return tc2_sub_off(nt, tri16, ksps, half, ksps); }
// byte offset of K-step ks's sub-block from the start of its pass image (the sub-blocks of a pass are stored in K-step order)
__host__ __device__ constexpr int tc2_ks_off(int nt, int tri16, int ks) { return 16 * (ks * nt - tri16 * (ks * (ks - 1) / 2)); }
// A K-step whose N' exceeds the 256 columns of one MMA (the whitening block of n_obs = 256: NT = 512) is issued as two MMAs, rows
// [skip, 256) and [256, NT); each piece is split between the two CTAs on its own (rank 0 holds the first half of the piece's rows),
// and the per-rank sub-block holds the first piece's rows, then the second's.  Width of the first piece:
__host__ __device__ constexpr int tc2_piece0(int np) { return np > 256 ? np - 256 : np; }
__host__ __device__ constexpr int tc2_rank_comp_bytes(int nt, int tri16, int ksps) {
    return 2 * (tc2_chunk_bytes(nt, tri16, ksps, 0) + tc2_chunk_bytes(nt, tri16, ksps, 1));
}

// ORDER 0 = tile-major (all chunks of a component for tile 0, then for tile 1: the accumulators complete half a component
// apart), ORDER 1 = chunk-major (each chunk feeds both tiles, then is released: two ring stages suffice -- the split
// launches of the large shapes, whose pilot tiles leave less than 100 KB for the ring)
// AC = 2: pilots that are not on an integer grid (Lloyd-Max labels, unquantised data) are staged as an FP16 (hi, lo) pair of tile
// images; the hi parameter image is then multiplied with both (three tensor passes instead of two)
// ACCB = 2: two TMEM accumulators per pilot tile.  The whitening-only launch of the fused shapes (NZ <= 128, NH = 0) uses 256 of the
// 512 columns and its MMAs per component are short (N' = 128 ... 16), so with one accumulator per tile the chain MMA(k) -> epilogue(k)
// -> MMA(k+1) of a tile was the cycle: tensor pipe 61 % active (profiles/r02_top1_whitening_ncu_summary.txt).  With two, the MMAs of
// component k+1 run while the epilogue drains component k.  The fused launch of the small shapes (N <= 32: Z|H is at most 128 columns)
// gains the same way: config 1 (N = 32, K = 16) 0.86 -> 0.74 ms per 2^20 pilots.  (The row-block launches -- NZ = 0, NH <= 128 -- would
// fit two accumulators as well; measured, neither the weighted nor the bucketed form gains: 1350 / 275 us either way.)
__host__ __device__ constexpr int tc_accb(int epi, int kd, int nz, int nh, int order, int ac) {
    return (((epi == 1 && nh == 0) || epi == 0 || epi == 3) && order == 0 && 2 * ((ac == 2 && kd > 128) ? 1 : TILES) * (nz + nh) <= 512) ? 2 : 1;
}

template <int KD_, int NZ, int NH, int CG, int ORDER = 0, int AC = 1, int ACCB_ = 1>
struct TcCfg {
    static constexpr int KD = KD_;                                  // GEMM reduction length 2*n_obs
    static constexpr int NT = NZ + NH;                              // fused MMA N: Z columns then H columns
    static constexpr int TRI16 = NZ > 0 ? 16 : 0;                   // CG=2 image: K-step ks skips the first 16 ks (Z) rows
    static constexpr int A_COPY_BYTES = TILE_M * KD * 2;
    static constexpr int A_TILE_BYTES = AC * A_COPY_BYTES;
    // resident pilot tiles per CTA: two (their epilogues ping-pong), or one when the (hi, lo) tile pairs of the large shapes would
    // not leave room for the operand ring (the second epilogue warpgroup then idles and the accumulator is not double-buffered)
    // (n_obs = 256: one pilot tile is 128 KB, so there is one per CTA whatever AC is)
    static constexpr int NTILES = ((AC == 2 && KD > 128) || KD > 256) ? 1 : TILES;
    static constexpr int KSPS = KD / 32;                            // K-steps (of 16) per staged chunk = half the K range
    // CG=1: a chunk is one K-half of the stacked hi (or lo) image, 4 chunks per component.
    // CG=2: a chunk is this CTA's share of the whole hi (or lo) image (triangular layout), 2 chunks per component -- or, at KD = 512
    // (KSLICED), of a K-slice of KSLICE K-steps: a whole pass is 132 KB (whitening) / 64 KB (row block) there, which does not fit next
    // to the 128 KB pilot tile; a slice is at most 31 KB / 8 KB, 2 KD / (16 KSLICE) chunks per component.
    static constexpr bool KSLICED = CG == 2 && KD > 256;
    static constexpr int KSLICE = KSLICED ? 4 : KD / 16;            // K-steps per chunk (CG=2)
    static constexpr int CPP = (KD / 16) / KSLICE;                  // chunks per pass (CG=2)
    static constexpr int NCHUNK = (CG == 2) ? 2 * CPP : 4;
    static constexpr int CB0 = tc2_chunk_bytes(NT, TRI16, KSPS, 0), CB1 = tc2_chunk_bytes(NT, TRI16, KSPS, 1);
    static constexpr int PASS_BYTES = CB0 + CB1;                    // CG=2: this CTA's share of one pass (hi or lo)
    // (the first K-slice of a pass is its largest)
    static constexpr int STAGE_BYTES = (CG == 2) ? (KSLICED ? tc2_ks_off(NT, TRI16, KSLICE) : PASS_BYTES) : NT * (KD / 2) * 2;
    // CG=2: chunk q = K-slice q % CPP of pass q / CPP, at this byte offset of the CTA's component image, this long
    __host__ __device__ static constexpr int chunk_off(int q) { return (q / CPP) * PASS_BYTES + tc2_ks_off(NT, TRI16, (q % CPP) * KSLICE); }
    __host__ __device__ static constexpr int chunk_bytes(int q) { return tc2_ks_off(NT, TRI16, (q % CPP + 1) * KSLICE) - tc2_ks_off(NT, TRI16, (q % CPP) * KSLICE); }
    static constexpr int CTRL_BYTES = 1024;
    static constexpr int STAGES_FIT = (SMEM_LIMIT - NTILES * A_TILE_BYTES - CTRL_BYTES) / STAGE_BYTES;
    // (more than 8 stages do not help -- the whitening-only launch waits as long for operands with 16 -- and the weighted combine
    // launch of the fused shapes got 12 % SLOWER with 10 instead of 8: profiles/r02_whitening_notes.md)
    static constexpr int STAGES = STAGES_FIT > 8 ? 8 : STAGES_FIT;
    static constexpr int SMEM_BYTES = NTILES * A_TILE_BYTES + STAGES * STAGE_BYTES + CTRL_BYTES;
    static constexpr int COMP_HALFS = 2 * NT * KD;                  // CG=1: halfs per component image: hi then lo
    static constexpr int ACCB = ACCB_;
    static constexpr int TMEM_COLS_USED = NTILES * NT * ACCB;
    static constexpr int TMEM_COLS = TMEM_COLS_USED <= 32 ? 32 : TMEM_COLS_USED <= 64 ? 64 : TMEM_COLS_USED <= 128 ? 128
                                     : TMEM_COLS_USED <= 256 ? 256 : 512;
    static_assert(STAGES >= (ORDER == 0 ? NCHUNK + 1 : 2), "tile-major schedule keeps the chunks of a component resident plus one prefetch");
    static_assert(NZ == 0 || NZ == KD, "the whitening block is square");
    static_assert(NT >= 32, "empty launch");
    static_assert(STAGE_BYTES % 128 == 0, "stage alignment");
    static_assert(NT <= 256 || (KSLICED && NH == 0 && NT <= 512), "fused MMA N exceeds 256 (wider: whitening-only K-sliced launch)");
    static_assert(!KSLICED || (AC == 1 && ORDER == 1 && (KD / 16) % KSLICE == 0), "K-sliced chunks: on-grid pilots, chunk-major order");
    static_assert(TMEM_COLS_USED <= 512, "accumulators exceed TMEM");
};

// control block at the end of dynamic smem
struct TcCtrl {
    uint64_t full[8], empty[8];
    uint64_t acc_full[2 * TILES], acc_empty[2 * TILES];      // [tile * ACCB + buffer]
    uint64_t a_full, a_free;
    uint32_t tmem_base;
    uint32_t pad;
};
static_assert(sizeof(TcCtrl) <= 1024, "control block");

// All MMAs of one staged chunk q for one tile (every argument but the two descriptor bases folds to an immediate after
// unrolling; the whole warp executes this with uniform control flow, the elected lane issues).
template <class Cfg, int CG>
__device__ __forceinline__ void tc_issue_chunk(const int q, const uint32_t d_tile, const uint32_t a_lo_t, const uint32_t b_addr_s,
                                               const int tri16, const bool elected) {
    constexpr int NT = Cfg::NT, KSPS = Cfg::KSPS;
    constexpr uint32_t A_LBO = (TILE_M / 8) * 128;                              // SBO = 128 for both operands
    constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);                      // SBO field | descriptor version 1
    constexpr uint32_t IDESC0 = (1u << 4) | ((uint32_t)((CG * TILE_M) >> 4) << 24);
    constexpr int KS_PER_CHUNK = (CG == 2) ? Cfg::KSLICE : KSPS;
    #pragma unroll
    for (int s2 = 0; s2 < KS_PER_CHUNK; ++s2) {
        const int ks = (CG == 2) ? (Cfg::KSLICED ? (q % Cfg::CPP) * Cfg::KSLICE + s2 : s2) : (q & 1) * KSPS + s2;      // K-step within the full K range
        const bool lo_pass = (CG == 2) ? (q >= Cfg::CPP) : (q >= 2);
        const uint32_t skip = (uint32_t)(tri16 * ks);                   // structurally zero leading columns
        const uint32_t np = NT - skip;                                  // N' of this MMA
        const uint32_t a_lo = a_lo_t + ks * ((2 * A_LBO) >> 4);
        uint32_t b_lo;
        if constexpr (CG == 2 && Cfg::KSLICED) {      // K-slice chunk: sub-blocks in K-step order from the slice's first
            const int off = tc2_ks_off(NT, Cfg::TRI16, ks) - tc2_ks_off(NT, Cfg::TRI16, (q % Cfg::CPP) * Cfg::KSLICE);
            const uint32_t n0 = (uint32_t)tc2_piece0((int)np);
            b_lo = (b_addr_s + (uint32_t)(off >> 4)) | ((n0 >> 1) << 16);
            const uint32_t accum = (lo_pass || ks > 0) ? 1u : 0u;
            if (elected) {
                umma2_f16(d_tile + skip, a_lo, b_lo, DESC_HI, IDESC0 | ((n0 >> 3) << 17), accum);
                if (n0 != np)      // columns [256, NT): the second piece follows the first's 16 n0 bytes
                    umma2_f16(d_tile + 256, a_lo, (b_addr_s + (uint32_t)((off + 16 * (int)n0) >> 4)) | ((256u >> 1) << 16), DESC_HI,
                              IDESC0 | ((256u >> 3) << 17), accum);
            }
            continue;
        }
        if (CG == 2) {  // per-CTA half image: sub-block of N'/2 rows, LBO = (N'/16) cores * 128 B (all immediates)
            const int half = ks / KSPS, sb = ks % KSPS;
            const int off = (half ? Cfg::CB0 : 0) + tc2_sub_off(NT, Cfg::TRI16, KSPS, half, sb);
            b_lo = (b_addr_s + (uint32_t)(off >> 4)) | ((np >> 1) << 16);
        } else {        // full stacked image: skip the leading row blocks
            b_lo = (b_addr_s + s2 * (((2 * NT / 8) * 128) >> 4) + (skip >> 3) * (128 >> 4)) | ((((NT / 8) * 128) >> 4) << 16);
        }
        const uint32_t idesc = IDESC0 | ((np >> 3) << 17);
        const uint32_t accum = (lo_pass || ks > 0) ? 1u : 0u;
        if (elected) {
            if (CG == 2) umma2_f16(d_tile + skip, a_lo, b_lo, DESC_HI, idesc, accum);
            else umma_f16(d_tile + skip, a_lo, b_lo, DESC_HI, idesc, accum);
            if (Cfg::A_TILE_BYTES != Cfg::A_COPY_BYTES && !lo_pass) {       // lo term of the pilots x hi term of the parameters
                if (CG == 2) umma2_f16(d_tile + skip, a_lo + (Cfg::A_COPY_BYTES >> 4), b_lo, DESC_HI, idesc, 1u);
                else umma_f16(d_tile + skip, a_lo + (Cfg::A_COPY_BYTES >> 4), b_lo, DESC_HI, idesc, 1u);
            }
        }
    }
}

__device__ __forceinline__ void tie_append(const unsigned char* bad, int* tie_buf, int64_t chunk_row);

// fused 'all' epilogue: a warp skips the LMMSE row of a component whose un-normalised weight is below this for all of its 32 pilots
// (the normaliser is >= 1, so the dropped terms are < TC_SKIP_THRESH each); measured: no effect on the speed up to 1e-9
constexpr float TC_SKIP_THRESH = 1e-30f;

// hi_a + lo_a > hi_b + lo_b, exactly (the FP64 sums of FP32 pairs are exact)
__device__ __noinline__ bool pair_greater_f64(float hi_a, float lo_a, float hi_b, float lo_b) {
    return ((double)hi_a + (double)lo_a) > ((double)hi_b + (double)lo_b);
}

// EPI selects the epilogue: 0 = fused 'all' estimate (online softmax), 1 = export the weighted log-probabilities l_k only (or, with
// TcArgs::top_out, keep only their running argmax: the top-1 label), 2 = combine with given per-pilot weights (the top-n /
// cumulative-probability modes run 1 -> select -> 2) or, with TcArgs::unit_comp, the single component of each work unit of pilots
// regrouped by label (top-1 on large batches: 1 -> bucket -> 2)
// KDC = n_obs / 16 (reduction length 32 KDC); NCHZ = 0 (no whitening columns: an H-part launch) or KDC; NCHH = H columns / 32
template <int KDC, int NCHZ, int NCHH, bool OFFS, int CG, int EPI, int ORDER, int AC>
__global__ void __launch_bounds__(NUM_THREADS, 1) dense_tc_kernel(const TcArgs a) {
    constexpr int NZ = 32 * NCHZ, NH = 32 * NCHH;
    constexpr int ACCB = tc_accb(EPI, 32 * KDC, NZ, NH, ORDER, AC);
    // (a second issuer warp, one per tile, was tried for this launch: the UTCHMMA issue of one thread is not the limit -- with two
    // issuers each spends as long issuing half as many MMAs, i.e. the issue stalls on the tensor pipe's queue -- and the launch got
    // 2 % slower: profiles/r02_whitening_notes.md)
    using Cfg = TcCfg<32 * KDC, NZ, NH, CG, ORDER, AC, ACCB>;
    constexpr int S = Cfg::STAGES;
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* sA = smem;
    constexpr int NTILES = Cfg::NTILES;
    unsigned char* sB = smem + NTILES * Cfg::A_TILE_BYTES;
    TcCtrl* ctrl = reinterpret_cast<TcCtrl*>(sB + S * Cfg::STAGE_BYTES);

    if (a.run_flag != nullptr && __ldg(a.run_flag) != a.run_flag_want) return;      // (uniform over the whole grid)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // work unit: CG * TILES tiles (256 pilots per CTA); the cluster (CG CTAs) walks the units round-robin
    const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
    int64_t n_units = (a.B + CG * NTILES * TILE_M - 1) / (CG * NTILES * TILE_M);
    // regrouped pilots (slot -> pilot through perm): one component per work unit (bucketed top-1, pair mode)
    const bool bucket = (EPI == 2) && a.unit_comp != nullptr;
    if (bucket) n_units = __ldg(a.n_units_dev);
    // components of a unit: (first, count)
    auto unit_comps = [&](int64_t unit, int& kb, int& nk) {
        kb = 0; nk = a.K;
        if (bucket) { kb = __ldg(a.unit_comp + unit); nk = 1; }
    };
    const int64_t unit0 = blockIdx.x / CG, unit_step = gridDim.x / CG;
    // the SM-pair variant is only launched for triangular Linv (the common, Cholesky case): its offsets are compile-time
    const int tri16 = (CG == 2) ? Cfg::TRI16 : (a.tri ? 16 : 0);

    if (threadIdx.x == 0) {
        // CG=2: the leader's "full" barriers also collect one remote arrival from the peer CTA ("my half has landed too")
        const uint32_t full_count = (CG == 2 && rank == 0) ? 2 : 1;
        for (int i = 0; i < S; ++i) { mbar_init(smem_u32(&ctrl->full[i]), full_count); mbar_init(smem_u32(&ctrl->empty[i]), 1); }
        for (int t = 0; t < 2 * TILES; ++t) {
            mbar_init(smem_u32(&ctrl->acc_full[t]), 1);
            mbar_init(smem_u32(&ctrl->acc_empty[t]), 4 * CG);       // one arrival per epilogue warp (of both CTAs)
        }
        mbar_init(smem_u32(&ctrl->a_full), full_count);
        mbar_init(smem_u32(&ctrl->a_free), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if (CG == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctrl->tmem_base)), "r"(Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctrl->tmem_base)), "r"(Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();       // barriers initialised in BOTH CTAs before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = ctrl->tmem_base;

    // register budget: the CTA owns 384 x 168 registers; 128 x 56 + 256 x 224 = 64512 redistributes exactly that pool
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 0 && lane == 0) {
            // ===================== bulk-TMA producer: NCHUNK chunks per component through the ring
            int stage = 0;
            uint32_t phase = 0;
            constexpr size_t COMP_BYTES = (CG == 2) ? (size_t)2 * Cfg::PASS_BYTES : (size_t)Cfg::COMP_HALFS * 2;
            const unsigned char* img = (CG == 2) ? a.image2 + (size_t)rank * COMP_BYTES : reinterpret_cast<const unsigned char*>(a.image);
            constexpr size_t COMP_STRIDE = COMP_BYTES * CG;      // CG=2: [k][rank]
            for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
                int kb, nk;
                unit_comps(unit, kb, nk);
                for (int ki = 0; ki < nk; ++ki) {
                    const int k = kb + ki;
                    const unsigned char* comp = img + (size_t)k * COMP_STRIDE;
                    #pragma unroll
                    for (int q = 0; q < Cfg::NCHUNK; ++q) {
                        mbar_wait(smem_u32(&ctrl->empty[stage]), phase ^ 1);
                        if constexpr (Cfg::KSLICED) {      // K-slices differ in length (triangular skip)
                            mbar_expect_tx(smem_u32(&ctrl->full[stage]), Cfg::chunk_bytes(q));
                            bulk_g2s(smem_u32(sB + stage * Cfg::STAGE_BYTES), comp + Cfg::chunk_off(q), Cfg::chunk_bytes(q), smem_u32(&ctrl->full[stage]));
                        } else {
                        mbar_expect_tx(smem_u32(&ctrl->full[stage]), Cfg::STAGE_BYTES);
                        bulk_g2s(smem_u32(sB + stage * Cfg::STAGE_BYTES), comp + (size_t)q * Cfg::STAGE_BYTES, Cfg::STAGE_BYTES,
                                 smem_u32(&ctrl->full[stage]));
                        }
                        if (++stage == S) { stage = 0; phase ^= 1; }
                    }
                }
            }
        } else if (warp == 3 && lane == 0) {
            // ===================== pilot-tile producer: the two pre-formatted 128-pilot tiles of each unit, one bulk copy each
            uint32_t fph = 0;
            for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
                mbar_wait(smem_u32(&ctrl->a_free), fph ^ 1);      // all MMAs of the previous unit have read the tiles
                fph ^= 1;
                mbar_expect_tx(smem_u32(&ctrl->a_full), NTILES * Cfg::A_TILE_BYTES);
                #pragma unroll
                for (int t = 0; t < NTILES; ++t)
                    bulk_g2s(smem_u32(sA + t * Cfg::A_TILE_BYTES),
                             reinterpret_cast<const unsigned char*>(a.a_img) + (size_t)((unit * CG + rank) * NTILES + t) * Cfg::A_TILE_BYTES,
                             Cfg::A_TILE_BYTES, smem_u32(&ctrl->a_full));
            }
        } else if (warp == 1 && rank == 0) {
            // ===================== MMA issuer (leader CTA).  The whole warp runs the loop (uniform control flow keeps the
            // descriptors in uniform registers); one elected lane issues.  Every instruction between two MMAs is exposed
            // latency, so descriptors are 32-bit base + compile-time immediate and barrier waits are kept to
            // NCHUNK + TILES per component.
            const bool elected = elect_one();
            constexpr int NT = Cfg::NT;
            constexpr uint32_t A_LBO = (TILE_M / 8) * 128;
            const uint32_t a_lo0 = ((smem_u32(sA) >> 4) & 0x3FFF) | ((A_LBO >> 4) << 16);
            const uint32_t b_addr0 = (smem_u32(sB) >> 4) & 0x3FFF;
            int stage0 = 0;                          // ring slot / parity of chunk 0 of the current component
            uint32_t phase0 = 0, a_phase = 0;
            uint32_t eph0 = 0, eph1 = 0;             // parity of acc_empty[t] waited on next
            uint32_t ephb = 0, accn = 0;             // ACCB = 2: parity bits per (tile, buffer), components issued so far
            long long w_empty = 0, w_full = 0, w_a = 0, t_begin = QCE_CLK();
            for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
                const long long ca = QCE_CLK();
                mbar_wait(smem_u32(&ctrl->a_full), a_phase);
                a_phase ^= 1;
                tc_fence_after();
                w_a += QCE_CLK() - ca;
                const int nk = bucket ? 1 : a.K;
                for (int k = 0; k < nk; ++k) {
                    if (ORDER == 0) {
                    #pragma unroll
                    for (int t = 0; t < NTILES; ++t) {
                        // the first MMA overwrites the accumulator: the epilogue must have drained component k-1
                        long long c0 = QCE_CLK();
                        uint32_t ai = t;                        // accumulator of this (tile, component)
                        if (ACCB == 2) {
                            ai = t * 2 + (accn & 1u);
                            mbar_wait(smem_u32(&ctrl->acc_empty[0]) + 8u * ai, ((ephb >> ai) & 1u) ^ 1u);
                            ephb ^= 1u << ai;
                        } else if (t == 0) { mbar_wait(smem_u32(&ctrl->acc_empty[0]), eph0 ^ 1); eph0 ^= 1; }
                        else { mbar_wait(smem_u32(&ctrl->acc_empty[1]), eph1 ^ 1); eph1 ^= 1; }
                        tc_fence_after();
                        w_empty += QCE_CLK() - c0;
                        const uint32_t d_tile = tmem_base + ai * NT;
                        const uint32_t a_lo_t = a_lo0 + t * (Cfg::A_TILE_BYTES >> 4);
                        int stage = stage0;
                        uint32_t phase = phase0;
                        #pragma unroll
                        for (int q = 0; q < Cfg::NCHUNK; ++q) {
                            if (t == 0) {
                                c0 = QCE_CLK();
                                mbar_wait(smem_u32(&ctrl->full[stage]), phase);
                                tc_fence_after();
                                w_full += QCE_CLK() - c0;
                            }
                            tc_issue_chunk<Cfg, CG>(q, d_tile, a_lo_t, b_addr0 + stage * (Cfg::STAGE_BYTES >> 4), tri16, elected);
                            if (t == NTILES - 1 && elected) { if (CG == 2) tc_commit2(smem_u32(&ctrl->empty[stage])); else tc_commit(smem_u32(&ctrl->empty[stage])); }
                            if (++stage == S) { stage = 0; phase ^= 1; }
                        }
                        if (elected) { if (CG == 2) tc_commit2(smem_u32(&ctrl->acc_full[0]) + 8u * ai); else tc_commit(smem_u32(&ctrl->acc_full[0]) + 8u * ai); }
                        __syncwarp();
                        if (t == NTILES - 1) { stage0 = stage; phase0 = phase; }
                    }
                    ++accn;
                    } else {
                    // chunk-major: a chunk feeds both tiles and is released at once
                    #pragma unroll
                    for (int q = 0; q < Cfg::NCHUNK; ++q) {
                        long long c0 = QCE_CLK();
                        mbar_wait(smem_u32(&ctrl->full[stage0]), phase0);
                        tc_fence_after();
                        w_full += QCE_CLK() - c0;
                        #pragma unroll
                        for (int t = 0; t < NTILES; ++t) {
                            if (q == 0) {
                                c0 = QCE_CLK();
                                if (t == 0) { mbar_wait(smem_u32(&ctrl->acc_empty[0]), eph0 ^ 1); eph0 ^= 1; }
                                else { mbar_wait(smem_u32(&ctrl->acc_empty[1]), eph1 ^ 1); eph1 ^= 1; }
                                tc_fence_after();
                                w_empty += QCE_CLK() - c0;
                            }
                            tc_issue_chunk<Cfg, CG>(q, tmem_base + t * NT, a_lo0 + t * (Cfg::A_TILE_BYTES >> 4),
                                                    b_addr0 + stage0 * (Cfg::STAGE_BYTES >> 4), tri16, elected);
                            if (q == Cfg::NCHUNK - 1 && elected) { if (CG == 2) tc_commit2(smem_u32(&ctrl->acc_full[t])); else tc_commit(smem_u32(&ctrl->acc_full[t])); }
                        }
                        if (elected) { if (CG == 2) tc_commit2(smem_u32(&ctrl->empty[stage0])); else tc_commit(smem_u32(&ctrl->empty[stage0])); }
                        __syncwarp();
                        if (++stage0 == S) { stage0 = 0; phase0 ^= 1; }
                    }
                    }
                }
                if (elected) { if (CG == 2) tc_commit2(smem_u32(&ctrl->a_free)); else tc_commit(smem_u32(&ctrl->a_free)); }
                __syncwarp();
            }
            if (a.prof && blockIdx.x == 0 && elected) { a.prof[0] = QCE_CLK() - t_begin; a.prof[1] = w_empty; a.prof[2] = w_full; a.prof[3] = w_a; }
        } else if (CG == 2 && warp == 1 && lane == 0 && rank == 1) {
            // ===================== relay (peer CTA): when this CTA's tiles / chunk have landed, arrive on the LEADER's barrier
            int stage = 0;
            uint32_t phase = 0, a_phase = 0;
            for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
                mbar_wait(smem_u32(&ctrl->a_full), a_phase);
                a_phase ^= 1;
                mbar_arrive_cluster(smem_u32(&ctrl->a_full), 0);
                const int nk = bucket ? 1 : a.K;
                for (int k = 0; k < nk; ++k) {
                    #pragma unroll
                    for (int q = 0; q < Cfg::NCHUNK; ++q) {
                        mbar_wait(smem_u32(&ctrl->full[stage]), phase);
                        mbar_arrive_cluster(smem_u32(&ctrl->full[stage]), 0);
                        if (++stage == S) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
        // ===================== epilogue warpgroups: one thread per pilot
        const int t = (warp - 4) >> 2;                 // tile within the pair
        const int wq = warp & 3;                       // TMEM lane quadrant of this warp
        const int row = wq * 32 + lane;
        const uint32_t tz = tmem_base + ((uint32_t)(wq * 32) << 16) + t * ACCB * (NZ + NH);
        const uint32_t th = tz + NZ;
        uint32_t fph = 0;                              // parity of acc_full (one bit per accumulator buffer of this tile)
        uint32_t accn = 0;                             // components drained so far (ACCB = 2: buffer = accn & 1)
        const int N = a.N;
        double err = 0.0, pw = 0.0, cnt = 0.0;     // cnt also gates the atomics (rows handled by this thread)
        long long w_acc = 0, c_z = 0, c_h = 0, c_pro = 0, c_ld = 0;

        for (int64_t unit = unit0; unit < n_units && t < NTILES; unit += unit_step) {
            const int64_t tile_base = ((unit * CG + rank) * NTILES + t) * TILE_M;
            long long c0 = QCE_CLK();

            float2 acc[NH > 0 ? NH / 2 : 1];           // the estimate row, (re, im) pairs: packed FFMA2 arithmetic
            #pragma unroll
            for (int j = 0; j < NH / 2; ++j) acc[j] = make_float2(0.f, 0.f);
            float mref_hi = 0.f, mref_lo = 0.f;
            float ssum = 0.f;
            float best_hi = -INFINITY, best_lo = 0.f;  // EPI=1 label mode: running maximum of l_k as an FP32 pair
            float best_q = 0.f;                        // quadratic form of the best component (the FP32 error of l grows with it)
            float second = -INFINITY;                  // ... and the runner-up (rounded): the selection is re-evaluated in complex128
            int best_k = 0;                            // when the two are closer than the FP32 log-likelihoods can tell apart

            // the pilot this thread handles, and the components of this unit
            int64_t src = tile_base + row;
            bool valid = src < a.B;
            int kb, nk;
            unit_comps(unit, kb, nk);
            if (bucket) {
                src = __ldg(a.perm + tile_base + row);
                valid = src >= 0;
            }
            int k_n = kb;                              // the component of the next iteration (its scalars are fetched one ahead)
            float zs_n = __ldg(a.zscale + k_n), hs_n = __ldg(a.hscale + k_n);
            float2 lc_n = __ldg(a.logc2 + k_n);
            const int64_t grow = valid ? src : 0;     // rows past the end read row 0, never write
            float w_n = 0.f;
            if (EPI == 2) {
                if (bucket) w_n = valid ? (a.slot_w ? __ldg(a.slot_w + tile_base + row) : 1.f) : 0.f;
                else w_n = __ldg(a.w_in + grow * a.K);
            }
            for (int ki = 0; ki < nk; ++ki) {
                const int k = k_n;
                // per-component scalars were fetched one iteration ahead (their L2 latency would otherwise sit on the
                // critical path between "accumulator ready" and "accumulator released")
                const float zs = zs_n, hs = hs_n;
                const float2 lc = lc_n;
                const float w_k = w_n;
                if (ki + 1 < nk) {
                    k_n = k + 1;
                    zs_n = __ldg(a.zscale + k_n); hs_n = __ldg(a.hscale + k_n); lc_n = __ldg(a.logc2 + k_n);
                    if (EPI == 2) w_n = __ldg(a.w_in + grow * a.K + k_n);
                }
                // ---- whitened residual -> quadratic form
                c0 = QCE_CLK();
                const uint32_t ab = (ACCB == 2) ? (accn & 1u) : 0u;
                const uint32_t ai = t * ACCB + ab;
                ++accn;
                mbar_wait(smem_u32(&ctrl->acc_full[0]) + 8u * ai, (fph >> ab) & 1u);
                fph ^= 1u << ab;
                const uint32_t tzk = tz + ab * (NZ + NH), thk = th + ab * (NZ + NH);
                tc_fence_after();
                long long c1 = QCE_CLK();
                w_acc += c1 - c0;
                float va[32], vb[32];
                float p;
                // whitening-only launch with at most 128 whitened columns: the whole row fits in registers (there is no estimate row to
                // keep), so it is fetched at once and the accumulator is handed back to the tensor core BEFORE the arithmetic
                constexpr bool EARLY = (EPI == 1 && NCHZ <= 4);
                float vall[EARLY ? NCHZ : 1][32];
                if (EPI != 2) {
                float q_hi = 0.f, q_lo = 0.f;        // quadratic form as an unevaluated FP32 pair (TwoSum accumulation)
                if (EARLY) {
                    #pragma unroll
                    for (int ch = 0; ch < NCHZ; ++ch) tmem_ld32(tzk + ch * 32, vall[EARLY ? ch : 0]);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (CG == 2) mbar_arrive_cluster(smem_u32(&ctrl->acc_empty[0]) + 8u * ai, 0); else mbar_arrive(smem_u32(&ctrl->acc_empty[0]) + 8u * ai);
                    }
                } else {
                // TMEM loads are double-buffered: chunk ch+1 (and finally the first H chunk) is in flight while chunk ch is
                // reduced, so their latency stays off the accumulator-release critical path
                tmem_ld32(tzk, va);
                tmem_ld_wait();
                }
                #pragma unroll
                for (int ch = 0; ch < NCHZ; ++ch) {
                    float (&v)[32] = EARLY ? vall[EARLY ? ch : 0] : ((ch & 1) ? vb : va);
                    float (&vn)[32] = (ch & 1) ? va : vb;
                    if (!EARLY) { if (ch + 1 < NCHZ) tmem_ld32(tzk + (ch + 1) * 32, vn); else if (EPI == 0 || EPI == 3) tmem_ld32(thk, vn); }
                    #pragma unroll
                    for (int g16 = 0; g16 < 2; ++g16) {
                        float2 s0 = make_float2(0.f, 0.f), s1 = s0;
                        #pragma unroll
                        for (int u = 0; u < 8; u += 2) {
                            float2 z0 = make_float2(v[g16 * 16 + 2 * u], v[g16 * 16 + 2 * u + 1]);
                            float2 z1 = make_float2(v[g16 * 16 + 2 * u + 2], v[g16 * 16 + 2 * u + 3]);
                            if (OFFS) {
                                const float2* zo = reinterpret_cast<const float2*>(a.zoff + (size_t)k * NZ + ch * 32 + g16 * 16 + 2 * u);
                                const float2 o0 = __ldg(zo), o1 = __ldg(zo + 1);
                                z0 = __ffma2_rn(z0, make_float2(zs, zs), make_float2(-o0.x, -o0.y));
                                z1 = __ffma2_rn(z1, make_float2(zs, zs), make_float2(-o1.x, -o1.y));
                            }
                            s0 = __ffma2_rn(z0, z0, s0);
                            s1 = __ffma2_rn(z1, z1, s1);
                        }
                        {   // q += (16 squares) without losing the rounding error (Knuth TwoSum, FP32 only)
                            const float g = (s0.x + s0.y) + (s1.x + s1.y);
                            const float tt = q_hi + g;
                            const float bp = tt - q_hi;
                            q_lo += (q_hi - (tt - bp)) + (g - bp);
                            q_hi = tt;
                        }
                    }
                    if (!EARLY) tmem_ld_wait();
                }
                if (!OFFS) { const float zs2 = zs * zs; q_hi *= zs2; q_lo *= zs2; }   // power of two: exact
                // l = logc - q as a pair: hi part plus the exact rounding error of the subtraction
                const float l_hi = lc.x - q_hi;
                const float bq = l_hi - lc.x;
                const float l_lo = ((lc.x - (l_hi - bq)) + (-q_hi - bq)) + (lc.y - q_lo);
                if (EPI == 1 || EPI == 3) {
                    if (EPI == 3 || a.top_out) {
                        // top-1 label only.  tc_select_kernel compares the FP64 sums hi + lo; the same decision in FP32 (FP64
                        // arithmetic next to the saturated tensor pipe cost 18 % of this launch): the difference of the pairs,
                        // with the exact FP64 comparison only where its rounding error could change the sign
                        const float d_hi = l_hi - best_hi, d_lo = l_lo - best_lo;
                        const float d = d_hi + d_lo;
                        const bool safe = fabsf(d) > 4.8e-7f * (fabsf(d_hi) + fabsf(d_lo));               // 2^-21 > the 3 x 2^-24 rounding bound
                        bool better = d > 0.f;
                        // ties, NaN, infinities, the first component: rare, and behind a warp-uniform branch and a call so that the
                        // compiler cannot turn the FP64 comparison into unconditional arithmetic + select
                        if (__any_sync(0xffffffffu, !safe)) { if (!safe) better = pair_greater_f64(l_hi, l_lo, best_hi, best_lo); }
                        if (better) { second = best_hi + best_lo; best_hi = l_hi; best_lo = l_lo; best_k = k; best_q = q_hi; }
                        else second = fmaxf(second, l_hi + l_lo);
                        p = 0.f;
                        if (EPI == 3 && better) {      // fused hard selection: the estimate row restarts with this component's LMMSE row
                            p = 1.f;
                            #pragma unroll
                            for (int j = 0; j < NH / 2; ++j) acc[j] = make_float2(0.f, 0.f);
                        }
                    } else {
                        if (tile_base + row < a.B) a.lp_out[(tile_base + row) * a.K + k] = make_float2(l_hi, l_lo);
                        p = 0.f;
                    }
                } else {
                // ---- lazily rescaled online softmax (reference maximum moves only on jumps > 8)
                if (ki == 0) {
                    mref_hi = l_hi; mref_lo = l_lo; p = 1.f; ssum = 1.f;
                } else {
                    float df = (l_hi - mref_hi) + (l_lo - mref_lo);
                    if (df > 8.f) {
                        const float sc = __expf(-df);
                        ssum *= sc;
                        #pragma unroll
                        for (int j = 0; j < NH / 2; ++j) acc[j] = __fmul2_rn(acc[j], make_float2(sc, sc));
                        mref_hi = l_hi; mref_lo = l_lo;
                        df = 0.f;
                    }
                    p = __expf(df);
                    ssum += p;
                }
                }
                } else {
                    p = w_k;                         // given weight; the first H chunk has to be fetched here
                    if (__any_sync(0xffffffffu, p != 0.f)) { tmem_ld32(thk, (NCHZ & 1) ? vb : va); tmem_ld_wait(); }
                }
                long long c2 = QCE_CLK();
                c_z += c2 - c1;
                // ---- LMMSE row, weighted accumulation (the first H chunk is already in registers)
                if (EPI != 1) {
                    const bool any = __any_sync(0xffffffffu, (EPI == 2) ? (p != 0.f) : (p > TC_SKIP_THRESH));
                    const float2 ph = make_float2(p * hs, p * hs);
                    #pragma unroll
                    for (int ch = 0; ch < NCHH; ++ch) {
                        float (&v)[32] = ((NCHZ + ch) & 1) ? vb : va;
                        float (&vn)[32] = ((NCHZ + ch) & 1) ? va : vb;
                        if (ch + 1 < NCHH && any) tmem_ld32(thk + (ch + 1) * 32, vn);
                        if (any) {
                            #pragma unroll
                            for (int u = 0; u < 16; ++u) {
                                acc[ch * 16 + u] = __ffma2_rn(ph, make_float2(v[2 * u], v[2 * u + 1]), acc[ch * 16 + u]);
                                if (OFFS) {
                                    const float2 ho = __ldg(reinterpret_cast<const float2*>(a.hoff + (size_t)k * a.h_stride + a.h_col0 + ch * 32 + 2 * u));
                                    acc[ch * 16 + u] = __ffma2_rn(make_float2(p, p), ho, acc[ch * 16 + u]);
                                }
                            }
                        }
                        tmem_ld_wait();
                    }
                }
                if (!EARLY) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {        // one arrival per warp on the LEADER's barrier
                    if (CG == 2) mbar_arrive_cluster(smem_u32(&ctrl->acc_empty[0]) + 8u * ai, 0); else mbar_arrive(smem_u32(&ctrl->acc_empty[0]) + 8u * ai);
                }
                }
                c_h += QCE_CLK() - c2;
            }

            // ---- finalise: normalise, write the estimate row, NMSE accumulators (FP32 per row: FP64 stalls behind the
            // tensor pipe; the per-row sums enter the FP64 accumulators once)
            const int64_t g = src;
            bool hard_tie = false;          // EPI = 3: this pilot's selection is too close to call -- the exact path answers it
            if (EPI == 3 && valid && a.tie_buf) {
                const float gap = (best_hi - second) + best_lo;
                hard_tie = !(gap > a.tie_eps * fmaxf(1.f, best_q * a.inv_nobs));
                // MFA argmax-of-exp quirk (label 0 when every exp(l_k) underflows): anything near or below the underflow edge is exact-path work
                if ((a.top_flags & QCE_FLAG_TOP1_EXP_ARGMAX) && !(best_hi > -745.f)) hard_tie = true;
                if (hard_tie) tie_append(a.bad, a.tie_buf, g);
            }
            if (EPI == 1 && a.top_out && valid) {
                if ((a.top_flags & QCE_FLAG_TOP1_EXP_ARGMAX) && exp((double)best_hi + (double)best_lo) == 0.0) best_k = 0;
                a.top_out[g] = best_k;
                // too close to call (or NaN), or on the edge of the exp() underflow the MFA argmax quirk tests: the pilot goes on the
                // tie list and tc_refine_kernel decides in complex128 before the labels are used
                const float gap = (best_hi - second) + best_lo;
                bool tie = !(gap > a.tie_eps * fmaxf(1.f, best_q * a.inv_nobs));
                if ((a.top_flags & QCE_FLAG_TOP1_EXP_ARGMAX) && fabsf(best_hi + 745.1332f) < 0.01f) tie = true;
                if (tie) tie_append(a.bad, a.tie_buf, g);
            }
            if (EPI != 1 && valid && !hard_tie && __ldg(a.bad + g) == 0) {
                const float invs = (EPI == 2 || EPI == 3) ? 1.f : 1.f / ssum;
                if (EPI == 2 && a.slot_w) {      // pair mode: this slot's weighted row is one of several addends of the pilot's estimate:
                    // vector reductions (4 floats each) into the FP32 row of the pilot; tc_pair_finish_kernel writes the estimate
                    float4* out = reinterpret_cast<float4*>(a.pair_acc + (size_t)g * 2 * N + a.h_col0);
                    #pragma unroll
                    for (int j = 0; j < NH / 4; ++j) atomicAdd(out + j, make_float4(acc[2 * j].x, acc[2 * j].y, acc[2 * j + 1].x, acc[2 * j + 1].y));
                } else {
                if (a.h_est) {
                    // 256-bit stores (sm_100: st.global.v4.f64): every lane writes whole 32-byte sectors of its own row, and half as many
                    // stores wait for the register pair of the previous conversion to be read (the F2F -> STG chain was 83 % of the
                    // one-component combine launch, profiles/r02_whitening_notes.md).  Rows are 32-byte aligned (N is a multiple of 2).
                    // (caller's buffers that are only 16-byte aligned take the 128-bit form)
                    double2* out = a.h_est + g * N + (a.h_col0 >> 1);
                    if (a.wide_io) {
                        #pragma unroll
                        for (int j = 0; j < NH / 2; j += 2)
                            asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(out + j), "d"((double)(acc[j].x * invs)), "d"((double)(acc[j].y * invs)),
                                         "d"((double)(acc[j + 1].x * invs)), "d"((double)(acc[j + 1].y * invs)) : "memory");
                    } else {
                        #pragma unroll
                        for (int j = 0; j < NH / 2; ++j) out[j] = make_double2((double)(acc[j].x * invs), (double)(acc[j].y * invs));
                    }
                }
                if (a.acc && a.h_true) {
                    float errf = 0.f, pwf = 0.f;
                    auto nmse_term = [&](const int j, const float hx, const float hy) {
                        const float dx = acc[j].x * invs - hx, dy = acc[j].y * invs - hy;
                        errf = fmaf(dx, dx, fmaf(dy, dy, errf));
                        pwf = fmaf(hx, hx, fmaf(hy, hy, pwf));
                    };
                    // the true channel row of this pilot, 32 bytes (whole sectors) per load: 256-bit loads as for the stores above
                    if (!a.wide_io) {
                        #pragma unroll
                        for (int j = 0; j < NH / 2; ++j) {      // full unroll: acc[] must stay in registers
                            if (a.h_true_c64) {
                                const float2 h = reinterpret_cast<const float2*>(a.h_true)[g * N + (a.h_col0 >> 1) + j];
                                nmse_term(j, h.x, h.y);
                            } else {
                                const double2 hd = reinterpret_cast<const double2*>(a.h_true)[g * N + (a.h_col0 >> 1) + j];
                                nmse_term(j, (float)hd.x, (float)hd.y);
                            }
                        }
                    } else if (a.h_true_c64) {
                        const float2* ht = reinterpret_cast<const float2*>(a.h_true) + g * N + (a.h_col0 >> 1);
                        #pragma unroll
                        for (int j = 0; j < NH / 2; j += 4) {
                            float h0, h1, h2, h3, h4, h5, h6, h7;
                            asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                                         : "=f"(h0), "=f"(h1), "=f"(h2), "=f"(h3), "=f"(h4), "=f"(h5), "=f"(h6), "=f"(h7) : "l"(ht + j));
                            nmse_term(j, h0, h1); nmse_term(j + 1, h2, h3); nmse_term(j + 2, h4, h5); nmse_term(j + 3, h6, h7);
                        }
                    } else {
                        const double2* ht = reinterpret_cast<const double2*>(a.h_true) + g * N + (a.h_col0 >> 1);
                        #pragma unroll
                        for (int j = 0; j < NH / 2; j += 2) {
                            double d0, d1, d2, d3;
                            asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(d0), "=d"(d1), "=d"(d2), "=d"(d3) : "l"(ht + j));
                            nmse_term(j, (float)d0, (float)d1); nmse_term(j + 1, (float)d2, (float)d3);
                        }
                    }
                    err += (double)errf;
                    pw += (double)pwf;
                }
                cnt += 1.0;
                }
            }
        }
        if (a.prof && blockIdx.x == 0 && lane == 0 && wq == 0) {
            a.prof[4 + t * 4 + 0] = w_acc; a.prof[4 + t * 4 + 1] = c_z; a.prof[4 + t * 4 + 2] = c_h; a.prof[4 + t * 4 + 3] = c_pro; a.prof[12 + t] = c_ld;
        }
        if (a.acc) {
            #pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                err += __shfl_xor_sync(0xffffffffu, err, off);
                pw += __shfl_xor_sync(0xffffffffu, pw, off);
                cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
            }
            if (lane == 0 && cnt > 0.0) {
                atomicAdd(a.acc + 0, err);
                atomicAdd(a.acc + 1, pw);
                if (a.count_rows) atomicAdd(a.acc + 2, cnt);
            }
        }
    }

    __syncwarp();                                                // single-lane roles rejoin their warp before the block-wide barriers
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();       // the peer's smem / TMEM stay valid until every MMA has retired
    if (warp == 2) {
        tc_fence_after();
        if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ parameter packing
// One block per (component, matrix).  Power-of-two scale putting the largest entry in [2^12, 2^13), then the FP16
// hi/lo terms of the real 2x2-block embedding, written into the component's stacked image [E(Linv); E(W)]
// ((2No + 2N) rows x 2No) in the canonical K-major core-matrix layout: core (nb, kb) at ((kb * NT/8) + nb) * 128 B,
// hi image then lo image.  flags[1] is raised if some Linv_k is not lower triangular.
__global__ void __launch_bounds__(256) tc_pack_kernel(const double2* __restrict__ Linv, const double2* __restrict__ W, int No, int N,
                                                      double data_scale, __half* __restrict__ image, float* __restrict__ zscale,
                                                      float* __restrict__ hscale, int* __restrict__ flags) {
    const int k = blockIdx.x >> 1, which = blockIdx.x & 1;
    const int R = which ? N : No, C = No;
    const double2* src = which ? W + (size_t)k * N * No : Linv + (size_t)k * No * No;
    __shared__ double smax[256];
    double mx = 0.0;
    int upper = 0;
    for (int i = threadIdx.x; i < R * C; i += 256) {
        const double2 v = src[i];
        mx = fmax(mx, fmax(fabs(v.x), fabs(v.y)));
        if (!which && (i % C) > (i / C) && (v.x != 0.0 || v.y != 0.0)) upper = 1;
    }
    if (upper) atomicOr(flags + 1, 1);
    smax[threadIdx.x] = mx;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) smax[threadIdx.x] = fmax(smax[threadIdx.x], smax[threadIdx.x + s]);
        __syncthreads();
    }
    mx = smax[0] * data_scale;
    int ex = 0;
    if (mx > 0.0 && isfinite(mx)) frexp(mx, &ex);          // mx = f * 2^ex, f in [0.5, 1)
    const int e = (mx > 0.0 && isfinite(mx)) ? 13 - ex : 0;
    const double sc = ldexp(data_scale, e);
    if (threadIdx.x == 0) (which ? hscale : zscale)[k] = (float)ldexp(1.0, -e);
    if (!image) return;                                    // split path: only the scales and the triangular flag are needed
    const int ncols = 2 * R, kd = 2 * No, nt = 2 * No + 2 * N;
    __half* hi = image + (size_t)k * 2 * nt * kd;
    __half* lo = hi + (size_t)nt * kd;
    const int nbs = ncols / 8, nb0 = which ? (2 * No) / 8 : 0;
    for (int idx = threadIdx.x; idx < ncols * kd; idx += 256) {
        const int core = idx >> 6, within = idx & 63;
        const int nb = core % nbs, kb = core / nbs;
        const int n = nb * 8 + (within >> 3), kk = kb * 8 + (within & 7);
        const double2 v = src[(size_t)(n >> 1) * C + (kk >> 1)];
        const int aa = n & 1, bb = kk & 1;
        const double x = (aa == bb ? v.x : (aa ? v.y : -v.y)) * sc;
        const __half h = __double2half(x);
        const size_t dst = ((size_t)kb * (nt / 8) + nb0 + nb) * 64 + within;
        hi[dst] = h;
        lo[dst] = __double2half(x - (double)__half2float(h));
    }
}

// CG=2 operand images (layout: see tc2_nprime / tc2_sub_off).  One block per (component, rank); the power-of-two scales
// were fixed by tc_pack_kernel.  The stacked operand consists of the first nz rows of E(Linv_k) (nz = 0 or 2No) followed by
// the rows [h0, h0 + nh) of E(W_k): the fused launch uses (2No, 0, 2N), the split launches (2No, -, 0) and (0, h0, nh).
__global__ void __launch_bounds__(256) tc2_pack_kernel(const double2* __restrict__ Linv, const double2* __restrict__ W, int No, int N,
                                                       double data_scale, const float* __restrict__ zscale, const float* __restrict__ hscale,
                                                       int tri16, int nz, int h0, int nh, unsigned char* __restrict__ image2) {
    const int k = blockIdx.x >> 1, rank = blockIdx.x & 1;
    const int kd = 2 * No, nt = nz + nh, ksps = kd / 32;
    const double scz = data_scale / (double)zscale[k], sch = data_scale / (double)hscale[k];
    const int cb0 = tc2_chunk_bytes(nt, tri16, ksps, 0), cb1 = tc2_chunk_bytes(nt, tri16, ksps, 1);
    unsigned char* base = image2 + ((size_t)k * 2 + rank) * (size_t)(2 * (cb0 + cb1));
    for (int half = 0; half < 2; ++half) {
        for (int s2 = 0; s2 < ksps; ++s2) {
            const int ks = half * ksps + s2;
            const int np = tc2_nprime(nt, tri16, ks), w0 = tc2_piece0(np);
            __half* hi = reinterpret_cast<__half*>(base + (half ? cb0 : 0) + tc2_sub_off(nt, tri16, ksps, half, s2));
            __half* lo = reinterpret_cast<__half*>(reinterpret_cast<unsigned char*>(hi) + (cb0 + cb1));
            for (int idx = threadIdx.x; idx < np * 8; idx += 256) {
                // MMA piece (one unless N' > 256): its width, first stacked row and the index within its per-rank block
                const bool p1 = idx >= w0 * 8;
                const int rows = (p1 ? np - w0 : w0) / 2, li = p1 ? idx - w0 * 8 : idx;
                const int n0 = (p1 ? tri16 * ks + w0 : tri16 * ks) + rank * rows;      // first stacked row of the piece held by this rank
                const int core = li >> 6, within = li & 63;                // core = kc * (rows/8) + nb
                const int nb = core % (rows / 8), kc = core / (rows / 8);
                const int n = n0 + nb * 8 + (within >> 3), kk = ks * 16 + kc * 8 + (within & 7);
                const bool isz = n < nz;
                const int rrow = isz ? n : h0 + n - nz;
                const double2 v = isz ? Linv[((size_t)k * No + (rrow >> 1)) * No + (kk >> 1)] : W[((size_t)k * N + (rrow >> 1)) * No + (kk >> 1)];
                const int aa = rrow & 1, bb = kk & 1;
                const double x = (aa == bb ? v.x : (aa ? v.y : -v.y)) * (isz ? scz : sch);
                const __half h = __double2half(x);
                hi[idx] = h;
                lo[idx] = __double2half(x - (double)__half2float(h));
            }
        }
    }
}

__global__ void tc_pack_small_kernel(const double2* __restrict__ zoff, const double2* __restrict__ hoff, const double* __restrict__ logc,
                                     int K, int No, int N, float* __restrict__ zoff_f, float* __restrict__ hoff_f,
                                     float2* __restrict__ logc2, int* __restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int nz = 0;
    if (i < K) logc2[i] = tc_logc_pair(logc[i]);
    if (i < K * No) { const double2 v = zoff[i]; zoff_f[2 * i] = (float)v.x; zoff_f[2 * i + 1] = (float)v.y; nz |= (v.x != 0.0 || v.y != 0.0); }
    if (i < K * N) { const double2 v = hoff[i]; hoff_f[2 * i] = (float)v.x; hoff_f[2 * i + 1] = (float)v.y; nz |= (v.x != 0.0 || v.y != 0.0); }
    if (nz) atomicOr(flags, 1);
}

// ------------------------------------------------------------------------------------------------ pilot tiles
// HBM-bound formatter: pilots -> exact FP16 integers m = r / data_scale, written as 128-pilot tiles in the canonical
// K-major core-matrix layout the MMA A-descriptor expects (core (mb, kb) at ((kb * 16) + mb) * 128 B), so that the
// estimate kernel stages a tile with ONE contiguous bulk copy.  One CTA per (tile, 8-row block): warp w reads pilot row w of
// the block in full (lane-contiguous elements: whole 128-byte lines per warp-load -- a first version in which every warp-load touched
// 8 rows x 32..64 B ran at 98 % L1TEX throughput and 59 % of DRAM), the formatted halves go through a 2..4 KB shared-memory
// image of the block's core matrices, and every warp then writes whole 128-byte core matrices.
// OBSERVE = true fuses get_observation_nbit + quant (modules/utils.py:241-251, :189-203) in front: y = h + s*n with
// two roundings, then the same sign / digitize decisions as quantize_kernel (bit-exact), then the level's grid index.
// SPLIT = true: arbitrary real data, written as the FP16 pair (hi, lo) of m = r / eff_scale into two consecutive tile images.
template <bool OBSERVE, bool H_C64, bool SPLIT>
__global__ void __launch_bounds__(256) tc_format_kernel(const void* __restrict__ src, const double2* __restrict__ noise, double noise_scale,
                                                        QuantTables qt, int64_t B, int No, double inv_data_scale,
                                                        __half* __restrict__ img, unsigned char* __restrict__ bad, int* __restrict__ fix_buf) {
    extern __shared__ __align__(16) unsigned char s_dyn[];   // [copies][kbs][8 rows][16 B] core matrices of this block, then thr / labels (f64)
    __shared__ int s_bad[8];
    const int KD = 2 * No, kbs = KD / 8;
    const int64_t tile = blockIdx.x / (TILE_M / 8);
    const int mb = blockIdx.x % (TILE_M / 8);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int COPIES = SPLIT ? 2 : 1;
    unsigned char* s_img = s_dyn;
    double* s_tab = reinterpret_cast<double*>(s_dyn + (size_t)COPIES * kbs * 128);
    if (OBSERVE && qt.n_bits > 1) {
        for (int i = threadIdx.x; i < 2 * qt.n_thr + 1; i += blockDim.x) s_tab[i] = (i < qt.n_thr) ? qt.thr[i] : qt.labels[i - qt.n_thr];
    }
    if (threadIdx.x < 8) s_bad[threadIdx.x] = 0;
    __syncthreads();
    const int64_t g = tile * TILE_M + mb * 8 + warp;           // this warp's pilot
    int my_bad = 0;
    uint32_t hbits[2] = {0u, 0u};                              // 1-bit observe path: the packed FP16 pair of an element
    for (int j0 = 0; j0 < No; j0 += 64) {                       // complex elements j0 + lane and j0 + 32 + lane of the row: every
        double2 v[2] = {make_double2(0.0, 0.0), make_double2(0.0, 0.0)};     // warp-load covers 256 / 512 contiguous bytes
        const int ja = j0 + lane, jb = j0 + 32 + lane;
        const bool oa = g < B && ja < No, ob = g < B && jb < No;
        if (OBSERVE) {
            double2 h[2] = {make_double2(0.0, 0.0), make_double2(0.0, 0.0)}, w[2] = {make_double2(0.0, 0.0), make_double2(0.0, 0.0)};
            if (H_C64) {
                if (oa) { const float2 hf = __ldcs(reinterpret_cast<const float2*>(src) + g * No + ja); h[0] = make_double2((double)hf.x, (double)hf.y); }
                if (ob) { const float2 hf = __ldcs(reinterpret_cast<const float2*>(src) + g * No + jb); h[1] = make_double2((double)hf.x, (double)hf.y); }
            } else {
                if (oa) h[0] = __ldcs(reinterpret_cast<const double2*>(src) + g * No + ja);
                if (ob) h[1] = __ldcs(reinterpret_cast<const double2*>(src) + g * No + jb);
            }
            if (oa) w[0] = __ldcs(noise + g * No + ja);
            if (ob) w[1] = __ldcs(noise + g * No + jb);
            hbits[0] = hbits[1] = 0u;
            #pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (!(u ? ob : oa)) continue;
                const double yx = __dadd_rn(h[u].x, __dmul_rn(noise_scale, w[u].x)), yy = __dadd_rn(h[u].y, __dmul_rn(noise_scale, w[u].y));
                if (qt.n_bits == 1 && !SPLIT) {
                    // value on the grid is sign(y) (x 1/sqrt(2) = data_scale): the FP16 bit patterns of +-1 / 0 directly -- no double
                    // selects, conversions or grid check (the formatter is issue-bound: ALU 61 %, XU 29 % in profiles/r02_format_ncu_summary.txt)
                    const uint32_t hx = yx > 0.0 ? 0x3C00u : (yx < 0.0 ? 0xBC00u : 0u), hy = yy > 0.0 ? 0x3C00u : (yy < 0.0 ? 0xBC00u : 0u);
                    if (yx != yx || yy != yy) my_bad = 1;          // NaN data: the row goes to the complex128 kernel
                    hbits[u] = hx | (hy << 16);
                } else if (qt.n_bits == 1) {
                    v[u].x = (yx > 0.0) ? 1.0 : ((yx < 0.0) ? -1.0 : ((yx == 0.0) ? 0.0 : yx));
                    v[u].y = (yy > 0.0) ? 1.0 : ((yy < 0.0) ? -1.0 : ((yy == 0.0) ? 0.0 : yy));
                } else {
                    const double* thr = s_tab;
                    const double* lab = s_tab + qt.n_thr;
                    int ir = qt.n_thr, ii = qt.n_thr;
                    if (yx == yx) { int lo = 0, hi = qt.n_thr; while (lo < hi) { int mid = (lo + hi) >> 1; if (thr[mid] <= yx) lo = mid + 1; else hi = mid; } ir = lo; }
                    if (yy == yy) { int lo = 0, hi = qt.n_thr; while (lo < hi) { int mid = (lo + hi) >> 1; if (thr[mid] <= yy) lo = mid + 1; else hi = mid; } ii = lo; }
                    v[u].x = lab[ir] * inv_data_scale;
                    v[u].y = lab[ii] * inv_data_scale;
                }
            }
        } else {
            if (oa) { v[0] = __ldcs(reinterpret_cast<const double2*>(src) + g * No + ja); v[0].x *= inv_data_scale; v[0].y *= inv_data_scale; }
            if (ob) { v[1] = __ldcs(reinterpret_cast<const double2*>(src) + g * No + jb); v[1].x *= inv_data_scale; v[1].y *= inv_data_scale; }
        }
        // complex j sits in K-core kb = j / 4 at byte (row % 8) * 16 + (j % 4) * 4 of the core
        #pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int j = u ? jb : ja;
            if (j >= No) continue;
            const int s_off = (j >> 2) * 128 + warp * 16 + (j & 3) * 4;
            if (OBSERVE && !SPLIT && qt.n_bits == 1) {
                *reinterpret_cast<uint32_t*>(s_img + s_off) = hbits[u];
            } else if (SPLIT) {
                if (!(fabs(v[u].x) <= 60000.0 && fabs(v[u].y) <= 60000.0)) { my_bad = 1; v[u] = make_double2(0.0, 0.0); }     // out of FP16 range / NaN
                const __half hr = __double2half(v[u].x), hi_ = __double2half(v[u].y);
                *reinterpret_cast<__half2*>(s_img + s_off) = __halves2half2(hr, hi_);
                *reinterpret_cast<__half2*>(s_img + kbs * 128 + s_off) =
                    __halves2half2(__double2half(v[u].x - (double)__half2float(hr)), __double2half(v[u].y - (double)__half2float(hi_)));
            } else {
                const float mr = (float)v[u].x, mi = (float)v[u].y;
                const float qr = rintf(mr), qi = rintf(mi);
                // off-grid / out-of-range / NaN data cannot be represented exactly: flag the row (re-evaluated by the complex128 kernel)
                if (!(fabsf(mr - qr) <= 1e-4f * fmaxf(1.f, fabsf(qr)) && fabsf(mi - qi) <= 1e-4f * fmaxf(1.f, fabsf(qi)) &&
                      fabsf(qr) <= 2048.f && fabsf(qi) <= 2048.f))
                    my_bad = 1;
                *reinterpret_cast<__half2*>(s_img + s_off) = __floats2half2_rn(qr, qi);
            }
        }
    }
    if (__any_sync(0xffffffffu, my_bad) && lane == 0) s_bad[warp] = 1;
    __syncthreads();
    // whole core matrices out: core (mb, kb) of copy c at tile image + c * TILE_M * KD halves + (kb * 16 + mb) * 128 B
    unsigned char* tile_img = reinterpret_cast<unsigned char*>(img + (size_t)tile * TILE_M * KD * COPIES);
    for (int c = warp; c < COPIES * kbs; c += 8) {
        const int copy = c / kbs, kb = c - copy * kbs;
        *reinterpret_cast<uint32_t*>(tile_img + (size_t)copy * TILE_M * KD * 2 + (size_t)(kb * (TILE_M / 8) + mb) * 128 + lane * 4) =
            *reinterpret_cast<const uint32_t*>(s_img + c * 128 + lane * 4);
    }
    if (threadIdx.x < 8) {      // rows that cannot be represented go on the fix list (complex128 re-evaluation after the tensor-core launches)
        const int64_t row = tile * TILE_M + mb * 8 + threadIdx.x;
        bad[row] = (unsigned char)s_bad[threadIdx.x];
        if (s_bad[threadIdx.x] && row < B) fix_buf[2 + atomicAdd(fix_buf, 1)] = (int)row;
    }
}

// ------------------------------------------------------------------------------------------------ mode selection
// One warp per pilot: weighted log-probabilities (FP32 pairs from the EPI=1 pass) -> combination weights per mode, with
// the reference's semantics (gmm:197-242 / mofa:125-158): softmax responsibilities; top-1 = argmax of l (MFA flag: argmax
// of exp(l), i.e. label 0 when everything underflows); top-n / cumulative-rho = descending selection, renormalised.
// K <= 1024 (32 values per lane).  Also exports l as float64 when asked.
// select_row: one warp, the K weighted log-probabilities of a pilot spread over the lanes (entry i of lane l is component 32 i + l,
// -inf where there is none).  Writes the weight row or the top-1 label; returns whether the selection is too close to call when the
// log-likelihoods carry an error of up to ~tie_eps nats (the deciding gap -- maximum vs runner-up, last selected vs first left out
// -- or a prefix sum vs rho): the caller then has the pilot re-evaluated in complex128 (tc_refine_kernel, which calls this again
// with tie_eps = 0 on the exact values).
// EXACT: the responsibilities are formed like the complex128 kernel forms them (FP64 exp, logsumexp: gmm:652) -- the re-selection of
// the listed near-ties must not decide a prefix sum that is within 1e-7 of rho with FP32 exponentials.
template <int PER, bool EXACT = false>      // entries per lane: K <= 32 PER
__device__ __forceinline__ bool select_row(double (&l)[PER], const int lane, const int K, const int mode, const int n_top, const double rho,
                                           const int flags, double tie_eps, float* __restrict__ w_row, int* __restrict__ top_slot,
                                           const double* __restrict__ logc = nullptr, const double inv_nobs = 0.0) {
    const int per = (K + 31) / 32;
    double mx = -INFINITY, mx2 = -INFINITY;      // maximum and runner-up (a second entry equal to the maximum counts as runner-up)
    int amax = 0;
    bool tie = false;
    #pragma unroll
    for (int i = 0; i < PER; ++i) {
        if (i < per && i * 32 + lane < K) {
            if (l[i] != l[i]) tie = true;                         // NaN: let the complex128 kernel reproduce numpy's answer
            if (l[i] > mx) { mx2 = mx; mx = l[i]; amax = i * 32 + lane; } else if (l[i] > mx2) mx2 = l[i];
        }
    }
    // warp argmax (first index among equal maxima, like np.argmax)
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double om = __shfl_xor_sync(0xffffffffu, mx, off), om2 = __shfl_xor_sync(0xffffffffu, mx2, off);
        const int oa = __shfl_xor_sync(0xffffffffu, amax, off);
        mx2 = fmax(fmax(mx2, om2), fmin(mx, om));
        if (om > mx || (om == mx && oa < amax)) { mx = om; amax = oa; }
    }
    tie = __any_sync(0xffffffffu, tie);
    if (!w_row && !top_slot) return false;
    // the error of an FP32-accumulated log-likelihood grows with its quadratic form q = logc - l (~n_obs for a pilot that fits the
    // component, much more for outliers): the gap scales with q / n_obs of the best component
    if (logc && amax >= 0 && amax < K) tie_eps *= fmax(1.0, (__ldg(logc + amax) - mx) * inv_nobs);
    if (mode == QCE_MODE_TOP1) {
        if (!(mx - mx2 > tie_eps) || ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && fabs(mx + 745.1332) < 0.01)) tie = true;
        if ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && exp(mx) == 0.0) amax = 0;
        if (top_slot) {      // bucketed combination: the label instead of a one-hot weight row
            if (lane == 0) *top_slot = amax;
            return tie;
        }
        #pragma unroll
        for (int i = 0; i < PER; ++i)
            if (i < per) { const int k = i * 32 + lane; if (k < K) w_row[k] = (k == amax) ? 1.f : 0.f; }
        return tie;
    }
    // responsibilities exp(l - logsumexp(l)): the difference to the maximum is formed in FP64 (the pair carries ~48 bits),
    // the exponential in FP32 (an FP64 exp per entry made this kernel 15 % of the top-n / split-path time)
    if (EXACT) {
        double sum = 0.0;
        #pragma unroll
        for (int i = 0; i < PER; ++i) if (i < per && i * 32 + lane < K) sum += exp(l[i] - mx);
        #pragma unroll
        for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
        const double lse = mx + log(sum);
        #pragma unroll
        for (int i = 0; i < PER; ++i) l[i] = (i < per && i * 32 + lane < K) ? exp(l[i] - lse) : -1.0;      // -1 = no entry
    } else {
        float sumf = 0.f;
        #pragma unroll
        for (int i = 0; i < PER; ++i) {
            const bool on = i < per && i * 32 + lane < K;
            const float e = on ? expf((float)(l[i] - mx)) : 0.f;
            l[i] = on ? (double)e : -1.0;                                                             // -1 = no entry
            sumf += e;
        }
        #pragma unroll
        for (int off = 16; off > 0; off >>= 1) sumf += __shfl_xor_sync(0xffffffffu, sumf, off);
        const double inv_sum = 1.0 / (double)sumf;
        #pragma unroll
        for (int i = 0; i < PER; ++i) if (l[i] >= 0.0) l[i] *= inv_sum;
    }
    if (mode == QCE_MODE_ALL) {
        #pragma unroll
        for (int i = 0; i < PER; ++i)
            if (i < per) { const int k = i * 32 + lane; if (k < K) w_row[k] = (float)l[i]; }
        return tie;
    }
    // descending selection; selected entries are flagged by a set bit in `sel`
    const int limit = (mode == QCE_MODE_TOPN) ? (n_top < K ? n_top : K) : K;
    unsigned sel = 0;
    double cum = 0.0, last = -1.0;
    bool done = false;                 // selection complete: one more pass looks at the best candidate left out
    for (int it = 0; it <= limit; ++it) {
        double bv = -1.0;
        int bk = 0x7fffffff;
        #pragma unroll
        for (int i = 0; i < PER; ++i)
            if (i < per && !((sel >> i) & 1u) && l[i] > bv) { bv = l[i]; bk = i * 32 + lane; }
        #pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
            const int ok = __shfl_xor_sync(0xffffffffu, bk, off);
            if (ov > bv || (ov == bv && ok < bk)) { bv = ov; bk = ok; }
        }
        if (bv < 0.0) break;           // no candidates left
        if (done || it == limit) {     // a near-tie between the last selected and the first left out could swap them
            if (bv > last * (1.0 - tie_eps)) tie = true;
            break;
        }
        if ((bk & 31) == lane) sel |= 1u << (bk >> 5);
        cum += bv;
        last = bv;
        if (mode == QCE_MODE_CUMPROB) {
            if (fabs(cum - rho) < tie_eps) tie = true;      // a prefix sum this close to rho: which side it falls on is not decidable here
            if (cum >= rho) done = true;                    // searchsorted(cumsum, rho) + 1 entries (gmm:234)
        }
    }
    #pragma unroll
    for (int i = 0; i < PER; ++i)
        if (i < per) { const int k = i * 32 + lane; if (k < K) w_row[k] = ((sel >> i) & 1u) ? (float)(l[i] / cum) : 0.f; }
    return tie;
}

// the tie list of a chunk: [0] = count, then chunk rows.  Rows that are off the quantiser grid (bad != 0) are not listed: the
// complex128 kernel answers them completely after the tensor-core launches.
__device__ __forceinline__ void tie_append(const unsigned char* bad, int* tie_buf, int64_t chunk_row) {
    if (bad[chunk_row] == 0) tie_buf[1 + atomicAdd(tie_buf, 1)] = (int)chunk_row;
}

// One warp per pilot: weighted log-probabilities (FP32 pairs from the EPI=1 pass) -> combination weights per mode, with
// the reference's semantics (gmm:197-242 / mofa:125-158): softmax responsibilities; top-1 = argmax of l (MFA flag: argmax
// of exp(l), i.e. label 0 when everything underflows); top-n / cumulative-rho = descending selection, renormalised.
// K <= 1024 (32 values per lane).  Also exports l as float64 when asked.
template <int PER, bool EXACT = false>
__global__ void __launch_bounds__(256) tc_select_kernel(const float2* __restrict__ lp2, int64_t B, int K, int mode, int n_top, double rho,
                                                        int flags, float* __restrict__ w_out, double* __restrict__ logp_out,
                                                        int* __restrict__ top_out, const unsigned char* __restrict__ bad, int* __restrict__ tie_buf,
                                                        double tie_eps, const int* __restrict__ list, const double* __restrict__ logc, double inv_nobs,
                                                        int* __restrict__ pair_cnt = nullptr, float pair_thresh = 0.f) {
    const int lane = threadIdx.x & 31;
    // list != null: re-selection of the pilots on the tie list after tc_refine_kernel made their log-probabilities exact
    const int64_t n = list ? (int64_t)__ldg(list) : B;
    for (int64_t e = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += (int64_t)gridDim.x * 8) {
        const int64_t b = list ? (int64_t)__ldg(list + 1 + e) : e;
        double l[PER];
        #pragma unroll
        for (int i = 0; i < PER; ++i) {
            l[i] = -INFINITY;
            const int k = i * 32 + lane;
            if (k < K) {
                const float2 v = lp2[b * K + k];
                l[i] = (double)v.x + (double)v.y;
                if (logp_out) logp_out[b * K + k] = tc_logp_export(l[i]);
            }
        }
        // (re-selection of a listed pilot: its pairs leave the histogram of the pair-bucketed combination and the new ones enter)
        if (pair_cnt && w_out) for (int k = lane; k < K; k += 32) if (w_out[b * K + k] > pair_thresh) atomicSub(pair_cnt + k, 1);
        const bool tie = select_row<PER, EXACT>(l, lane, K, mode, n_top, rho, flags, tie_eps, w_out ? w_out + b * K : nullptr, top_out ? top_out + b : nullptr,
                                                logc, inv_nobs);
        if (pair_cnt && w_out) { __syncwarp(); for (int k = lane; k < K; k += 32) if (w_out[b * K + k] > pair_thresh) atomicAdd(pair_cnt + k, 1); }
        if (tie && lane == 0 && tie_buf) tie_append(bad, tie_buf, b);
    }
}

// The same selection with ONE THREAD PER PILOT (K <= 256): the warp-per-pilot form above spends its time in shuffles (~100 per pilot
// at K = 64: 552 us per 2^19 pilots, the launch was half as long as the whitening launch it follows).  A block stages the FP32
// (hi, lo) pairs of R pilots transposed in shared memory ([k][pilot]: conflict-free for thread = pilot), every thread then scans
// its own K values: maximum / runner-up in exact FP64, responsibilities with FP32 exponentials, descending selection by repeated
// scans (n + 1 of them for top-n), the same too-close-to-call rules.  The weight rows go back through shared memory so that the
// global stores are coalesced.  pair_cnt != null: histogram of the selected (pilot, component) pairs with a weight above pair_thresh
// (the count pass of the pair-bucketed combination, fused).
// SEL_ROWS pilots and 128 threads per block (all of them stage, SEL_ROWS of them select).  The staging loop is latency-bound, so
// small tiles -- many blocks, many loads in flight per SM -- win: one 132 KB block of 256 pilots per SM 503 us per 2^19 pilots at
// K = 64, 128 pilots (66 KB) 265 us, 64: 222 us, 32: 198 us, 16: 301 us.
constexpr int SEL_THREADS = 128;
constexpr int SEL_ROWS = 32;
__global__ void __launch_bounds__(SEL_THREADS) tc_select_rows_kernel(const float2* __restrict__ lp2, int64_t B, int K, int mode, int n_top, double rho, int flags,
                                                             float* __restrict__ w_out, double* __restrict__ logp_out, int* __restrict__ top_out,
                                                             const unsigned char* __restrict__ bad, int* __restrict__ tie_buf, double tie_eps0,
                                                             const double* __restrict__ logc, double inv_nobs, int* __restrict__ pair_cnt, float pair_thresh) {
    extern __shared__ __align__(16) unsigned char sel_smem[];
    constexpr int P = SEL_ROWS + 1;                            // pitch: thread = pilot reads column `pilot` of every row k
    float* s_hi = reinterpret_cast<float*>(sel_smem);          // [K][P]  l_hi, later e_k = exp(l_k - max), later the weight
    float* s_lo = s_hi + (size_t)K * P;                        // [K][P]  l_lo
    int* s_cnt = reinterpret_cast<int*>(s_lo + (size_t)K * P); // [K] pair histogram of this block
    const int64_t row0 = (int64_t)blockIdx.x * SEL_ROWS;
    const int nrow = (int)((B - row0) < SEL_ROWS ? (B - row0) : SEL_ROWS);
    {
        const float2* src = lp2 + row0 * K;
        const int n = nrow * K;
        #pragma unroll 1
        for (int i0 = threadIdx.x; i0 < n; i0 += 8 * SEL_THREADS) {       // 8 independent loads per thread in flight
            float2 v[8];
            #pragma unroll
            for (int u = 0; u < 8; ++u) { const int i = i0 + u * SEL_THREADS; v[u] = i < n ? __ldcs(src + i) : make_float2(0.f, 0.f); }
            #pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = i0 + u * SEL_THREADS;
                if (i < n) {
                    const int r = i / K, k = i - r * K;
                    s_hi[k * P + r] = v[u].x;
                    s_lo[k * P + r] = v[u].y;
                    if (logp_out) logp_out[(row0 + r) * K + k] = tc_logp_export((double)v[u].x + (double)v[u].y);
                }
            }
        }
    }
    if (pair_cnt) for (int k = threadIdx.x; k < K; k += SEL_THREADS) s_cnt[k] = 0;
    __syncthreads();
    if (!w_out && !top_out) return;
    const int r = threadIdx.x;
    if (r < nrow) {
        // FP32 throughout (the FP64 pipe issues 2 warp-instructions per clock per SM: O(K) FP64 work per pilot made this launch
        // FP64-bound): the maximum is located on the hi parts; every l_k is then taken RELATIVE to it, d_k = (hi_k - hi_max) +
        // (lo_k - lo_max), exact to ~1e-7 |d_k|; a component whose lo part overturns the order of the hi parts has d_k > 0, which
        // counts as too close to call like every |d_k| <= tie_eps -- the exact selection then decides.
        float m_hi = -INFINITY;
        int amax = 0;
        bool tie = false;
        #pragma unroll 8
        for (int k = 0; k < K; ++k) {
            const float hi = s_hi[k * P + r];
            if (hi != hi) tie = true;
            if (hi > m_hi) { m_hi = hi; amax = k; }
        }
        const float m_lo = s_lo[amax * P + r];
        const double mx = (double)m_hi + (double)m_lo;
        double tie_eps = tie_eps0;
        if (logc) tie_eps *= fmax(1.0, (__ldg(logc + amax) - mx) * inv_nobs);
        const float epsf = (float)tie_eps;
        float d2 = -INFINITY, sumf = 0.f;            // runner-up (relative to the maximum), normaliser
        #pragma unroll 8
        for (int k = 0; k < K; ++k) {
            const float d = (s_hi[k * P + r] - m_hi) + (s_lo[k * P + r] - m_lo);
            if (k != amax && d > d2) d2 = d;
            const float e = mode == QCE_MODE_TOP1 ? 0.f : expf(d);
            s_hi[k * P + r] = e;
            sumf += e;
        }
        if (mode == QCE_MODE_TOP1) {
            if (!(-d2 > epsf) || ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && fabs(mx + 745.1332) < 0.01)) tie = true;
            if ((flags & QCE_FLAG_TOP1_EXP_ARGMAX) && exp(mx) == 0.0) amax = 0;
            if (top_out) top_out[row0 + r] = amax;
            else for (int k = 0; k < K; ++k) s_hi[k * P + r] = (k == amax) ? 1.f : 0.f;
        } else {
            if (d2 > 0.f) tie = true;                 // (the lo parts overturned the order: exact selection)
            const float inv_sum = 1.f / sumf;
            const bool count = pair_cnt != nullptr && bad[row0 + r] == 0;
            if (mode == QCE_MODE_ALL) {
                #pragma unroll 8
                for (int k = 0; k < K; ++k) {
                    const float wk = s_hi[k * P + r] * inv_sum;
                    s_hi[k * P + r] = wk;
                    if (count && wk > pair_thresh) atomicAdd(&s_cnt[k], 1);
                }
            } else {
                // descending selection: selected entries move to s_lo (responsibilities), their s_hi slot becomes -1
                #pragma unroll 8
                for (int k = 0; k < K; ++k) s_lo[k * P + r] = 0.f;
                const int limit = (mode == QCE_MODE_TOPN) ? (n_top < K ? n_top : K) : K;
                double cum = 0.0;
                float last = -1.f;
                bool done = false;
                for (int it = 0; it <= limit; ++it) {
                    float bvf = -1.f;
                    int bk = -1;
                    #pragma unroll 8
                    for (int k = 0; k < K; ++k) { const float e = s_hi[k * P + r]; if (e > bvf) { bvf = e; bk = k; } }
                    if (bk < 0) break;                        // no candidates left
                    const float bv = bvf * inv_sum;
                    if (done || it == limit) { if (bv > last * (1.f - epsf)) tie = true; break; }
                    s_hi[bk * P + r] = -1.f;
                    s_lo[bk * P + r] = bv > 0.f ? bv : 1e-45f;      // (the marker must survive a responsibility that underflowed)
                    cum += (double)bv;
                    last = bv;
                    if (mode == QCE_MODE_CUMPROB) {
                        if (fabs(cum - rho) < tie_eps) tie = true;
                        if (cum >= rho) done = true;
                    }
                }
                const float inv_cum = (float)(1.0 / cum);
                #pragma unroll 8
                for (int k = 0; k < K; ++k) {
                    const float sel = s_lo[k * P + r];
                    const float wk = sel > 0.f ? sel * inv_cum : 0.f;
                    s_hi[k * P + r] = wk;
                    if (count && wk > pair_thresh) atomicAdd(&s_cnt[k], 1);
                }
            }
        }
        if (tie && tie_buf) tie_append(bad, tie_buf, row0 + r);
    }
    __syncthreads();
    if (w_out) for (int i = threadIdx.x; i < nrow * K; i += SEL_THREADS) { const int rr = i / K, k = i - rr * K; w_out[(row0 + rr) * K + k] = s_hi[k * P + rr]; }
    if (pair_cnt) for (int k = threadIdx.x; k < K; k += SEL_THREADS) if (s_cnt[k]) atomicAdd(pair_cnt + k, s_cnt[k]);
}

// ------------------------------------------------------------------------------------------------ exact re-selection of near-ties
// The pilots on the tie list get their K weighted log-probabilities in complex128 (the arithmetic of dense_fp64_kernel's phase 1:
// l_k = logc_k - |Linv_k r - zoff_k|^2, gmm:380-386, 413-417, 435), written over the FP32-derived pairs in lp2; tc_select_kernel
// then runs again on the listed pilots (tie_eps = 0) and overwrites their weight rows / labels, and the combine launch answers
// them like every other pilot.  Work item = (8 listed pilots) x (8 components, one per warp): the parameters of a component are
// read once for 8 pilots (one pilot per CTA made this launch L2-bandwidth bound: K x 32 KB per pilot), and a short list still
// spreads over many CTAs (the launch sits between the whitening and the combine launch: its latency counts).  Lane l takes the
// rows l and 63 - l of every 64 rows of Linv_k (equal work under the triangular skip).
// The length of the list lives on the device: the grid is fixed and walks the work items grid-stride.
constexpr int REFINE_RT = 8;
struct RefineArgs {
    int No, K, tri;
    const double2* Linv;
    const double2* zoff;
    const double* logc;
    RowSource src;
    int64_t row0;               // batch row of chunk row 0 (the source arrays are indexed by batch row)
    const int* tie_buf;         // [0] count, then chunk rows
    int* tie_total;             // running total over the chunks of a batch (qce_last_fix_count)
    float2* lp2;                // [chunk rows][K]
    double* logp_out;           // [chunk rows][K] or null: exact values for the listed pilots
};

__global__ void __launch_bounds__(256) tc_refine_kernel(const RefineArgs a) {
    extern __shared__ __align__(16) unsigned char refine_smem[];
    double2* r_s = reinterpret_cast<double2*>(refine_smem);                 // [RT][No]
    __shared__ int s_crow[REFINE_RT];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int No = a.No, K = a.K;
    const int n_list = __ldg(a.tie_buf);
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_list > 0) atomicAdd(a.tie_total, n_list);
    const int kblocks = (K + 7) / 8;
    const int n_items = ((n_list + REFINE_RT - 1) / REFINE_RT) * kblocks;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        const int tile = w / kblocks, kb = w - tile * kblocks;
        const int e0 = tile * REFINE_RT, nv = (n_list - e0) < REFINE_RT ? (n_list - e0) : REFINE_RT;
        if (threadIdx.x < REFINE_RT) s_crow[threadIdx.x] = threadIdx.x < nv ? __ldg(a.tie_buf + 1 + e0 + threadIdx.x) : -1;
        __syncthreads();
        for (int o = threadIdx.x; o < REFINE_RT * No; o += 256) {
            const int t = o / No, j = o - t * No;
            double2 v = make_double2(0.0, 0.0);
            if (t < nv) {
                const int64_t idx = (a.row0 + s_crow[t]) * No + j;
                if (a.src.r) {
                    v = reinterpret_cast<const double2*>(a.src.r)[idx];
                } else {      // get_observation_nbit with A = I (utils.py:241-251): two roundings, then the quantiser
                    double2 h;
                    if (a.src.obs_h_c64) { const float2 hf = reinterpret_cast<const float2*>(a.src.obs_h)[idx]; h = make_double2((double)hf.x, (double)hf.y); }
                    else h = reinterpret_cast<const double2*>(a.src.obs_h)[idx];
                    const double2 wn = reinterpret_cast<const double2*>(a.src.obs_noise)[idx];
                    const double2 y = make_double2(__dadd_rn(h.x, __dmul_rn(a.src.obs_noise_scale, wn.x)), __dadd_rn(h.y, __dmul_rn(a.src.obs_noise_scale, wn.y)));
                    v = quantize_value(a.src.qt.n_bits, a.src.qt.n_thr, a.src.qt.thr, a.src.qt.labels, y, nullptr);
                }
            }
            r_s[o] = v;
        }
        __syncthreads();
        {
            const int k = kb * 8 + warp;
            if (k < K) {
            const double2* __restrict__ Lk = a.Linv + (size_t)k * No * No;
            double q[REFINE_RT];
            #pragma unroll
            for (int t = 0; t < REFINE_RT; ++t) q[t] = 0.0;
            for (int i0 = 0; i0 < 2 * No; i0 += 64) {
                const int i = (i0 >> 7) * 64 + ((i0 & 64) ? 63 - lane : lane);
                if (i >= No) continue;
                const double2 zo = __ldg(a.zoff + (size_t)k * No + i);
                double2 z[REFINE_RT];
                #pragma unroll
                for (int t = 0; t < REFINE_RT; ++t) z[t] = make_double2(-zo.x, -zo.y);
                const int jn = a.tri ? i + 1 : No;
                const double2* __restrict__ Lrow = Lk + (size_t)i * No;
                #pragma unroll 4
                for (int j = 0; j < jn; ++j) {
                    const double2 l = __ldg(Lrow + j);
                    #pragma unroll
                    for (int t = 0; t < REFINE_RT; ++t) {
                        const double2 r = r_s[t * No + j];
                        z[t].x = fma(l.x, r.x, z[t].x); z[t].x = fma(-l.y, r.y, z[t].x);
                        z[t].y = fma(l.x, r.y, z[t].y); z[t].y = fma(l.y, r.x, z[t].y);
                    }
                }
                #pragma unroll
                for (int t = 0; t < REFINE_RT; ++t) q[t] += z[t].x * z[t].x + z[t].y * z[t].y;
            }
            #pragma unroll
            for (int t = 0; t < REFINE_RT; ++t) {
                #pragma unroll
                for (int off = 16; off > 0; off >>= 1) q[t] += __shfl_xor_sync(0xffffffffu, q[t], off);
            }
            double mine = 0.0;
            #pragma unroll
            for (int t = 0; t < REFINE_RT; ++t) if (lane == t) mine = q[t];
            if (lane < nv) {
                const double lv = a.logc[k] - mine;
                const size_t o = (size_t)s_crow[lane] * K + k;
                a.lp2[o] = tc_logc_pair(lv);      // 48 significant bits: ~1e-13 nats
                if (a.logp_out) a.logp_out[o] = lv;
            }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ bucketed top-1 combination
// Top-1 needs ONE LMMSE row block per pilot, not K: regroup the pilots by their selected component into buckets padded to whole
// work units, so that the combine launch runs a single component per unit (1/K of the tensor work of the weighted launch).
// Bucket sizes: block-level histogram in shared memory, one global atomic per (block, non-empty bucket) -- per-pilot global atomics
// on K addresses serialise in L2.
__global__ void __launch_bounds__(1024) tc_bucket_count_kernel(const int* __restrict__ top, int64_t B, int K, int* __restrict__ cnt) {
    __shared__ int s_cnt[1024];
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0;
    __syncthreads();
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) atomicAdd(&s_cnt[top[b]], 1);
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) if (s_cnt[k]) atomicAdd(cnt + k, s_cnt[k]);
}

// cnt[K] -> off[K] first slot of each bucket, unit_comp[u], n_units; cursor[K] zeroed.
__global__ void __launch_bounds__(1024) tc_bucket_scan_kernel(const int* __restrict__ cnt, int K, int unit_rows, int* __restrict__ off,
                                                              int* __restrict__ cursor, int* __restrict__ unit_comp, int* __restrict__ n_units) {
    __shared__ int s_first[1024];        // first unit of bucket k
    if (threadIdx.x == 0) {
        int u = 0;
        for (int k = 0; k < K; ++k) { s_first[k] = u; u += (cnt[k] + unit_rows - 1) / unit_rows; }
        *n_units = u;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const int u0 = s_first[k], nu = (cnt[k] + unit_rows - 1) / unit_rows;
        off[k] = u0 * unit_rows;
        cursor[k] = 0;
        for (int u = 0; u < nu; ++u) unit_comp[u0 + u] = k;
    }
}

// slot of every pilot inside its bucket (order within a bucket is irrelevant: pilots are independent): rank within the block from
// a shared-memory histogram, one global atomic per (block, non-empty bucket) reserves the block's range
__global__ void __launch_bounds__(1024) tc_bucket_place_kernel(const int* __restrict__ top, int64_t B, int K, const int* __restrict__ off,
                                                               int* __restrict__ cursor, int* __restrict__ perm) {
    __shared__ int s_cnt[1024];
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0;
    __syncthreads();
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int k = 0, local = 0;
    if (b < B) { k = top[b]; local = atomicAdd(&s_cnt[k], 1); }
    __syncthreads();
    for (int j = threadIdx.x; j < K; j += blockDim.x) { const int c = s_cnt[j]; s_cnt[j] = c ? off[j] + atomicAdd(cursor + j, c) : 0; }
    __syncthreads();
    if (b < B) perm[s_cnt[k] + local] = (int)b;
}

// pilot tiles in bucket order: one block per destination tile, a thread moves the 16-byte K-core pieces of one pilot row
// (row r of a tile keeps its piece of core column kb at byte (kb * 16) * 128 + r * 16 of each copy)
__global__ void __launch_bounds__(256) tc_bucket_gather_kernel(const unsigned char* __restrict__ img, const int* __restrict__ perm,
                                                               const int* __restrict__ n_units, int tiles_per_unit, int kbs, int copies,
                                                               unsigned char* __restrict__ img2) {
    const int64_t tile = blockIdx.x;
    if (tile >= (int64_t)__ldg(n_units) * tiles_per_unit) return;
    const int r = threadIdx.x & (TILE_M - 1);
    const size_t tile_bytes = (size_t)copies * kbs * TILE_M * 16;
    const int src = __ldg(perm + tile * TILE_M + r);
    const unsigned char* from = img + (size_t)(src >= 0 ? src / TILE_M : 0) * tile_bytes + (size_t)(src >= 0 ? src % TILE_M : 0) * 16;
    unsigned char* to = img2 + (size_t)tile * tile_bytes + (size_t)r * 16;
    for (int c = threadIdx.x / TILE_M; c < copies * kbs; c += 256 / TILE_M) {
        const uint4 v = src >= 0 ? __ldg(reinterpret_cast<const uint4*>(from + (size_t)c * TILE_M * 16)) : make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(to + (size_t)c * TILE_M * 16) = v;
    }
}

// ---- pair mode: the (pilot, component) pairs with a non-negligible combination weight (top-n, cumulative rho, and 'all' when most of
// the K weights of a pilot cannot change an FP32 accumulator) are regrouped by component exactly like the top-1 labels; a pilot
// then owns several slots.  thresh: weights <= thresh are not pairs (0 for the hard selections, whose unselected weights are 0).
__global__ void __launch_bounds__(1024) tc_pair_count_kernel(const float* __restrict__ w, const unsigned char* __restrict__ bad, int64_t B, int K,
                                                             float thresh, int* __restrict__ cnt) {
    __shared__ int s_cnt[1024];
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b0 = (int64_t)blockIdx.x * 1024;
    for (int64_t b = b0 + warp; b < b0 + 1024 && b < B; b += 32) {
        if (bad[b]) continue;
        for (int k = lane; k < K; k += 32) if (w[b * K + k] > thresh) atomicAdd(&s_cnt[k], 1);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) if (s_cnt[k]) atomicAdd(cnt + k, s_cnt[k]);
}

// as tc_bucket_scan_kernel, plus the decision: more than max_units work units of pairs (a flat posterior: nearly every component
// matters for nearly every pilot) -> the dense weighted launch is the cheaper one: flags[0] = 1 and no units
__global__ void __launch_bounds__(1024) tc_pair_scan_kernel(const int* __restrict__ cnt, int K, int unit_rows, int max_units, int* __restrict__ off,
                                                            int* __restrict__ cursor, int* __restrict__ unit_comp, int* __restrict__ n_units,
                                                            int* __restrict__ dense_flag) {
    __shared__ int s_first[1024];
    __shared__ int s_dense;
    if (threadIdx.x == 0) {
        int u = 0;
        for (int k = 0; k < K; ++k) { s_first[k] = u; u += (cnt[k] + unit_rows - 1) / unit_rows; }
        s_dense = u > max_units;
        *n_units = s_dense ? 0 : u;
        *dense_flag = s_dense;
    }
    __syncthreads();
    if (s_dense) return;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const int u0 = s_first[k], nu = (cnt[k] + unit_rows - 1) / unit_rows;
        off[k] = u0 * unit_rows;
        cursor[k] = 0;
        for (int u = 0; u < nu; ++u) unit_comp[u0 + u] = k;
    }
}

__global__ void __launch_bounds__(1024) tc_pair_place_kernel(const float* __restrict__ w, const unsigned char* __restrict__ bad, int64_t B, int K,
                                                             float thresh, const int* __restrict__ off, int* __restrict__ cursor,
                                                             const int* __restrict__ dense_flag, int* __restrict__ perm, float* __restrict__ slot_w) {
    // a block owns 1024 consecutive pilots; a warp walks pilots with its lanes over the components (coalesced weight rows).  Pass 1:
    // block histogram; one global atomic per (block, component) reserves the block's slot range; pass 2: slots within the range.
    if (__ldg(dense_flag)) return;
    __shared__ int s_cnt[1024], s_base[1024];
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b0 = (int64_t)blockIdx.x * 1024;
    for (int pass = 0; pass < 2; ++pass) {
        for (int64_t b = b0 + warp; b < b0 + 1024 && b < B; b += 32) {
            if (bad[b]) continue;
            for (int k = lane; k < K; k += 32) {
                const float wk = w[b * K + k];
                if (wk > thresh) {
                    const int local = atomicAdd(&s_cnt[k], 1);
                    if (pass) { const int slot = s_base[k] + local; perm[slot] = (int)b; slot_w[slot] = wk; }
                }
            }
        }
        __syncthreads();
        if (!pass) for (int k = threadIdx.x; k < K; k += blockDim.x) { const int c = s_cnt[k]; s_base[k] = c ? off[k] + atomicAdd(cursor + k, c) : 0; s_cnt[k] = 0; }
        __syncthreads();
    }
}

// pair mode, last step: the FP32 rows the pair launches added into -> complex128 estimates (and the NMSE accumulators)
__global__ void __launch_bounds__(256) tc_pair_finish_kernel(const float2* __restrict__ rows, double2* __restrict__ h_est, const void* __restrict__ h_true,
                                                             int h_true_c64, const unsigned char* __restrict__ bad, int64_t B, int N,
                                                             const int* __restrict__ dense_flag, double* __restrict__ acc) {
    if (__ldg(dense_flag)) return;                 // the dense weighted launch wrote the estimates and did the accumulation itself
    double err = 0.0, pw = 0.0, cnt = 0.0;
    const int lane = threadIdx.x & 31;
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < B; b += (int64_t)gridDim.x * 8) {
        if (bad[b]) continue;
        for (int j = lane; j < N; j += 32) {
            const float2 e = rows[b * N + j];
            if (h_est) h_est[b * N + j] = make_double2((double)e.x, (double)e.y);
            if (acc && h_true) {
                float2 h;
                if (h_true_c64) h = reinterpret_cast<const float2*>(h_true)[b * N + j];
                else { const double2 hd = reinterpret_cast<const double2*>(h_true)[b * N + j]; h = make_float2((float)hd.x, (float)hd.y); }
                const float dx = e.x - h.x, dy = e.y - h.y;
                err += (double)(dx * dx + dy * dy);
                pw += (double)(h.x * h.x + h.y * h.y);
            }
        }
        if (lane == 0) cnt += 1.0;
    }
    if (!acc) return;
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        err += __shfl_xor_sync(0xffffffffu, err, off);
        pw += __shfl_xor_sync(0xffffffffu, pw, off);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    }
    if (lane == 0 && cnt > 0.0) { atomicAdd(acc + 0, err); atomicAdd(acc + 1, pw); atomicAdd(acc + 2, cnt); }
}

static int sm_count() {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, current_device());
    return sms;
}

// bytes of one FP16 pilot tile: TILE_M rows of 2 n_obs halves, twice for (hi, lo) pairs of pilots off the integer grid
static size_t tc_tile_bytes(const qce_model* m) { return (size_t)TILE_M * 2 * m->n_obs * sizeof(__half) * (m->tc.split_a ? 2 : 1); }

static qce_status tc_scratch(const qce_model* m, cudaStream_t s, int64_t rows, TileScratch** out) {
    StreamScratch* sc = scratch_for(s);
    TileScratch& t = sc->tc;
    const size_t tiles = (size_t)((rows + TILE_M - 1) / TILE_M + 4);   // the last work unit (up to 4 tiles) may reach past the end
    const size_t need_img = tiles * tc_tile_bytes(m), need_bad = tiles * TILE_M;
    qce_status st = grow(t.img, need_img, true);
    if (!st) st = grow(t.bad, need_bad, true);
    if (!st) st = grow(t.fix, (need_bad + 2) * sizeof(int));        // [0] rows on the list, [1] near-ties re-selected so far, then the list
    if (st) return st;
    QCE_CUDA_TRY(cudaMemsetAsync(t.fix.p, 0, 2 * sizeof(int), s));      // a new batch is about to be formatted: empty fix list
    sc->last_fix = t.fix_list();
    *out = &t;
    return QCE_OK;
}

// complex128 re-evaluation of the rows on the fix list (pilots off the tensor-core grid, hard selections too close to call): they
// were neither written nor accumulated by the tensor-core launches.  The list is short (typically 1e-4 of the batch), its length
// lives on the device: the launch is sized independently of it.
static qce_status tc_fix_rows(const qce_model* m, const TileScratch* ts, cudaStream_t s, int64_t B, int mode, int n_top, double rho,
                              double* h_est, double* logp_out, const void* h_true, int h_true_c64, double* acc) {
    if (!h_est && !logp_out && !acc) return QCE_OK;
    return launch_dense_fp64_rows(m, s, ts->src, ts->fix_list() + 2, ts->fix_list(), B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
}

// tie list and [rows][K] log-probability / weight scratch of a chunk of `rows` pilots
static qce_status tc_scratch_aux(TileScratch* t, size_t rows, size_t K) {
    qce_status st = grow(t->tie, (rows + 1) * sizeof(int));
    if (!st) st = grow(t->lp2, rows * K * sizeof(float2));
    if (!st) st = grow(t->wts, rows * K * sizeof(float));
    return st;
}

// The instantiated shapes, as X(n_obs / 16, part_cols / 32): the 2 n_obs whitening columns and one block of part_cols estimate
// columns.  Fused shapes (n_obs, n_ant <= 64): Z|H in one MMA, estimate row in registers, part_cols = 2 n_ant; every launch family
// is instantiated for them.
#define QCE_TC_FUSED_SHAPES(X) X(4, 4) X(2, 2) X(1, 1) X(3, 3) X(4, 2) X(2, 1)
// Split-only shapes: the 2 n_ant estimate columns are produced in row blocks of part_cols <= 128 (64 packed register accumulators
// per pilot), the 2 n_obs whitening columns by a launch of their own; only the split launches are instantiated for them.  n_ant is
// n_obs (one pilot per antenna) or n_obs / 2 (two pilots per antenna, A = kron([1, j], I)).
#define QCE_TC_SPLIT_SHAPES(X) X(16, 4) X(8, 4) X(6, 3)

static bool tc_instantiated(const qce_model* m) {
#define QCE_TC_FUSED_HIT(Z, H) if (m->n_obs == 16 * Z && m->n_ant == 16 * H) return true;
    QCE_TC_FUSED_SHAPES(QCE_TC_FUSED_HIT)
#undef QCE_TC_FUSED_HIT
    return false;
}

static bool tc_split_shape(int No, int N, int* parts, int* part_cols) {
#define QCE_TC_SPLIT_HIT(Z, H) if (No == 16 * Z && (N == No || 2 * N == No)) { *part_cols = 32 * H; *parts = 2 * N / (32 * H); return true; }
    QCE_TC_SPLIT_SHAPES(QCE_TC_SPLIT_HIT)
#undef QCE_TC_SPLIT_HIT
    return false;
}

static qce_status tc_not_instantiated(const qce_model* m) {
    set_error("tensor-core kernel: n_obs=%d n_ant=%d not instantiated", m->n_obs, m->n_ant);
    return QCE_ERR_UNSUPPORTED;
}

// n_obs = 256 with pilots off the integer grid: a (hi, lo) pilot tile pair would take 256 KB of shared memory
static bool tc_off_grid_too_wide(const qce_model* m) { return m->n_obs > 128 && !(m->data_scale > 0.0); }

bool tc_supported(const qce_model* m, int mode) {
    if (!(m->data_scale >= 0.0)) return false;
    int parts = 0, pc = 0;
    if (tc_split_shape(m->n_obs, m->n_ant, &parts, &pc)) return !tc_off_grid_too_wide(m) && (!m->tc.ready || m->tc.triangular);
    if (m->data_scale == 0.0 && m->tc.ready && !m->tc.triangular) return false;      // off-grid pilots: SM-pair variant only
    // the modes other than the fused 'all' need the SM-pair variant (triangular whitening factor)
    if (mode != QCE_MODE_ALL && m->tc.ready && !m->tc.triangular) return false;
    return tc_instantiated(m);
}

const char* tc_unsupported_reason(const qce_model* m) {
    return tc_off_grid_too_wide(m) ? ": pilots off the integer grid (Lloyd-Max labels, unquantised data) at n_obs > 128 would need a "
                                     "256 KB (hi, lo) pilot tile pair per CTA, more than the shared memory holds" : "";
}

void tc_free(qce_model* m) {
    TcParams& p = m->tc;
    cudaFree(p.image); cudaFree(p.image2); cudaFree(p.zoff); cudaFree(p.hoff); cudaFree(p.zscale); cudaFree(p.hscale); cudaFree(p.logc2); cudaFree(p.flags);
    cudaFree(p.image_z);
    for (void* h : p.image_h) cudaFree(h);
    p = TcParams();
}

qce_status tc_pack_params(qce_model* m, cudaStream_t s) {
    TcParams& p = m->tc;
    const size_t K = m->n_comp, No = m->n_obs, N = m->n_ant;
    const size_t comp_halfs = 2 * (2 * No + 2 * N) * (2 * No);
    p.split = tc_split_shape((int)No, (int)N, &p.h_parts, &p.part_cols);
    p.split_a = !(m->data_scale > 0.0);
    p.eff_scale = p.split_a ? 1.0 / 256.0 : m->data_scale;
    if (!p.zoff) {
        if (!p.split) {
            p.image_bytes = K * comp_halfs * sizeof(__half);
            QCE_CUDA_TRY(cudaMalloc(&p.image, p.image_bytes));
        }
        QCE_CUDA_TRY(cudaMalloc(&p.zoff, K * 2 * No * sizeof(float)));
        QCE_CUDA_TRY(cudaMalloc(&p.hoff, K * 2 * N * sizeof(float)));
        QCE_CUDA_TRY(cudaMalloc(&p.zscale, K * sizeof(float)));
        QCE_CUDA_TRY(cudaMalloc(&p.hscale, K * sizeof(float)));
        QCE_CUDA_TRY(cudaMalloc(&p.logc2, K * sizeof(float2)));
        QCE_CUDA_TRY(cudaMalloc(&p.flags, 2 * sizeof(int)));
    }
    QCE_CUDA_TRY(cudaMemsetAsync(p.flags, 0, 2 * sizeof(int), s));
    tc_pack_kernel<<<(unsigned)(2 * K), 256, 0, s>>>((const double2*)m->Linv, (const double2*)m->W, (int)No, (int)N, p.eff_scale,
                                                     (__half*)p.image, p.zscale, p.hscale, p.flags);
    QCE_CHECK_LAUNCH("tc_pack_kernel");
    const size_t nmax = K * (No > N ? No : N);
    tc_pack_small_kernel<<<(unsigned)((nmax + 255) / 256), 256, 0, s>>>((const double2*)m->zoff, (const double2*)m->hoff, m->logc, (int)K, (int)No,
                                                                        (int)N, p.zoff, p.hoff, (float2*)p.logc2, p.flags);
    QCE_CHECK_LAUNCH("tc_pack_small_kernel");
    int h_flags[2] = {0, 0};
    QCE_CUDA_TRY(cudaMemcpyAsync(h_flags, p.flags, sizeof(h_flags), cudaMemcpyDeviceToHost, s));
    QCE_CUDA_TRY(cudaStreamSynchronize(s));
    p.has_offsets = h_flags[0] != 0;
    p.triangular = h_flags[1] == 0;
    const int ksps = (int)(2 * No) / 32;
    if (p.split && !p.triangular) { p.ready = false; return QCE_OK; }       // only the SM-pair (triangular) layout exists for these shapes
    if (!p.split) {   // fused image: per-CTA half images of the SM-pair kernel (their layout depends on the triangular flag)
        if (p.split_a && !p.triangular) { p.ready = false; return QCE_OK; }      // off-grid pilots: SM-pair variant only
        const int nt = (int)(2 * No + 2 * N), tri16 = p.triangular ? 16 : 0;
        const size_t bytes = K * 2 * (size_t)tc2_rank_comp_bytes(nt, tri16, ksps);
        if (p.image2 && bytes > p.image2_bytes) { QCE_CUDA_TRY(cudaFree(p.image2)); p.image2 = nullptr; }
        if (!p.image2) { QCE_CUDA_TRY(cudaMalloc(&p.image2, bytes)); p.image2_bytes = bytes; }
        tc2_pack_kernel<<<(unsigned)(2 * K), 256, 0, s>>>((const double2*)m->Linv, (const double2*)m->W, (int)No, (int)N, p.eff_scale,
                                                          p.zscale, p.hscale, tri16, (int)(2 * No), 0, (int)(2 * N), (unsigned char*)p.image2);
        QCE_CHECK_LAUNCH("tc2_pack_kernel");
        p.h_parts = 1;
        p.part_cols = (int)(2 * N);
    }
    if (p.triangular) {
        // per-purpose images: whitening rows only (log-probability launch) and LMMSE row blocks (given-weights launches).  The
        // large shapes run every mode through them, the others the top-1 / top-n / cumulative modes and the log-prob export.
        const size_t bytes_z = K * 2 * (size_t)tc2_rank_comp_bytes((int)(2 * No), 16, ksps);
        const size_t bytes_h = K * 2 * (size_t)tc2_rank_comp_bytes(p.part_cols, 0, ksps);
        if (!p.image_z) QCE_CUDA_TRY(cudaMalloc(&p.image_z, bytes_z));
        tc2_pack_kernel<<<(unsigned)(2 * K), 256, 0, s>>>((const double2*)m->Linv, (const double2*)m->W, (int)No, (int)N, p.eff_scale,
                                                          p.zscale, p.hscale, 16, (int)(2 * No), 0, 0, (unsigned char*)p.image_z);
        QCE_CHECK_LAUNCH("tc2_pack_kernel");
        for (int part = 0; part < p.h_parts; ++part) {
            if (!p.image_h[part]) QCE_CUDA_TRY(cudaMalloc(&p.image_h[part], bytes_h));
            tc2_pack_kernel<<<(unsigned)(2 * K), 256, 0, s>>>((const double2*)m->Linv, (const double2*)m->W, (int)No, (int)N, p.eff_scale,
                                                              p.zscale, p.hscale, 0, 0, part * p.part_cols, p.part_cols,
                                                              (unsigned char*)p.image_h[part]);
            QCE_CHECK_LAUNCH("tc2_pack_kernel");
        }
    } else if (p.image_z) {     // parameters replaced by a non-triangular set
        QCE_CUDA_TRY(cudaFree(p.image_z)); p.image_z = nullptr;
        for (void*& h : p.image_h) { QCE_CUDA_TRY(cudaFree(h)); h = nullptr; }
    }
    QCE_CUDA_TRY(cudaStreamSynchronize(s));
    p.ready = true;
    return QCE_OK;
}

// QCE_TC_PROF (with a -DQCE_TC_PROFILE build): per-role cycle counters of CTA 0, printed after every dense_tc_kernel launch
static long long* tc_prof_counters(cudaStream_t s) {
    static long long* prof = nullptr;
    static const bool want_prof = getenv("QCE_TC_PROF") != nullptr;
    if (!want_prof) return nullptr;
    if (!prof) cudaMalloc(&prof, 16 * sizeof(long long));
    cudaMemsetAsync(prof, 0, 16 * sizeof(long long), s);
    return prof;
}

static void tc_prof_print(const TcArgs& a, int epi, cudaStream_t s) {
    long long h[16];
    cudaMemcpyAsync(h, a.prof, sizeof(h), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    fprintf(stderr, "[qce tc prof] epi %d B=%lld K=%d | mma: total %lld wait_acc_empty %lld wait_full %lld wait_a %lld | epi t0: wait %lld z %lld h %lld pro %lld | epi t1: wait %lld z %lld h %lld pro %lld | zld t0 %lld t1 %lld\n",
            epi, (long long)a.B, a.K, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9], h[10], h[11], h[12], h[13]);
}

template <int KDC, int NCHZ, int NCHH, bool OFFS, int CG, int EPI, int ORDER, int AC = 1>
static qce_status launch_cfg(TcArgs a, cudaStream_t s) {
    using Cfg = TcCfg<32 * KDC, 32 * NCHZ, 32 * NCHH, CG, ORDER, AC, tc_accb(EPI, 32 * KDC, 32 * NCHZ, 32 * NCHH, ORDER, AC)>;
    static PerDeviceOnce once;
    auto kern = dense_tc_kernel<KDC, NCHZ, NCHH, OFFS, CG, EPI, ORDER, AC>;
    if (once.first(current_device())) QCE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    const int64_t n_units = (a.B + CG * Cfg::NTILES * TILE_M - 1) / (CG * Cfg::NTILES * TILE_M);
    const int64_t max_clusters = sm_count() / CG;
    const unsigned grid = (unsigned)((n_units < max_clusters ? n_units : max_clusters) * CG);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    a.prof = tc_prof_counters(s);
    QCE_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a));
    QCE_CHECK_LAUNCH("dense_tc_kernel");
    if (a.prof) tc_prof_print(a, EPI, s);
    return QCE_OK;
}

// fused 'all' launch (Z|H in one MMA, online softmax)
template <int NCHZ, int NCHH>
static qce_status launch_offs(const TcArgs& a, bool offs, int cg, bool split_a, cudaStream_t s) {
    if (split_a) {      // pilots as FP16 (hi, lo) pairs: SM-pair variant only
        if (cg != 2) { set_error("tensor-core kernel: pilots off the integer grid need the SM-pair (triangular whitening) variant"); return QCE_ERR_UNSUPPORTED; }
        return offs ? launch_cfg<NCHZ, NCHZ, NCHH, true, 2, 0, 0, 2>(a, s) : launch_cfg<NCHZ, NCHZ, NCHH, false, 2, 0, 0, 2>(a, s);
    }
    if (cg == 2) return offs ? launch_cfg<NCHZ, NCHZ, NCHH, true, 2, 0, 0>(a, s) : launch_cfg<NCHZ, NCHZ, NCHH, false, 2, 0, 0>(a, s);
    return offs ? launch_cfg<NCHZ, NCHZ, NCHH, true, 1, 0, 0>(a, s) : launch_cfg<NCHZ, NCHZ, NCHH, false, 1, 0, 0>(a, s);
}

// per-purpose launches: epi 1 = whitening-only (log-probabilities), epi 2 = one LMMSE row block with the given weights.
// ORDER 1 (chunk-major) for the large shapes, whose pilot tiles leave room for only 2-3 ring stages.
template <int KDC, int NCHH, int ORDER, int AC>
static qce_status launch_split_ac(const TcArgs& a, bool offs, int epi, cudaStream_t s) {
    if (epi == 1) return offs ? launch_cfg<KDC, KDC, 0, true, 2, 1, ORDER, AC>(a, s) : launch_cfg<KDC, KDC, 0, false, 2, 1, ORDER, AC>(a, s);
    return offs ? launch_cfg<KDC, 0, NCHH, true, 2, 2, ORDER, AC>(a, s) : launch_cfg<KDC, 0, NCHH, false, 2, 2, ORDER, AC>(a, s);
}
template <int KDC, int NCHH>
static qce_status launch_split(const TcArgs& a, bool offs, int epi, bool split_a, cudaStream_t s) {
    if constexpr (KDC > 8) {      // n_obs = 256: on-grid pilots only (tc_supported)
        if (split_a) { set_error("tensor-core kernel: pilots off the integer grid at n_obs = %d are not supported", a.No); return QCE_ERR_UNSUPPORTED; }
        return launch_split_ac<KDC, NCHH, 1, 1>(a, offs, epi, s);
    } else if constexpr (KDC > 4) {
        return split_a ? launch_split_ac<KDC, NCHH, 1, 2>(a, offs, epi, s) : launch_split_ac<KDC, NCHH, 1, 1>(a, offs, epi, s);
    } else {
        return split_a ? launch_split_ac<KDC, NCHH, 0, 2>(a, offs, epi, s) : launch_split_ac<KDC, NCHH, 0, 1>(a, offs, epi, s);
    }
}

// Log-likelihood gap (nats) below which a hard selection is re-made in complex128.  Measured error of the DIFFERENCE of two
// FP16-split / FP32-accumulated log-likelihoods of a pilot (profiles/r02_flip_rate.json, max over 2^16..2^18 pilots): 2.2e-5 nats
// at n_obs = 64, 3.5e-5 at n_obs = 128 and on the three-pass (off-grid) path, 6.8e-5 at n_obs = 256 (profiles/n256_flip_rate.jsonl,
// 2^16 model-drawn pilots, K = 64): the gap (4e-4 at n_obs = 256) keeps a margin of >= 4x, and grows per pilot with the quadratic
// form of its best component.  QCE_TC_TIE_EPS overrides (0 disables the re-evaluation: A/B runs).
static double tc_tie_eps(const qce_model* m) {
    if (const char* e = getenv("QCE_TC_TIE_EPS")) return atof(e);
    const double scale = m->n_obs > 64 ? (double)m->n_obs / 64.0 : 1.0;
    return 1e-4 * scale * (m->tc.split_a ? 1.5 : 1.0);
}

static void tc_fill_args(const qce_model* m, const TileScratch* ts, int64_t B, double* h_est, const void* h_true, int h_true_c64, double* acc,
                         TcArgs* out) {
    const TcParams& p = m->tc;
    TcArgs& a = *out;
    a.image = (const __half*)p.image; a.image2 = (const unsigned char*)p.image2; a.zscale = p.zscale; a.hscale = p.hscale; a.zoff = p.zoff; a.hoff = p.hoff;
    a.logc2 = (const float2*)p.logc2; a.a_img = (const __half*)ts->img.p; a.bad = (const unsigned char*)ts->bad.p;
    a.h_est = (double2*)h_est; a.h_true = h_true; a.h_true_c64 = h_true_c64;
    a.lp_out = (float2*)ts->lp2.p; a.w_in = (const float*)ts->wts.p;
    a.acc = acc; a.B = B; a.K = m->n_comp; a.No = m->n_obs; a.N = m->n_ant;
    a.tri = p.triangular ? 1 : 0;
    a.prof = nullptr;
    a.h_stride = 2 * m->n_ant; a.h_col0 = 0; a.count_rows = 1;
    a.wide_io = (reinterpret_cast<uintptr_t>(h_est) % 32 == 0 && reinterpret_cast<uintptr_t>(h_true) % 32 == 0 && m->n_ant % 4 == 0) ? 1 : 0;
    a.unit_comp = nullptr; a.perm = nullptr; a.n_units_dev = nullptr;
    a.slot_w = nullptr; a.run_flag = nullptr; a.run_flag_want = 0; a.pair_acc = nullptr;
    a.top_out = nullptr; a.top_flags = m->flags;
    a.tie_buf = ts->tie_list();
    a.tie_eps = (float)tc_tie_eps(m); a.inv_nobs = 1.f / (float)m->n_obs;
}

// one split launch: epi 1 = the whitening columns (part 0), epi 2 = LMMSE row block `part`.  The caller fills `a` (tc_fill_args, then
// the fields of its variant: regrouped units, pair weights, run flag, label output).
static qce_status tc_launch_split(const qce_model* m, TcArgs a, int epi, int part, cudaStream_t s) {
    const TcParams& p = m->tc;
    a.image2 = (const unsigned char*)(epi == 1 ? p.image_z : p.image_h[part]);
    a.h_col0 = part * p.part_cols;
    a.count_rows = part == 0;
    const int cz = m->n_obs / 16, ch = p.part_cols / 32;
#define QCE_TC_SPLIT_LAUNCH(Z, H) if (cz == Z && ch == H) return launch_split<Z, H>(a, p.has_offsets, epi, p.split_a, s);
    QCE_TC_SPLIT_SHAPES(QCE_TC_SPLIT_LAUNCH) QCE_TC_FUSED_SHAPES(QCE_TC_SPLIT_LAUNCH)
#undef QCE_TC_SPLIT_LAUNCH
    return tc_not_instantiated(m);
}

// the given-weights combination: every LMMSE row block
static qce_status tc_combine_parts(const qce_model* m, const TcArgs& a, cudaStream_t s) {
    for (int part = 0; part < m->tc.h_parts; ++part) {
        const qce_status st = tc_launch_split(m, a, 2, part, s);
        if (st) return st;
    }
    return QCE_OK;
}

// fused Z|H launch: epi 0 = 'all' (online softmax), epi 3 = hard top-1 (running argmax, SM-pair variant only)
static qce_status tc_launch_fused(const qce_model* m, const TcArgs& a, int epi, cudaStream_t s) {
    const TcParams& p = m->tc;
    const bool offs = p.has_offsets;
    const int cz = m->n_obs / 16, ch = m->n_ant / 16;
    // the SM-pair (cta_group::2) variant needs a lower-triangular whitening factor; any other runs on single CTAs (cta_group::1)
    const int cg = p.triangular ? 2 : 1;
#define QCE_TC_FUSED_LAUNCH(Z, H)                                                                                                      \
    if (cz == Z && ch == H) return epi == 3 ? (offs ? launch_cfg<Z, Z, H, true, 2, 3, 0>(a, s) : launch_cfg<Z, Z, H, false, 2, 3, 0>(a, s)) \
                                            : launch_offs<Z, H>(a, offs, cg, p.split_a, s);
    QCE_TC_FUSED_SHAPES(QCE_TC_FUSED_LAUNCH)
#undef QCE_TC_FUSED_LAUNCH
    return tc_not_instantiated(m);
}

// Formats B pilots into the stream's FP16 tile image: the complex128 values src.r, or (src.r null) the channels src.obs_h observed
// (A = I) and quantised with src.qt on the fly.  The complex128 re-evaluation of flagged rows reads the pilots again from `src`.
static qce_status tc_format_tiles(qce_model* m, cudaStream_t s, int64_t B, const RowSource& src, TileScratch** out) {
    if (!tc_instantiated(m) && !m->tc.split) return tc_not_instantiated(m);
    TileScratch* ts = nullptr;
    qce_status st = tc_scratch(m, s, B, &ts);
    if (st) return st;
    const bool observe = !src.r, split_a = m->tc.split_a;
    const int64_t tiles = (B + TILE_M - 1) / TILE_M;
    // [copies][kbs][8 rows][16 B] core matrices of a block, then the quantiser's thresholds and labels
    const size_t smem = (size_t)(split_a ? 2 : 1) * (2 * m->n_obs / 8) * 128 +
                        ((observe && src.qt.n_bits > 1) ? (size_t)(2 * src.qt.n_thr + 1) * sizeof(double) : 0);
    auto kern = !observe        ? (split_a ? tc_format_kernel<false, false, true> : tc_format_kernel<false, false, false>)
                : src.obs_h_c64 ? (split_a ? tc_format_kernel<true, true, true> : tc_format_kernel<true, true, false>)
                                : (split_a ? tc_format_kernel<true, false, true> : tc_format_kernel<true, false, false>);
    kern<<<(unsigned)(tiles * (TILE_M / 8)), 256, smem, s>>>(observe ? src.obs_h : src.r, (const double2*)src.obs_noise, src.obs_noise_scale,
                                                             src.qt, B, m->n_obs, 1.0 / m->tc.eff_scale, (__half*)ts->img.p,
                                                             (unsigned char*)ts->bad.p, ts->fix_list());
    QCE_CHECK_LAUNCH("tc_format_kernel");
    ts->owner = m; ts->rows = B;
    ts->src = src;
    *out = ts;
    return QCE_OK;
}

qce_status tc_format(qce_model* m, cudaStream_t s, const double* r, int64_t B) {
    RowSource src;
    src.r = r;
    TileScratch* ts = nullptr;
    return tc_format_tiles(m, s, B, src, &ts);
}

// Rows per chunk of the paths that keep [rows][K] scratch: whole work units, at most 2^27 / K rows (1 GiB + 0.5 GiB of
// log-probabilities and weights) however large the batch is.  Each path clamps it to its batch.
constexpr int64_t TC_UNIT_ROWS = 4 * TILE_M;
static int64_t tc_chunk_rows(const qce_model* m) {
    int64_t chunk = (((int64_t)1 << 27) / m->n_comp) / TC_UNIT_ROWS * TC_UNIT_ROWS;
    if (const char* ce = getenv("QCE_TC_MODE_CHUNK")) chunk = atoll(ce) / TC_UNIT_ROWS * TC_UNIT_ROWS;      // test hook
    return chunk < TC_UNIT_ROWS ? TC_UNIT_ROWS : chunk;
}

// the chunk of a formatted batch that starts at row b0 (a multiple of the tile size): a view of its pilot tiles, and its rows of the outputs
struct TcChunk {
    TileScratch v;
    double* h_est;
    double* logp;
    const void* h_true;
};

static TcChunk tc_chunk(const qce_model* m, const TileScratch* ts, int64_t b0, double* h_est, double* logp, const void* h_true, int h_true_c64) {
    TcChunk c{*ts, nullptr, nullptr, nullptr};
    c.v.img.p = (unsigned char*)ts->img.p + (size_t)(b0 / TILE_M) * tc_tile_bytes(m);
    c.v.bad.p = (unsigned char*)ts->bad.p + b0;
    if (h_est) c.h_est = h_est + (size_t)b0 * m->n_ant * 2;
    if (logp) c.logp = logp + (size_t)b0 * m->n_comp;
    if (h_true) c.h_true = (const char*)h_true + (size_t)b0 * m->n_ant * (h_true_c64 ? 8 : 16);
    return c;
}

// Near-tie re-selection of a chunk: exact log-probabilities of the pilots on its tie list (complex128), then their hard selection
// again, overwriting their labels (`top`) and weight rows (`wts`)
static qce_status tc_reselect_ties(const qce_model* m, const TileScratch* ts, cudaStream_t s, int64_t b0, int64_t nb, int mode, int n_top,
                                   double rho, double* logp, float* wts, int* top, int* pair_cnt, float pair_thresh) {
    RefineArgs ra;
    ra.No = m->n_obs; ra.K = m->n_comp; ra.tri = m->tc.triangular ? 1 : 0;
    ra.Linv = (const double2*)m->Linv; ra.zoff = (const double2*)m->zoff; ra.logc = m->logc;
    ra.src = ts->src; ra.row0 = b0; ra.tie_buf = ts->tie_list(); ra.tie_total = ts->fix_list() + 1;
    ra.lp2 = (float2*)ts->lp2.p; ra.logp_out = logp;
    const int sms = sm_count();
    tc_refine_kernel<<<(unsigned)(4 * sms), 256, (size_t)REFINE_RT * m->n_obs * sizeof(double2), s>>>(ra);
    QCE_CHECK_LAUNCH("tc_refine_kernel");
    const int K = m->n_comp;
    auto sel = K <= 64 ? tc_select_kernel<2, true> : K <= 256 ? tc_select_kernel<8, true> : tc_select_kernel<32, true>;
    sel<<<(unsigned)sms, 256, 0, s>>>((const float2*)ts->lp2.p, nb, K, mode, n_top, rho, m->flags, wts, nullptr, top, nullptr, nullptr, 0.0,
                                      ts->tie_list(), nullptr, 0.0, pair_cnt, pair_thresh);
    QCE_CHECK_LAUNCH("tc_select_kernel(list)");
    return QCE_OK;
}

// pair mode: at most this many (pilot, component) pairs per pilot on average, else the dense weighted launch (a tuning constant)
constexpr int TC_PAIR_CAP = 4;

// the general path: log-probabilities -> per-mode weights -> weighted combination (three launches)
static qce_status tc_run_modes(qce_model* m, TileScratch* ts, cudaStream_t s, int64_t B, int mode, int n_top, double rho, double* h_est,
                               double* logp_out, const void* h_true, int h_true_c64, double* acc) {
    if (m->n_comp > 1024) { set_error("tensor-core mode selection supports K <= 1024"); return QCE_ERR_UNSUPPORTED; }
    if (!m->tc.image_z) { set_error("tensor-core mode selection needs a lower-triangular whitening factor"); return QCE_ERR_UNSUPPORTED; }
    int64_t chunk = tc_chunk_rows(m);
    const bool want_est = h_est || acc;
    // Pair mode (top-n, cumulative rho, and 'all' on the large shapes): only the (pilot, component) pairs with a weight that matters
    // are combined, regrouped by component like the top-1 labels.  'all': weights <= 1e-9 are below half an ulp of the FP32
    // accumulators the weighted launch sums them in (64 of them together still are), so dropping them changes nothing that path
    // could represent.  When a batch has more than TC_PAIR_CAP pairs per pilot on average -- a flat posterior -- the dense
    // weighted launch runs instead; the decision is made on the device (both are enqueued, one returns at once).
    // Default: on for the large shapes (n_obs > 64: an LMMSE row block launch over all K components costs 2-4x the whitening launch),
    // off for the fused shapes, where the weighted launch is as fast (measured at config 2, profiles/r02_modes.jsonl);
    // QCE_TC_PAIRS=1 / 0 forces it on / off.
    const int pair_env = getenv("QCE_TC_PAIRS") ? atoi(getenv("QCE_TC_PAIRS")) : -1;
    const bool pair_on = pair_env < 0 ? m->tc.split : pair_env != 0;
    const bool pair_mode_ok = (mode == QCE_MODE_TOPN && n_top <= TC_PAIR_CAP) || mode == QCE_MODE_CUMPROB || (mode == QCE_MODE_ALL && m->tc.split);
    const bool pairs = pair_on && want_est && pair_mode_ok && m->n_comp >= 8 && B >= 16 * TC_UNIT_ROWS;
    // (a selected component whose renormalised weight is below 1e-9 -- the tail of a top-n / cumulative selection at a peaked posterior
    // -- is not a pair either: it cannot change the FP32 row the pairs are added into)
    const float pair_thresh = 1e-9f;
    if (pairs && chunk > ((int64_t)1 << 19)) chunk = (int64_t)1 << 19;      // (the regrouped pilot tiles take TC_PAIR_CAP x the chunk's tiles)
    if (chunk > B) chunk = B;
    qce_status st = tc_scratch_aux(ts, (size_t)chunk, (size_t)m->n_comp);
    if (st) return st;
    const size_t tile_bytes = tc_tile_bytes(m);
    // top-1: regroup the pilots by selected component and run ONE component per work unit (QCE_TC_BUCKET=0: weighted launch instead)
    const int tiles_per_unit = 2 * (((m->tc.split_a && 2 * m->n_obs > 128) || 2 * m->n_obs > 256) ? 1 : TILES);      // CG * Cfg::NTILES of the split launches
    const int bucket_rows = tiles_per_unit * TILE_M;
    const bool bucket_env = !(getenv("QCE_TC_BUCKET") && atoi(getenv("QCE_TC_BUCKET")) == 0);      // read per call (A/B runs, parity test)
    const bool bucketed = bucket_env && want_est && mode == QCE_MODE_TOP1 && m->n_comp >= 4 && chunk >= 4 * (int64_t)bucket_rows;
    const int64_t cap_units = chunk / bucket_rows + m->n_comp + 1, cap_rows = cap_units * bucket_rows;
    int *b_top = nullptr, *b_perm = nullptr, *b_ucomp = nullptr, *b_cnt = nullptr, *b_off = nullptr, *b_cur = nullptr, *b_nu = nullptr;
    if (bucketed) {
        st = grow(ts->img2, (size_t)(cap_rows / TILE_M + 4) * tile_bytes);
        if (!st) st = grow(ts->bidx, (size_t)(chunk + cap_rows + cap_units + 3 * m->n_comp + 1) * sizeof(int));
        if (st) return st;
        b_top = (int*)ts->bidx.p; b_perm = b_top + chunk; b_ucomp = b_perm + cap_rows; b_cnt = b_ucomp + cap_units;
        b_off = b_cnt + m->n_comp; b_cur = b_off + m->n_comp; b_nu = b_cur + m->n_comp;
    }
    // pair mode: perm[slots] | slot_w[slots] | unit_comp[units] | cnt[K] off[K] cursor[K] | n_units | dense_flag
    const int64_t p_units = (int64_t)TC_PAIR_CAP * (chunk / bucket_rows) + m->n_comp + 1, p_rows = p_units * bucket_rows;
    int *p_perm = nullptr, *p_ucomp = nullptr, *p_cnt = nullptr, *p_off = nullptr, *p_cur = nullptr, *p_nu = nullptr, *p_dense = nullptr;
    float* p_w = nullptr;
    if (pairs && !bucketed) {
        st = grow(ts->img2, (size_t)(p_rows / TILE_M + 4) * tile_bytes);
        if (!st) st = grow(ts->bidx, (size_t)(2 * p_rows + p_units + 3 * m->n_comp + 2) * sizeof(int));
        if (!st) st = grow(ts->tmp_est, (size_t)chunk * m->n_ant * 8);          // FP32 rows the pair launches add into
        if (st) return st;
        p_perm = (int*)ts->bidx.p; p_w = (float*)(p_perm + p_rows); p_ucomp = p_perm + 2 * p_rows; p_cnt = p_ucomp + p_units;
        p_off = p_cnt + m->n_comp; p_cur = p_off + m->n_comp; p_nu = p_cur + m->n_comp; p_dense = p_nu + 1;
    }
    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
        const int64_t nb = (B - b0) < chunk ? (B - b0) : chunk;
        const TcChunk c = tc_chunk(m, ts, b0, h_est, logp_out, h_true, h_true_c64);
        // arguments of a split launch over `rows` pilot rows of this chunk (or of its regrouped tiles)
        auto args = [&](int64_t rows, double* he, const void* ht, int ht_c64, double* ac) {
            TcArgs a;
            tc_fill_args(m, &c.v, rows, he, ht, ht_c64, ac, &a);
            a.pair_acc = (float*)ts->tmp_est.p;
            return a;
        };
        // top-1 without log-probability export: the whitening launch keeps the running argmax itself (no [rows][K] export, no selection launch)
        const bool label_in_kernel = bucketed && !logp_out;
        // hard selections: pilots whose selection is too close to call go on the chunk's tie list (QCE_TC_TIE_EPS=0: nobody does)
        const double eps = tc_tie_eps(m);
        const bool refine = want_est && mode != QCE_MODE_ALL && eps > 0.0 && (ts->src.r || ts->src.obs_h);
        QCE_CUDA_TRY(cudaMemsetAsync(ts->tie_list(), 0, sizeof(int), s));
        TcArgs wa = args(nb, nullptr, nullptr, 0, nullptr);
        wa.top_out = label_in_kernel ? b_top : nullptr;
        st = tc_launch_split(m, wa, 1, 0, s);
        if (st) return st;
        if (bucketed) {
            QCE_CUDA_TRY(cudaMemsetAsync(b_cnt, 0, m->n_comp * sizeof(int), s));
            QCE_CUDA_TRY(cudaMemsetAsync(b_perm, 0xFF, (size_t)cap_rows * sizeof(int), s));        // -1 = padding slot
        }
        const bool pair_chunk = pairs && !bucketed;
        const bool fused_count = pair_chunk && m->n_comp <= 256;      // the thread-per-pilot selection counts the pairs itself
        if (pair_chunk) QCE_CUDA_TRY(cudaMemsetAsync(p_cnt, 0, m->n_comp * sizeof(int), s));
        const unsigned char* vb = (const unsigned char*)c.v.bad.p;
        if (!label_in_kernel) {
            float* wts = (want_est && !bucketed) ? (float*)c.v.wts.p : nullptr;
            const int K = m->n_comp;
            if (K <= 256) {
                const size_t sm = (size_t)2 * K * (SEL_ROWS + 1) * sizeof(float) + (size_t)K * sizeof(int);
                static PerDeviceOnce once;
                if (once.first(current_device()))
                    QCE_CUDA_TRY(cudaFuncSetAttribute(tc_select_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                tc_select_rows_kernel<<<(unsigned)((nb + SEL_ROWS - 1) / SEL_ROWS), SEL_THREADS, sm, s>>>((const float2*)c.v.lp2.p, nb, K, mode, n_top, rho, m->flags,
                    wts, c.logp, b_top, vb, ts->tie_list(), eps, m->logc, 1.0 / m->n_obs, fused_count ? p_cnt : nullptr, pair_thresh);
            } else {
                tc_select_kernel<32><<<(unsigned)((nb + 7) / 8), 256, 0, s>>>((const float2*)c.v.lp2.p, nb, K, mode, n_top, rho, m->flags, wts, c.logp, b_top, vb, ts->tie_list(), eps, nullptr, m->logc, 1.0 / m->n_obs);
            }
            QCE_CHECK_LAUNCH("tc_select kernel");
        }
        if (!want_est) continue;
        if (refine) {      // (weight rows / labels overwritten)
            st = tc_reselect_ties(m, ts, s, b0, nb, mode, n_top, rho, c.logp, bucketed ? nullptr : (float*)c.v.wts.p, b_top,
                                  fused_count ? p_cnt : nullptr, pair_thresh);
            if (st) return st;
        }
        if (bucketed) {
            tc_bucket_count_kernel<<<(unsigned)((nb + 1023) / 1024), 1024, 0, s>>>(b_top, nb, m->n_comp, b_cnt);
            tc_bucket_scan_kernel<<<1, 1024, 0, s>>>(b_cnt, m->n_comp, bucket_rows, b_off, b_cur, b_ucomp, b_nu);
            tc_bucket_place_kernel<<<(unsigned)((nb + 1023) / 1024), 1024, 0, s>>>(b_top, nb, m->n_comp, b_off, b_cur, b_perm);
            tc_bucket_gather_kernel<<<(unsigned)(cap_rows / TILE_M), 256, 0, s>>>((const unsigned char*)c.v.img.p, b_perm, b_nu, tiles_per_unit,
                                                                                  2 * m->n_obs / 8, m->tc.split_a ? 2 : 1, (unsigned char*)ts->img2.p);
            QCE_CHECK_LAUNCH("tc_bucket kernels");
            TcArgs ba = args(cap_rows, c.h_est, c.h_true, h_true_c64, acc);
            ba.unit_comp = b_ucomp; ba.perm = b_perm; ba.n_units_dev = b_nu; ba.a_img = (const __half*)ts->img2.p;
            st = tc_combine_parts(m, ba, s);
            if (st) return st;
            continue;
        }
        if (pair_chunk) {
            const unsigned g1 = (unsigned)((nb + 1023) / 1024);
            QCE_CUDA_TRY(cudaMemsetAsync(p_perm, 0xFF, (size_t)p_rows * sizeof(int), s));          // -1 = padding slot
            QCE_CUDA_TRY(cudaMemsetAsync(ts->tmp_est.p, 0, (size_t)nb * m->n_ant * 8, s));           // the pair rows are added into zeros
            if (!fused_count) tc_pair_count_kernel<<<g1, 1024, 0, s>>>((const float*)c.v.wts.p, vb, nb, m->n_comp, pair_thresh, p_cnt);
            tc_pair_scan_kernel<<<1, 1024, 0, s>>>(p_cnt, m->n_comp, bucket_rows, (int)(p_units - 1), p_off, p_cur, p_ucomp, p_nu, p_dense);
            tc_pair_place_kernel<<<g1, 1024, 0, s>>>((const float*)c.v.wts.p, vb, nb, m->n_comp, pair_thresh, p_off, p_cur, p_dense, p_perm, p_w);
            tc_bucket_gather_kernel<<<(unsigned)(p_rows / TILE_M), 256, 0, s>>>((const unsigned char*)c.v.img.p, p_perm, p_nu, tiles_per_unit,
                                                                                2 * m->n_obs / 8, m->tc.split_a ? 2 : 1, (unsigned char*)ts->img2.p);
            QCE_CHECK_LAUNCH("tc_pair kernels");
            count_launch(fused_count ? 2 : 3);
            TcArgs pa = args(p_rows, nullptr, nullptr, 0, nullptr);
            pa.unit_comp = p_ucomp; pa.perm = p_perm; pa.n_units_dev = p_nu; pa.a_img = (const __half*)ts->img2.p; pa.slot_w = p_w;
            st = tc_combine_parts(m, pa, s);
            if (st) return st;
            tc_pair_finish_kernel<<<(unsigned)(8 * sm_count()), 256, 0, s>>>((const float2*)ts->tmp_est.p, (double2*)c.h_est, c.h_true, h_true_c64, vb, nb,
                                                                             m->n_ant, p_dense, acc);
            QCE_CHECK_LAUNCH("tc_pair_finish_kernel");
            // ... or, when the pairs were too many, the weighted launch over all K components (returns at once otherwise)
            TcArgs da = args(nb, c.h_est, c.h_true, h_true_c64, acc);
            da.run_flag = p_dense; da.run_flag_want = 1;
            st = tc_combine_parts(m, da, s);
            if (st) return st;
            continue;
        }
        st = tc_combine_parts(m, args(nb, c.h_est, c.h_true, h_true_c64, acc), s);
        if (st) return st;
    }
    return QCE_OK;
}

// ------------------------------------------------------------------------------------------------ fused hard top-1 (small shapes)
// For N <= 32 (any K) and for K <= 8 the three-launch top-1 path (whitening with in-epilogue label -> regroup -> one-component
// combine) costs more than the fused 'all' launch (config 1: 0.91 vs 0.75 ms per 2^20 pilots): there EPI = 3 runs the fused Z|H
// launch with a running argmax in place of the online softmax -- a component that beats the best so far REPLACES the estimate row.
// Pilots whose best two components are too close to call are neither written nor accumulated; they go on the tie list, get their
// K log-likelihoods in complex128 (tc_refine_kernel) and an exact label (tc_select_kernel<., true>), and this kernel writes their
// estimate h = hoff_k + W_k r in complex128 (one warp per listed pilot; the list is 1e-5 .. 1e-3 of the batch).
struct Top1RowsArgs {
    int No, N, K;
    const double2* W;           // [K][N][No]
    const double2* hoff;        // [K][N]
    RowSource src;
    int64_t row0;               // batch row of chunk row 0
    const int* tie_buf;         // [0] count, then chunk rows
    const int* top;             // [chunk rows] exact labels of the listed rows
    double2* h_est;             // chunk base or null
    const void* h_true;         // chunk base or null
    int h_true_c64;
    double* acc;
};

__global__ void __launch_bounds__(256) tc_top1_rows_kernel(const Top1RowsArgs a) {
    extern __shared__ __align__(16) unsigned char t1_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double2* r_s = reinterpret_cast<double2*>(t1_smem) + (size_t)warp * a.No;
    const int n_list = __ldg(a.tie_buf);
    double err = 0.0, pw = 0.0, cnt = 0.0;
    for (int e = blockIdx.x * 8 + warp; e < n_list; e += gridDim.x * 8) {
        const int crow = __ldg(a.tie_buf + 1 + e);
        const int k = __ldg(a.top + crow);
        for (int j = lane; j < a.No; j += 32) {
            const int64_t idx = (a.row0 + crow) * a.No + j;
            double2 v;
            if (a.src.r) {
                v = reinterpret_cast<const double2*>(a.src.r)[idx];
            } else {      // get_observation_nbit with A = I (utils.py:241-251), as in tc_refine_kernel
                double2 h;
                if (a.src.obs_h_c64) { const float2 hf = reinterpret_cast<const float2*>(a.src.obs_h)[idx]; h = make_double2((double)hf.x, (double)hf.y); }
                else h = reinterpret_cast<const double2*>(a.src.obs_h)[idx];
                const double2 wn = reinterpret_cast<const double2*>(a.src.obs_noise)[idx];
                const double2 y = make_double2(__dadd_rn(h.x, __dmul_rn(a.src.obs_noise_scale, wn.x)), __dadd_rn(h.y, __dmul_rn(a.src.obs_noise_scale, wn.y)));
                v = quantize_value(a.src.qt.n_bits, a.src.qt.n_thr, a.src.qt.thr, a.src.qt.labels, y, nullptr);
            }
            r_s[j] = v;
        }
        __syncwarp();
        const double2* __restrict__ Wk = a.W + (size_t)k * a.N * a.No;
        for (int i = lane; i < a.N; i += 32) {
            double2 h = __ldg(a.hoff + (size_t)k * a.N + i);
            const double2* __restrict__ Wrow = Wk + (size_t)i * a.No;
            for (int j = 0; j < a.No; ++j) {
                const double2 w = __ldg(Wrow + j), r = r_s[j];
                h.x = fma(w.x, r.x, h.x); h.x = fma(-w.y, r.y, h.x);
                h.y = fma(w.x, r.y, h.y); h.y = fma(w.y, r.x, h.y);
            }
            if (a.h_est) a.h_est[(size_t)crow * a.N + i] = h;
            if (a.acc && a.h_true) {
                double2 t;
                if (a.h_true_c64) { const float2 tf = reinterpret_cast<const float2*>(a.h_true)[(size_t)crow * a.N + i]; t = make_double2((double)tf.x, (double)tf.y); }
                else t = reinterpret_cast<const double2*>(a.h_true)[(size_t)crow * a.N + i];
                const double dx = h.x - t.x, dy = h.y - t.y;
                err += dx * dx + dy * dy;
                pw += t.x * t.x + t.y * t.y;
            }
        }
        if (lane == 0) cnt += 1.0;
        __syncwarp();
    }
    if (!a.acc) return;
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        err += __shfl_xor_sync(0xffffffffu, err, off);
        pw += __shfl_xor_sync(0xffffffffu, pw, off);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    }
    if (lane == 0 && cnt > 0.0) { atomicAdd(a.acc + 0, err); atomicAdd(a.acc + 1, pw); atomicAdd(a.acc + 2, cnt); }
}

// shapes the fused hard top-1 launch is used for (QCE_TC_HARD=1 / 0 forces it on / off where it is instantiated)
static bool tc_hard_top1_ok(const qce_model* m) {
    if (!tc_instantiated(m) || m->tc.split || m->tc.split_a || !m->tc.triangular) return false;
    if (const char* e = getenv("QCE_TC_HARD")) return atoi(e) != 0;
    return m->n_obs <= 32 || m->n_comp <= 8;          // measured (2^20 pilots): N = 64, K = 16 is already faster regrouped (1.42 vs 1.56 ms)
}

static qce_status tc_run_hard_top1(qce_model* m, TileScratch* ts, cudaStream_t s, int64_t B, double* h_est, const void* h_true, int h_true_c64,
                                   double* acc) {
    const int K = m->n_comp;
    int64_t chunk = tc_chunk_rows(m);
    if (chunk > B) chunk = (B + TC_UNIT_ROWS - 1) / TC_UNIT_ROWS * TC_UNIT_ROWS;
    const double eps = tc_tie_eps(m);
    const bool refine = eps > 0.0 && (ts->src.r || ts->src.obs_h);
    qce_status st = QCE_OK;
    if (refine) {
        st = tc_scratch_aux(ts, (size_t)chunk, (size_t)K);                       // tie list, FP32 pairs of the listed pilots
        if (st) return st;
        st = grow(ts->bidx, (size_t)chunk * sizeof(int));                        // exact labels of the listed pilots
        if (st) return st;
    }
    const int sms = sm_count();
    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
        const int64_t nb = (B - b0) < chunk ? (B - b0) : chunk;
        const TcChunk c = tc_chunk(m, ts, b0, h_est, nullptr, h_true, h_true_c64);
        TcArgs a;
        tc_fill_args(m, &c.v, nb, c.h_est, c.h_true, h_true_c64, acc, &a);
        if (refine) QCE_CUDA_TRY(cudaMemsetAsync(ts->tie_list(), 0, sizeof(int), s));
        else a.tie_buf = nullptr;                                              // nobody is handed to the exact path: every pilot is answered here
        st = tc_launch_fused(m, a, 3, s);
        if (st) return st;
        if (!refine) continue;
        int* top = (int*)ts->bidx.p;
        st = tc_reselect_ties(m, ts, s, b0, nb, QCE_MODE_TOP1, 1, 0.0, nullptr, nullptr, top, nullptr, 0.f);
        if (st) return st;
        Top1RowsArgs ta;
        ta.No = m->n_obs; ta.N = m->n_ant; ta.K = K;
        ta.W = (const double2*)m->W; ta.hoff = (const double2*)m->hoff;
        ta.src = ts->src; ta.row0 = b0; ta.tie_buf = ts->tie_list(); ta.top = top;
        ta.h_est = (double2*)c.h_est; ta.h_true = c.h_true; ta.h_true_c64 = h_true_c64; ta.acc = acc;
        tc_top1_rows_kernel<<<(unsigned)sms, 256, (size_t)8 * m->n_obs * sizeof(double2), s>>>(ta);
        QCE_CHECK_LAUNCH("tc_top1_rows_kernel");
        count_launch(3);
    }
    return QCE_OK;
}

// One estimate of a formatted batch: the fused 'all' launch where the shape has one and nothing is exported, the fused hard top-1
// where tc_hard_top1_ok picks it, the log-probability -> weights -> combination path otherwise; then the complex128 rows.
static qce_status tc_estimate(qce_model* m, TileScratch* ts, cudaStream_t s, int64_t B, int mode, int n_top, double rho, double* h_est,
                              double* logp_out, const void* h_true, int h_true_c64, double* acc) {
    qce_status st;
    if (mode == QCE_MODE_ALL && !logp_out && !m->tc.split) {
        TcArgs a;
        tc_fill_args(m, ts, B, h_est, h_true, h_true_c64, acc, &a);
        st = tc_launch_fused(m, a, 0, s);
    } else if (mode == QCE_MODE_TOP1 && !logp_out && (h_est || acc) && tc_hard_top1_ok(m)) {
        st = tc_run_hard_top1(m, ts, s, B, h_est, h_true, h_true_c64, acc);
    } else {
        st = tc_run_modes(m, ts, s, B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
    }
    if (st) return st;
    return tc_fix_rows(m, ts, s, B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
}

qce_status tc_estimate_formatted(qce_model* m, cudaStream_t s, int64_t B, double* h_est, const void* h_true, int h_true_c64, double* acc) {
    StreamScratch* sc = scratch_find(s);
    TileScratch* ts = sc ? &sc->tc : nullptr;
    if (!ts || ts->owner != m || B > ts->rows) {
        set_error("qce_estimate_formatted: no pilots of this model are formatted on this stream (or fewer than %lld)", (long long)B);
        return QCE_ERR_INVALID;
    }
    if (B == 0) return QCE_OK;
    return tc_estimate(m, ts, s, B, QCE_MODE_ALL, 0, 0.0, h_est, nullptr, h_true, h_true_c64, acc);
}

// pilots given as complex128 values (estimate_from_y): format, then estimate
qce_status launch_dense_tc(qce_model* m, cudaStream_t s, const double* r, int64_t B, int mode, int n_top, double rho,
                           double* h_est, double* logp_out, const void* h_true, int h_true_c64, double* acc) {
    if (B == 0) return QCE_OK;
    RowSource src;
    src.r = r;
    TileScratch* ts = nullptr;
    qce_status st = tc_format_tiles(m, s, B, src, &ts);
    if (st) return st;
    return tc_estimate(m, ts, s, B, mode, n_top, rho, h_est, logp_out, h_true, h_true_c64, acc);
}

// fused Monte-Carlo step: observe (A = I) -> quantise -> estimate -> NMSE accumulators; the quantised pilots never exist in HBM
// other than as the FP16 tile image
qce_status launch_pipeline_tc(qce_model* m, const QuantTables* qt, cudaStream_t s, const void* h, int h_is_c64, const double* noise,
                              double noise_scale, int64_t B, int mode, int n_top, double rho, double* h_est, double* acc) {
    if (B == 0) return QCE_OK;
    RowSource src;
    src.obs_h = h; src.obs_noise = noise; src.obs_noise_scale = noise_scale; src.obs_h_c64 = h_is_c64; src.qt = *qt;
    TileScratch* ts = nullptr;
    qce_status st = tc_format_tiles(m, s, B, src, &ts);
    if (st) return st;
    return tc_estimate(m, ts, s, B, mode, n_top, rho, h_est, nullptr, h, h_is_c64, acc);
}

}  // namespace qce
