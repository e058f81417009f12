// tcgen05 GEMM for sm_100a:  D[M,N] = epilogue( A[M,K] * W[N,K]^T ) on split16 activations (common.cuh).
//
// Precision: the 1e-3 parity bar on predicted (x,y) rules out single-pass bf16 / tf32 / fp16 operands
// (SURVEY.md appendix E.3).  Every operand is a pair of fp16 values (x ~= hi + lo, ~22 mantissa bits) and a product
// is formed as  hi*hi + hi*lo + lo*hi  with fp32 accumulation in TMEM - three kind::f16 MMAs per K step on wide tiles,
// two on narrow ones (the hi and lo weight planes are adjacent in the stage, so one MMA of N = 2 BN computes
// A_hi * [B_hi; B_lo]; see Cfg::kStacked).  Weights are pre-multiplied by a per-tensor power of two so that their lo
// terms stay in fp16's normal range; the epilogue multiplies the accumulator by the inverse (exact).  The tensor core
// adds into its fp32 accumulator with truncation (measured: ~1e-7 relative per chained MMA,
// profiles/r01_tc_precision.md), so the K steps are dealt round-robin onto several TMEM accumulators and the small
// hi*lo / lo*hi products onto separate columns; the epilogue adds them up with fp32 round-to-nearest.
//
// Data movement per CTA (one 128 x BN output tile, K walked in chunks of 64).  Both operands sit in shared memory in
// the SWIZZLE_128B K-major layout (128-byte rows, 16-byte chunks XOR-swizzled by row % 8):
//   * weights: pre-split, pre-swizzled in HBM at model creation (tc_pack_weight) as [k chunk][plane][row][128 B], so a
//     pipeline stage is two contiguous bulk-TMA copies (cp.async.bulk -> UBLKCP, one per plane) completing on an mbarrier;
//   * activations: already split16 in HBM (the producer's epilogue split them), so warps 0-3 stage the A tile with
//     asynchronous 16-byte copies (cp.async -> LDGSTS, zero-filled for im2col padding / row tails; 8 lanes cover one
//     128-byte row on both sides: coalesced reads, conflict-free writes) whose completion arrives on the stage's
//     mbarrier (cp.async.mbarrier.arrive.noinc) - no registers, no conversion, up to kStages chunks in flight.  The
//     7x7 stem reads a zero-bordered split16 NHWC4 copy of the canvas (common.cuh) with the same 16-byte copies; the
//     weight TMA of a stage completes on the SAME mbarrier (128 loader arrivals + 1 expect_tx), one wait per stage;
//   * warp 4 (one lane) issues the TMA copies, warp 5 (one lane) issues tcgen05.mma and owns TMEM;
//   * long reductions on under-filled grids are split over a thread-block cluster (1 x 1 x {2,4}) and reduce-scattered
//     over TMEM lane quarters through distributed shared memory (st.async + mbarrier, no cluster barrier);
//   * all 8 warps then run the epilogue out of TMEM (the epilogue is instruction-issue bound, so it gets two warps per
//     scheduler: warp w owns TMEM lanes 32 (w % 4).. and the column half w / 4 of the tile; software pipelined: the
//     global operands of chunk c+1 are in flight while chunk c is combined): bias / constant add-matrix / residual /
//     ReLU, or - on warps 0-3 only - the fused residual + LayerNorm over the full 256-wide row (each thread owns one
//     row, so no cross-thread reduction), and write split16 (optionally with the value-projection blocks transposed
//     for the attention kernels).
// The kernel is templated on the A-operand addressing mode so that each instantiation carries exactly one loader
// (an earlier all-modes-in-one kernel was ~30k SASS instructions and instruction-cache bound, profiles/r01_*).
#include <cmath>
#include <cstring>
#include <vector>

#include "a_loader.cuh"
#include "tc_common.cuh"

namespace cotr {

int g_tc_variant = 0;                   // bring-up switch (reserved)
int g_use_pdl = 1;                      // programmatic dependent launch (common.cuh); cotr_debug_set_variant bit 8 clears it
long long* g_tc_timestamps = nullptr;   // debug: 64 clock64() stamps per CTA (cotr_debug_set_timestamps), else null
int g_tc_trace_idx = 0;                 // trace mode: launch counter (common.cuh next_trace_block)

namespace {

using namespace tc;

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kThreads = 256;
constexpr uint32_t kAPlane = BM * 128;         // one fp16 plane (hi or lo) of the 128 x 64 A tile: 128 rows x 128 bytes

enum LoaderMode : int { LD_GATHER = 0, LD_CONV = 1, LD_STEM4 = 2 };

__host__ __device__ inline int tc_npad(int N) { return N >= 64 ? ((N + 63) / 64) * 64 : ((N + 15) / 16) * 16; }

template <int BN>
struct Cfg {
    static constexpr uint32_t kBPlane = BN * 128u;                      // BN rows x 128 bytes
    static constexpr uint32_t kStage = 2 * kAPlane + 2 * kBPlane;
    static constexpr int kStagesRaw = (int)((227u * 1024u - 3072u) / kStage);
    static constexpr int kStages = kStagesRaw > 4 ? 4 : kStagesRaw;
    // TMEM accumulators: kMain slots take the hi*hi products round-robin over K steps (the truncating accumulate is a
    // systematic bias that grows with the chain length and adds up across layers), the small lo*hi / hi*lo products
    // go to separate columns.  Consecutive MMAs never chain on the same accumulator where TMEM allows (a chained MMA
    // waits ~110 cycles for its predecessor).
    // Narrow tiles (BN <= 64) are bound by the ~60-cycle issue cost of an M = 128 MMA, not by its math, so there the
    // weight planes are used STACKED: B_hi and B_lo are adjacent in the stage, one MMA of N = 2 BN forms
    // A_hi * [B_hi; B_lo] (main | hi*lo correction in adjacent columns) and a second one of N = BN adds A_lo * B_hi:
    // two MMAs per K step instead of three.
    static constexpr bool kStacked = BN <= 64;
    static constexpr int kMain = BN >= 256 ? 1 : (BN >= 128 ? 2 : (BN == 64 ? 3 : 4));
    static constexpr int kCorr = BN >= 256 ? 1 : 2;                     // separate correction slots of BN columns
    static constexpr uint32_t kMainStride = kStacked ? 2u * BN : BN;    // stacked: [main | hi*lo] pairs
    static constexpr uint32_t kCorrBase = kMain * kMainStride;
    static constexpr uint32_t kAccCols = kCorrBase + kCorr * BN;
    static constexpr int kSmall = kStacked ? kMain + kCorr : kCorr;     // 16-column loads of correction terms per chunk
    // epilogue staging (re-uses the pipeline stages): per warp 2 planes x 32 rows, row pitch padded by 16 bytes
    static constexpr uint32_t kOutPitch = BN * 2u + 16u;
    static constexpr uint32_t kWarpStaging = 2u * 32u * kOutPitch;
    static constexpr int kChunksN = BN / 16;
    // Epilogue warps: the four TMEM lane quarters x kEpiHalves column halves (warp w reads lanes 32 (w % 4) ...,
    // columns [w / 4 * BN / 2, ...)).  The LayerNorm tile (BN = 256) keeps one thread per full row.
    static constexpr int kEpiHalves = (BN >= 32 && BN < 256) ? 2 : 1;
    static constexpr int kChunksW = kChunksN / kEpiHalves;             // 16-column chunks per epilogue warp
    static constexpr int kRing = kChunksW < 4 ? kChunksW : 4;          // epilogue operand prefetch depth
    static constexpr uint32_t kTmemCols = kAccCols <= 32 ? 32 : (kAccCols <= 64 ? 64 : (kAccCols <= 128 ? 128 : (kAccCols <= 256 ? 256 : 512)));
    // behind the stages: 256 bytes of barriers, then the per-column vectors of the deferred LayerNorm (column sums of
    // W' or gamma | beta of this tile's BN columns, staged by two idle warps while the main loop runs), then split-K partials
    static constexpr uint32_t kVecOffset = kStages * kStage + 256;
    static constexpr uint32_t kVecBytes = 2u * BN * 4u + 2u * BM * 8u;   // + (mean, rstd) of the 128 A rows and of the 128 residual rows
    static constexpr uint32_t kSmemBytes = kStages * kStage + 2048 + kVecBytes;     // + alignment slack + barriers + vectors
    // split-K (reduce-scatter over the rows): every CTA of the cluster finishes 128 / ksplit rows of the tile and
    // receives the other CTAs' fp32 partial rows behind the barriers (a dedicated region, so peers may push while this
    // CTA's pipeline is still running); rows of BN * 4 bytes, 16-byte pieces XOR-swizzled by row % 8 (thread-per-row
    // accesses would otherwise all land in the same banks)
    static constexpr uint32_t kPartOffset = kVecOffset + kVecBytes;
    static constexpr uint32_t kPartPitch = BN * 4u;
    static constexpr int kMaxSplit = BN <= 64 ? 4 : 1;
    static constexpr uint32_t kPartMaxBytes = kMaxSplit > 1 ? 96u * kPartPitch : 0u;   // ksplit 4: 3 x 32 rows; 2: 1 x 64 rows
    static_assert(kSmemBytes + kPartMaxBytes <= 227u * 1024u, "split-K partial tiles do not fit");
    static_assert(kStages >= 2, "pipeline needs at least two stages");
    static_assert(kAccCols <= 512, "TMEM has 512 columns");
    static_assert(kStage % 1024 == 0, "stages must stay 1024-byte aligned for SWIZZLE_128B");
};

// global operands of one 16-column epilogue chunk, fetched one chunk ahead of their use
struct EpiOperands {
    float4 bias[4];
    float4 add[4];
    uint4 res_hi[2], res_lo[2];
};

// DLN: the instantiation carries the deferred-LayerNorm operands (GemmParams::a_ln_cs / res_ln_part / ln_part_out) and the
// dataflow dependencies (GemmParams::sync).  The default schedule uses DLN = false kernels, which contain none of it.
template <int BN, bool LN, int MODE, bool DLN>
__global__ void __launch_bounds__(kThreads, 1) gemm_tc_kernel(const GemmParams p, const int npad, long long* __restrict__ ts) {
    using C = Cfg<BN>;
    // debug timeline (ts != null): slot layout documented in tools/bringup.py::gemm_timeline
    long long* my_ts = ts ? ts + (size_t)((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 64 : nullptr;
    const long long t_start = ts ? clock64() : 0;
#define COTR_TS(slot) do { if (my_ts) my_ts[(slot)] = clock64() - t_start; } while (0)
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_addr = smem_u32(smem_raw);
    uint8_t* stage_base = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);      // SWIZZLE_128B needs 1024-byte alignment
    uint64_t* bars = reinterpret_cast<uint64_t*>(stage_base + C::kStages * C::kStage);
    uint64_t* full_a = bars;
    uint64_t* full_b = bars + C::kStages;
    uint64_t* empty = bars + 2 * C::kStages;
    uint64_t* accum_full = bars + 3 * C::kStages;
    uint64_t* part_full = bars + 3 * C::kStages + 1;       // split-K leader: all peers' partial tiles have landed
    uint64_t* vec_full = bars + 3 * C::kStages + 2;        // deferred LayerNorm: the per-column vectors are staged
    uint64_t* dep_ready = bars + 3 * C::kStages + 3;       // dataflow mode: the polling thread has seen the producer's counters
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 3 * C::kStages + 4);
    const bool dflow = DLN && p.sync.dep_mode != DEP_PDL;  // counters in global memory instead of griddepcontrol.wait (common.cuh)
    float* vec_a = reinterpret_cast<float*>(stage_base + C::kVecOffset);      // a_ln: column sums of W'; res_ln: gamma
    float* vec_b = vec_a + BN;                                                  //                         res_ln: beta
    float2* st_a = reinterpret_cast<float2*>(vec_b + BN);                       // (mean, rstd) of the A rows of this tile
    float2* st_r = st_a + BM;                                                   // (mean, rstd) of the residual rows
    // deferred LayerNorm (GemmParams::a_ln_cs / res_ln_part / ln_part_out): only the row-major loader instantiations carry it
    static_assert(!DLN || (MODE == LD_GATHER && !LN), "deferred LayerNorm / dataflow: row-major operand tiles only");
    constexpr bool kCanLnA = DLN;
    const bool has_aln = kCanLnA && p.a_ln_cs != nullptr;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    // split-K: gridDim.z CTAs of one cluster (cluster dims 1 x 1 x gridDim.z) share the output tile; CTA z walks the
    // K chunks [it0, it0 + KC) and then finishes the TMEM lane quarters (32-row groups) it owns: the other CTAs hand
    // it their partial sums of those rows through distributed shared memory - asynchronous remote stores (st.async)
    // that complete transaction bytes on an mbarrier of the owner, so the hand-over needs no cluster-wide barrier
    // (measured ~2.3k cycles) and each CTA receives only (ksplit-1)/ksplit of a tile (DSMEM moves ~20 bytes / cycle).
    const int ksplit = gridDim.z;
    const int kz = blockIdx.z;
    const int KC = ((p.K + BK - 1) / BK) / ksplit;
    const int it0 = kz * KC;

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::kStages; ++s) {
            mbar_init(&full_a[s], 129);
            mbar_init(&full_b[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accum_full, 1);
        mbar_init(part_full, 1);
        if (DLN) {
            mbar_init(vec_full, 64);
            mbar_init(dep_ready, 1);
        }
        mbar_fence_init();
        if (ksplit > 1) mbar_arrive_expect_tx(part_full, (uint32_t)(ksplit - 1) * (uint32_t)(BM / ksplit) * C::kPartPitch);
    }
    if (warp == 5) tmem_alloc(tmem_ptr, C::kTmemCols);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // split-K: tell the cluster that this CTA runs and its barriers exist (waited for just before the first remote access)
    if (ksplit > 1) cluster_arrive();
    if (threadIdx.x == 0) COTR_TS(1);

    if (warp < 4) {
        // ================= A producer ===========================================================================
        const int t = threadIdx.x;
        const int kg = t & 7;          // 16-byte K group (8 halves) inside the 64-wide chunk
        const int rb = t >> 3;         // rows rb, rb+16, ..., rb+112  (row % 8 == rb % 8 for all of them)
        ARow rows[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) rows[i] = decode_a_row(p, m0 + rb + 16 * i);
        const uint32_t a_off = (uint32_t)rb * 128u + (uint32_t)((kg ^ (rb & 7)) << 4);   // swizzled chunk position
        const uint32_t dst0 = smem_u32(stage_base) + a_off;
        // everything above (and the weight TMA of warp 4) overlaps the previous kernel; activations do not
        // Let the next kernel of the stream / graph start its prologue (barriers, TMEM, weight TMA) on idle SMs now; it
        // still waits (griddepcontrol.wait) for this grid to complete before touching activations.  (Same-box A/B:
        // triggering here beats triggering after the wait by 0.5%, triggering at kernel entry loses 1.4%.)
        if (threadIdx.x == 0) {
            pdl_launch_dependents();
            if (dflow) { dep_wait_thread(p.sync, blockIdx.x); mbar_arrive(dep_ready); }
        }
        if (dflow) mbar_wait(dep_ready, 0); else pdl_wait();
        if (threadIdx.x == 0) COTR_TS(2);

#pragma unroll 1
        for (int it = 0; it < KC; ++it) {
            const int s = it % C::kStages;
            const uint32_t ph = (uint32_t)(it / C::kStages) & 1u;
            mbar_wait(&empty[s], ph ^ 1u);
            if (threadIdx.x == 0 && it < 8) COTR_TS(3 + 2 * it);
            const int k0 = (it0 + it) * BK;
            {
                const uint32_t dst = dst0 + (uint32_t)s * C::kStage;
                int kh = 0, kw = 0, koff = k0 + kg * 8;          // LD_GATHER: koff = column inside the row
                if constexpr (MODE == LD_CONV) {                 // C % 64 == 0: the chunk lies inside one filter tap
                    const int tap = k0 / p.C;
                    koff = k0 - tap * p.C + kg * 8;
                    kh = tap / p.KW;
                    kw = tap - kh * p.KW;
                }
                if constexpr (MODE == LD_STEM4) {               // filter row kh = 64 contiguous bytes of the bordered canvas
                    const int kk = k0 + kg * 8;
                    koff = (kk >> 5) * (kStemCanvasPitch * 4) + (kk & 31);
                }
                const bool k_ok = (k0 + kg * 8) < p.K;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    bool ok = rows[i].valid && k_ok;
                    size_t off = rows[i].off + koff;
                    if constexpr (MODE == LD_CONV) {
                        const int ih = rows[i].ih0 + kh, iw = rows[i].iw0 + kw;
                        ok = ok && ih >= 0 && ih < p.H && iw >= 0 && iw < p.W;
                        off = rows[i].off + ((size_t)ih * p.W + iw) * p.C + koff;
                    }
                    if (!ok) off = 0;                            // src-size 0 -> 16 bytes of zeros, address unused
                    const uint32_t bytes = ok ? 16u : 0u;
                    cp_async16(dst + i * 2048, p.a.hi + off, bytes);                  // 16 rows x 128 bytes further down
                    cp_async16(dst + kAPlane + i * 2048, p.a.lo + off, bytes);
                }
                cp_async_mbar_arrive_noinc(&full_a[s]);
            }
            if (threadIdx.x == 0 && it < 8) COTR_TS(4 + 2 * it);
        }
    } else if (warp == 4) {
        // ================= weight producer: bulk TMA of the pre-swizzled fp16 hi/lo image ========================
        if (lane == 0) {
            const uint8_t* wimg = reinterpret_cast<const uint8_t*>(p.Wtc);
#pragma unroll 1
            for (int it = 0; it < KC; ++it) {
                const int s = it % C::kStages;
                const uint32_t ph = (uint32_t)(it / C::kStages) & 1u;
                mbar_wait(&empty[s], ph ^ 1u);
                mbar_arrive_expect_tx(&full_a[s], 2u * C::kBPlane);
                uint8_t* b_dst = stage_base + (size_t)s * C::kStage + 2 * kAPlane;
                // image: [k chunk][plane][npad rows][128 bytes]; the BN rows of this tile are contiguous per plane
                const uint8_t* src = wimg + (((size_t)(it0 + it) * 2) * npad + n0) * 128;
                tma_bulk_g2s(b_dst, src, C::kBPlane, &full_a[s]);
                tma_bulk_g2s(b_dst + C::kBPlane, src + (size_t)npad * 128, C::kBPlane, &full_a[s]);
                if (it < 8) COTR_TS(44 + it);
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        // ================= MMA issuer ===========================================================================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_f16_f32(BM, BN);
            constexpr uint32_t idesc2 = make_idesc_f16_f32(BM, C::kStacked ? 2 * BN : BN);
            const uint32_t hi_word = desc_hi_sw128();
            const uint32_t corr_a = tmem_base + C::kCorrBase;
            const uint32_t corr_b = tmem_base + C::kCorrBase + (uint32_t)(C::kCorr - 1) * BN;
#pragma unroll 1
            for (int it = 0; it < KC; ++it) {
                const int s = it % C::kStages;
                const uint32_t ph = (uint32_t)(it / C::kStages) & 1u;
                mbar_wait(&full_a[s], ph);
                if (it < 8) COTR_TS(24 + 2 * it);
                tcgen05_fence_after();
                const uint32_t a_addr = smem_u32(stage_base + (size_t)s * C::kStage);
                const uint32_t a_h0 = desc_lo_sw128(a_addr);
                const uint32_t b_h0 = desc_lo_sw128(a_addr + 2 * kAPlane);
#pragma unroll
                for (int ks = 0; ks < BK / 16; ++ks) {
                    const int g = it * (BK / 16) + ks;                       // global K step
                    // a K step of 16 halves = 32 bytes inside the 128-byte swizzle atom: +2 in the address field
                    const uint64_t dah = make_desc(a_h0 + 2 * ks, hi_word);
                    const uint64_t dal = make_desc(a_h0 + (kAPlane >> 4) + 2 * ks, hi_word);
                    const uint64_t dbh = make_desc(b_h0 + 2 * ks, hi_word);
                    const uint64_t dbl = make_desc(b_h0 + (C::kBPlane >> 4) + 2 * ks, hi_word);
                    const uint32_t main_col = tmem_base + (uint32_t)(g % C::kMain) * C::kMainStride;
                    if constexpr (C::kStacked) {
                        // the descriptor of B_hi with N = 2 BN runs on into the B_lo plane (next 8-row groups)
                        umma_f16_ss(tmem_base + C::kCorrBase + (uint32_t)(g & 1) * BN, dal, dbh, idesc, g >= 2);
                        umma_f16_ss(main_col, dah, dbh, idesc2, g >= C::kMain);
                    } else {
                        umma_f16_ss(corr_a, dal, dbh, idesc, g != 0);
                        umma_f16_ss(main_col, dah, dbh, idesc, g >= C::kMain);
                        umma_f16_ss(corr_b, dah, dbl, idesc, C::kCorr == 1 ? true : g != 0);
                    }
                }
                umma_commit(&empty[s]);          // frees the stage once these MMAs have read it
                if (it < 8) COTR_TS(25 + 2 * it);
            }
            umma_commit(accum_full);
            COTR_TS(41);
        }
        __syncwarp();
    } else if (kCanLnA && !LN && (has_aln || p.res_ln_part != nullptr)) {
        // ================= warps 6-7: operands of the deferred LayerNorm ==========================================
        // (1) the constant per-column vectors of this tile (model constants: their loads are issued before the
        // dependency wait and land while it lasts);
        const int u = (warp - 6) * 32 + lane;
        const float* src_a = has_aln ? p.a_ln_cs : p.res_ln_gamma;
        float va[(BN + 63) / 64], vb[(BN + 63) / 64];
#pragma unroll
        for (int k = 0; k < (BN + 63) / 64; ++k) {
            const int i = u + 64 * k;
            const bool ok = i < BN && n0 + i < p.N;
            va[k] = ok ? __ldg(src_a + n0 + i) : 0.f;
            vb[k] = (ok && !has_aln) ? __ldg(p.res_ln_beta + n0 + i) : 0.f;
        }
        if (dflow) mbar_wait(dep_ready, 0); else pdl_wait();
        // (2) (mean, rstd) of the 128 rows of this tile from the 16 partial statistics per row their producer's epilogue
        // left behind ((mean, M2) per 16-column chunk, GemmParams::ln_part_out).  8 lanes read one row's 128-byte line
        // (coalesced: 4 rows per instruction, all 16 loads of a lane in flight before the first use) and add up
        //     S1 = sum mean_i,  S2 = sum mean_i^2,  S3 = sum M2_i     (3 butterfly steps)
        // -> mean = S1 / 16,  M2 = S3 + 16 (S2 - S1^2 / 16)  (the chunk means are of the row's own magnitude, so the
        // difference is benign).  ld.global.cg, never .nc: the producer may still have been running when this CTA
        // became resident (see load8_split).
        auto stage_stats = [&](const float2* part, float2* dst) {
            const int sub = lane & 7;                      // which 16 bytes (2 partials) of the row's line
            float4 ld[16];
#pragma unroll
            for (int it = 0; it < 16; ++it) {
                const int grow = m0 + (warp - 6) * 64 + it * 4 + (lane >> 3);
                ld[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (grow < p.M) ld[it] = __ldcg(reinterpret_cast<const float4*>(part + (size_t)grow * 16) + sub);
            }
#pragma unroll
            for (int it = 0; it < 16; ++it) {
                const float4 t4 = ld[it];
                // chunk means relative to the row's first chunk mean: the sums below then do not cancel
                const float ref = __shfl_sync(0xffffffffu, t4.x, lane & ~7);
                const float d0 = t4.x - ref, d1 = t4.z - ref;
                float s1 = d0 + d1;
                float s2 = fmaf(d0, d0, d1 * d1);
                float s3 = t4.y + t4.w;
#pragma unroll
                for (int step = 1; step < 8; step <<= 1) {
                    s1 += __shfl_xor_sync(0xffffffffu, s1, step);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, step);
                    s3 += __shfl_xor_sync(0xffffffffu, s3, step);
                }
                const float mean = fmaf(s1, 1.f / 16.f, ref);
                const float m2 = s3 + fmaxf(fmaf(16.f, s2, -s1 * s1), 0.f);          // sum M2_i + 16 sum (mean_i - mean)^2
                if (sub == 0) dst[(warp - 6) * 64 + it * 4 + (lane >> 3)] = make_float2(mean, rsqrtf(m2 * (1.f / 256.f) + 1e-5f));
            }
        };
        for (int k = 0; k < (BN + 63) / 64; ++k) {
            const int i = u + 64 * k;
            if (i < BN) { vec_a[i] = va[k]; vec_b[i] = vb[k]; }
        }
        if (has_aln) stage_stats(p.a_ln_part, st_a);
        if (p.res_ln_part != nullptr) stage_stats(p.res_ln_part, st_r);
        mbar_arrive(vec_full);
    }

    // ================= epilogue: TMEM -> registers -> global ======================================================
    // Warps 0-3 arrive here when their last copies are issued, warps 4/5 when the last TMA / MMA is issued, 6/7 at once.
    const int ew = warp & 3;                 // TMEM lane quarter this warp may read
    const int half = warp >> 2;              // column half of the tile it handles
    if (ksplit > 1) cluster_wait();          // every CTA of the cluster has started (long ago by now)
    if (half < C::kEpiHalves) {
        if (warp >= 4) { if (dflow) mbar_wait(dep_ready, 0); else pdl_wait(); }      // residual / add operands come from the previous kernels
        const int cbeg = half * C::kChunksW * 16;
        const int row = m0 + ew * 32 + lane;
        // split-K: lane quarter q is finished by CTA q * ksplit / 4; the other CTAs only contribute partial sums
        const int owner = (ew * ksplit) >> 2;
        const bool mine = owner == kz;
        const bool row_ok = mine && row < p.M;
        const uint32_t trow = tmem_base + ((uint32_t)(ew * 32) << 16);
        const float* add_row = (row_ok && p.addmat) ? p.addmat + (size_t)(row % p.add_period) * p.ld_add : nullptr;
        const bool has_res = row_ok && p.res.hi != nullptr;
        const size_t res_off = (size_t)(row_ok ? row : 0) * p.ldr;
        const float acc_scale = p.acc_scale;
        // Deferred LayerNorm: (mean, rstd) of this thread's A row / residual row, staged by warps 6-7
        const bool res_ln = kCanLnA && has_res && p.res_ln_part != nullptr;
        float2 res_st = make_float2(0.f, 1.f);
        float res_shift = 0.f;                          // -mean * rstd of the residual row
        float2 a_st = make_float2(0.f, 1.f);
        const bool emit_part = kCanLnA && row_ok && p.ln_part_out != nullptr;
        const bool tail = p.out_f32 != nullptr && (p.N & 15) != 0;      // only the N = 2 prediction head
        const bool has_bias = p.bias != nullptr && !tail;

        // issue the global loads of the chunk starting at column nb (bias / add-matrix / residual); N % 16 == 0 here
        auto prefetch = [&](int nb, EpiOperands& o) {
            if (nb >= p.N || tail) return;
            if (has_bias) {
#pragma unroll
                for (int j = 0; j < 4; ++j) o.bias[j] = __ldg(reinterpret_cast<const float4*>(p.bias + nb) + j);
            }
            if (add_row) {
#pragma unroll
                for (int j = 0; j < 4; ++j) o.add[j] = __ldg(reinterpret_cast<const float4*>(add_row + nb) + j);
            }
            if (has_res) {
                // 16 halves of one plane = one 32-byte sector: a single 256-bit ld.global.cg per plane (two 128-bit
                // loads would be two L2 requests for the same sector - activations bypass L1, see load8_split)
                ld_cg_256(p.res.hi + res_off + nb, o.res_hi[0], o.res_hi[1]);
                ld_cg_256(p.res.lo + res_off + nb, o.res_lo[0], o.res_lo[1]);
            }
        };
        auto apply = [&](const EpiOperands& o, float (&v)[16], int nb) {
            const int cl = nb - n0;                   // column inside the tile (the staged vectors are tile-local)
            if (kCanLnA && has_aln) {                 // y = rstd * (x W'^T - mean * colsum(W'))
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 cs4 = *reinterpret_cast<const float4*>(vec_a + cl + 4 * j);
                    v[4 * j] = a_st.y * fmaf(-a_st.x, cs4.x, v[4 * j]);
                    v[4 * j + 1] = a_st.y * fmaf(-a_st.x, cs4.y, v[4 * j + 1]);
                    v[4 * j + 2] = a_st.y * fmaf(-a_st.x, cs4.z, v[4 * j + 2]);
                    v[4 * j + 3] = a_st.y * fmaf(-a_st.x, cs4.w, v[4 * j + 3]);
                }
            }
            if (has_bias) {
#pragma unroll
                for (int j = 0; j < 4; ++j) { v[4 * j] += o.bias[j].x; v[4 * j + 1] += o.bias[j].y; v[4 * j + 2] += o.bias[j].z; v[4 * j + 3] += o.bias[j].w; }
            }
            if (add_row) {
#pragma unroll
                for (int j = 0; j < 4; ++j) { v[4 * j] += o.add[j].x; v[4 * j + 1] += o.add[j].y; v[4 * j + 2] += o.add[j].z; v[4 * j + 3] += o.add[j].w; }
            }
            if (has_res) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const uint32_t h[4] = {o.res_hi[j].x, o.res_hi[j].y, o.res_hi[j].z, o.res_hi[j].w};
                    const uint32_t l[4] = {o.res_lo[j].x, o.res_lo[j].y, o.res_lo[j].z, o.res_lo[j].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float2 f = join_f16x2(h[q], l[q]);
                        if (kCanLnA && res_ln) {      // the residual is a deferred LayerNorm of the stored rows
                            const float2 g2 = *reinterpret_cast<const float2*>(vec_a + cl + 8 * j + 2 * q);
                            const float2 b2 = *reinterpret_cast<const float2*>(vec_b + cl + 8 * j + 2 * q);
                            f.x = fmaf(fmaf(f.x, res_st.y, res_shift), g2.x, b2.x);
                            f.y = fmaf(fmaf(f.y, res_st.y, res_shift), g2.y, b2.y);
                        }
                        v[8 * j + 2 * q] += f.x;
                        v[8 * j + 2 * q + 1] += f.y;
                    }
                }
            }
        };
        // v[0..15] = acc_scale * (sum over all accumulators of columns [c, c+16)); all TMEM loads of the chunk are
        // issued back to back and waited for once.
        constexpr uint32_t kPartPitch = C::kPartPitch, kPartOffset = C::kPartOffset;
        const uint32_t part_slot = (uint32_t)(BM / ksplit) * kPartPitch;       // one source CTA's rows in the owner's region
        const uint32_t part_row = (uint32_t)((ew - owner * (4 / ksplit)) * 32 + lane) * kPartPitch;   // row inside a slot
        const uint32_t part_swz = (uint32_t)(lane & 7);                        // == row % 8
        // v = sum over all accumulators of columns [c, c+16), unscaled: the correction terms first (small), then the
        // main slots, RN adds; the TMEM loads of each group are issued back to back and waited for once.
        auto sum_acc = [&](int c, float (&v)[16]) {
            float x[16];
            {
                uint32_t r[C::kSmall][16];
                __syncwarp();
#pragma unroll
                for (int a = 0; a < C::kCorr; ++a) tmem_ld16_issue(trow + C::kCorrBase + a * BN + c, r[a]);
                if constexpr (C::kStacked) {
#pragma unroll
                    for (int a = 0; a < C::kMain; ++a) tmem_ld16_issue(trow + a * C::kMainStride + BN + c, r[C::kCorr + a]);
                }
#pragma unroll
                for (int a = 0; a < C::kSmall; ++a) tmem_ld16_fence(r[a]);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    x[j] = __uint_as_float(r[0][j]);
#pragma unroll
                    for (int a = 1; a < C::kSmall; ++a) x[j] += __uint_as_float(r[a][j]);
                }
            }
            uint32_t r[C::kMain][16];
#pragma unroll
            for (int a = 0; a < C::kMain; ++a) tmem_ld16_issue(trow + a * C::kMainStride + c, r[a]);
#pragma unroll
            for (int a = 0; a < C::kMain; ++a) tmem_ld16_fence(r[a]);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float y = __uint_as_float(r[0][j]);
#pragma unroll
                for (int a = 1; a < C::kMain; ++a) y += __uint_as_float(r[a][j]);
                v[j] = x[j] + y;
            }
        };
        // own sums -> final accumulator: add the peers' partial rows (split-K owner), undo the weight pre-scaling
        auto finish_acc = [&](int c, float (&v)[16]) {
            if (ksplit > 1) {                             // owner: add the partial sums the peers pushed over DSMEM
                const uint8_t* part = stage_base + kPartOffset + part_row;
                for (int peer = 0; peer < ksplit - 1; ++peer) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const uint32_t piece = ((uint32_t)((c + j) >> 2) ^ part_swz) << 4;
                        const float4 t4 = *reinterpret_cast<const float4*>(part + (uint32_t)peer * part_slot + piece);
                        v[j] += t4.x; v[j + 1] += t4.y; v[j + 2] += t4.z; v[j + 3] += t4.w;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] *= acc_scale;
        };
        auto load_acc = [&](int c, float (&v)[16]) {
            sum_acc(c, v);
            finish_acc(c, v);
        };

        // Output path.  split16 row-major tiles are staged in shared memory (the pipeline stages are idle once the
        // accumulator is complete) and written out as full coalesced rows; a thread-per-row direct store would touch
        // 32 different cache lines per instruction.  The two warps of a lane quarter stage their column halves into the
        // same 32-row region, meet on a named barrier and drain one fp16 plane each.  Transposed value blocks and the
        // fp32 prediction head keep the direct path.
        size_t tile_base = 0;
        const bool direct = p.out_f32 != nullptr || out_location(p, m0, n0, tile_base);
        uint8_t* stg = stage_base + (uint32_t)ew * C::kWarpStaging + (uint32_t)lane * C::kOutPitch;
        auto emit16 = [&](int c, const float (&v)[16]) {          // c = column inside the tile
            if (direct) {
                if (row_ok && n0 + c < p.N) store16(p, row, n0 + c, v);
                return;
            }
            uint4 h0, l0, h1, l1;
            split_f16x2(v[0], v[1], h0.x, l0.x);   split_f16x2(v[2], v[3], h0.y, l0.y);
            split_f16x2(v[4], v[5], h0.z, l0.z);   split_f16x2(v[6], v[7], h0.w, l0.w);
            split_f16x2(v[8], v[9], h1.x, l1.x);   split_f16x2(v[10], v[11], h1.y, l1.y);
            split_f16x2(v[12], v[13], h1.z, l1.z); split_f16x2(v[14], v[15], h1.w, l1.w);
            uint8_t* d = stg + c * 2;
            *reinterpret_cast<uint4*>(d) = h0;
            *reinterpret_cast<uint4*>(d + 16) = h1;
            *reinterpret_cast<uint4*>(d + 32 * C::kOutPitch) = l0;
            *reinterpret_cast<uint4*>(d + 32 * C::kOutPitch + 16) = l1;
        };
        auto drain_plane = [&](int plane) {
            constexpr int kLanesPerRow = BN * 2 / 16;                     // 16-byte pieces per row of one plane
            constexpr int kRowsPerPass = kLanesPerRow >= 32 ? 1 : 32 / kLanesPerRow;
            constexpr int kPiecesPerLane = kLanesPerRow > 32 ? kLanesPerRow / 32 : 1;
            const uint8_t* wbase = stage_base + (uint32_t)ew * C::kWarpStaging;
            const int r_in = kLanesPerRow >= 32 ? 0 : lane / kLanesPerRow;
            const int piece0 = kLanesPerRow >= 32 ? lane : lane % kLanesPerRow;
            __half* gout = (plane == 0 ? p.out.hi : p.out.lo) + tile_base;     // element (m0, n0 mapped)
#pragma unroll 4
            for (int r0 = 0; r0 < 32; r0 += kRowsPerPass) {
                const int rr = r0 + r_in;
                const int grow_ = m0 + ew * 32 + rr;
#pragma unroll
                for (int q = 0; q < kPiecesPerLane; ++q) {
                    const int piece = piece0 + q * 32;
                    const uint4 val = *reinterpret_cast<const uint4*>(wbase + (uint32_t)(plane * 32 + rr) * C::kOutPitch + piece * 16);
                    if (grow_ < p.M)
                        *reinterpret_cast<uint4*>(gout + (size_t)(ew * 32 + rr) * p.ldc + piece * 8) = val;
                }
            }
        };
        auto drain = [&]() {
            if (direct) return;
            if constexpr (C::kEpiHalves == 2) {
                named_barrier_sync(1 + ew, 64);                           // both column halves of these 32 rows are staged
                drain_plane(half);
            } else {
                __syncwarp();
                drain_plane(0);
                drain_plane(1);
            }
        };

        // The loader warps finish issuing their copies several pipeline stages before the last MMA retires: use that
        // slack to get the epilogue's global operands in flight (kRing chunks deep), then keep the ring full.
        EpiOperands ops[C::kRing];
        const int nbase = (LN ? 0 : n0) + cbeg;
#pragma unroll
        for (int i = 0; i < C::kRing; ++i) prefetch(nbase + 16 * i, ops[i]);
        mbar_wait(accum_full, 0);
        tcgen05_fence_after();
        if (kCanLnA && (has_aln || p.res_ln_part != nullptr)) {
            mbar_wait(vec_full, 0);
            if (has_aln) a_st = st_a[ew * 32 + lane];
            if (res_ln) { res_st = st_r[ew * 32 + lane]; res_shift = -res_st.x * res_st.y; }
        }
        if (threadIdx.x == 0) COTR_TS(20);
        // Narrow tiles read their own accumulators into registers right away: senders push them, owners overlap the
        // TMEM round trips with the wait for the peers' partial rows.
        constexpr bool kPreload = !LN && C::kChunksW <= 2;
        float pre[kPreload ? C::kChunksW : 1][16];
        if constexpr (kPreload) {
#pragma unroll
            for (int ci = 0; ci < C::kChunksW; ++ci) sum_acc(cbeg + ci * 16, pre[ci]);
        }
        if (C::kMaxSplit > 1 && ksplit > 1) {
            if (!mine) {
                // the partial rows have their own region in the owner's shared memory: push as soon as this CTA's
                // MMAs have retired, whatever the owner is doing (source slot: this CTA's rank among the non-owners)
                const uint32_t local = smem_u32(stage_base) + kPartOffset + (uint32_t)(kz < owner ? kz : kz - 1) * part_slot + part_row;
                const uint32_t remote = map_to_cta(local, (uint32_t)owner);
                const uint32_t remote_bar = map_to_cta(smem_u32(part_full), (uint32_t)owner);
                // unscaled partial sums travel; the leader applies acc_scale once in load_acc
#pragma unroll
                for (int ci = 0; ci < C::kChunksW; ++ci) {
                    const int c = cbeg + ci * 16;
                    const float (&v)[16] = pre[kPreload ? ci : 0];      // (split-K only exists on preloading tiles)
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                        st_async_f32x4(remote + (((uint32_t)((c + j) >> 2) ^ part_swz) << 4), v[j], v[j + 1], v[j + 2], v[j + 3], remote_bar);
                }
                if (threadIdx.x == 0) COTR_TS(22);
            } else {
                if (threadIdx.x == 0) COTR_TS(22);
                mbar_wait(part_full, 0);             // (ksplit - 1) x (128 / ksplit) rows x BN floats have landed
                if (threadIdx.x == 0) COTR_TS(23);
            }
        }
        if (mine) {

        if constexpr (!LN) {
#pragma unroll
            for (int ci = 0; ci < C::kChunksW; ++ci) {
                const int c = cbeg + ci * 16;
                const int nb = n0 + c;
                float v[16];
                if constexpr (kPreload) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = pre[ci][j];
                    finish_acc(c, v);
                } else {
                    load_acc(c, v);
                }
                if (threadIdx.x == 0 && ci < 2) COTR_TS(30 + 4 * ci);
                if (BN > 16 || !tail) {                          // (a ragged N only exists in the 16-wide instantiation)
                    apply(ops[ci % C::kRing], v, nb);
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)                 // static indexing keeps v[] in registers
                        if (p.bias && nb + j < p.N) v[j] += __ldg(p.bias + nb + j);
                }
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
                }
                if (kCanLnA && emit_part) {
                    // (mean, M2) of these 16 final values for the consumers' deferred LayerNorm
                    float sm = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) sm += v[j];
                    sm *= (1.f / 16.f);
                    float m2 = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) { const float d = v[j] - sm; m2 = fmaf(d, d, m2); }
                    p.ln_part_out[(size_t)row * 16 + (nb >> 4)] = make_float2(sm, m2);
                }
                if (threadIdx.x == 0 && ci < 2) COTR_TS(31 + 4 * ci);
                emit16(c, v);
                if (threadIdx.x == 0 && ci < 2) COTR_TS(32 + 4 * ci);
                if (ci + C::kRing < C::kChunksW) prefetch(nb + 16 * C::kRing, ops[ci % C::kRing]);
            }
            if (threadIdx.x == 0) COTR_TS(38);
            drain();
        } else {
            // fused residual + LayerNorm (eps 1e-5, biased variance) over the 256 columns this thread owns.  One pass
            // over the accumulators: sum and shifted sum of squares (shift = the row's first value, so the
            // E[(x-s)^2] - (mean-s)^2 form does not cancel), values parked back in TMEM for the normalisation pass.
            float sum = 0.f, sq = 0.f, shift = 0.f;
#pragma unroll
            for (int ci = 0; ci < C::kChunksN; ++ci) {
                const int c = ci * 16;
                float v[16];
                load_acc(c, v);
                apply(ops[ci % C::kRing], v, c);
                if (ci + C::kRing < C::kChunksN) prefetch(c + 16 * C::kRing, ops[ci % C::kRing]);
                if (ci == 0) shift = v[0];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    sum += v[j];
                    const float d = v[j] - shift;
                    sq = fmaf(d, d, sq);
                }
                tmem_st16(trow + c, v);
            }
            tmem_st_wait();
            const float mean = sum * (1.f / 256.f);
            const float dm = mean - shift;
            const float var = fmaxf(sq * (1.f / 256.f) - dm * dm, 0.f);
            const float rstd = 1.f / sqrtf(var + 1e-5f);
#pragma unroll 1
            for (int c = 0; c < BN; c += 32) {
                uint32_t r[2][16];
                __syncwarp();
                tmem_ld16_issue(trow + c, r[0]);
                tmem_ld16_issue(trow + c + 16, r[1]);
                tmem_ld16_fence(r[0]);
                tmem_ld16_fence(r[1]);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.ln_gamma + c + h * 16 + j));
                        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.ln_beta + c + h * 16 + j));
                        v[j] = (__uint_as_float(r[h][j]) - mean) * rstd * g4.x + b4.x;
                        v[j + 1] = (__uint_as_float(r[h][j + 1]) - mean) * rstd * g4.y + b4.y;
                        v[j + 2] = (__uint_as_float(r[h][j + 2]) - mean) * rstd * g4.z + b4.z;
                        v[j + 3] = (__uint_as_float(r[h][j + 3]) - mean) * rstd * g4.w + b4.w;
                    }
                    emit16(c + h * 16, v);
                }
            }
            drain();
        }
        }   // leader / unsplit epilogue
        if (threadIdx.x == 0) COTR_TS(21);
    }

    tcgen05_fence_before();
    __syncthreads();
    if (DLN && threadIdx.x == 0) dep_signal_thread(p.sync, blockIdx.x);       // every store of this CTA precedes the barrier above
    if (warp == 5) tmem_dealloc(tmem_base, C::kTmemCols);
    if (threadIdx.x == 160) COTR_TS(60);
    if (my_ts && threadIdx.x == 160) my_ts[62] = global_ns();
#undef COTR_TS
}

thread_local GemmLaunchInfo* g_launch_info = nullptr;       // where launch_one reports the grid it chose

template <int BN, bool LN, int MODE, bool DLN = false>
int launch_one(const GemmParams& p, cudaStream_t s) {
    using C = Cfg<BN>;
    static unsigned long long configured = 0;      // bit per device
    if (first_use_on_device(&configured)) {
        COTR_CHECK_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, LN, MODE, DLN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(C::kSmemBytes + C::kPartMaxBytes)));
    }
    const int npad = tc_npad(p.N);
    dim3 grid((p.M + BM - 1) / BM, (p.N + BN - 1) / BN);
    // Split-K over a thread-block cluster for long reductions on under-filled grids (the K loop is the serial part of
    // these latency-bound launches): 4 or 2 CTAs per output tile, each >= 4 chunks, at most ~one wave of CTAs.
    // The grid fill is that of the scheduling row count (GemmParams::M_sched): a larger launch may run split-K over
    // several waves, so that its rows are summed in the same order as at the scheduling size.
    int ksplit = 1;
    if constexpr (!LN && BN <= 64 && MODE != LD_STEM4) {
        const int kc = (p.K + BK - 1) / BK;
        const int m_sched = p.M_sched > 0 ? p.M_sched : p.M;
        const long long ctas = (long long)((m_sched + BM - 1) / BM) * grid.y;
        if (!(g_tc_variant & 512) && kc >= (16 >> ((g_tc_variant >> 14) & 3))) {     // bring-up knob: bits 14-15
            if (C::kMaxSplit >= 4 && kc % 4 == 0 && ctas * 4 <= 160) ksplit = 4;
            else if (C::kMaxSplit >= 2 && kc % 2 == 0 && ctas * 2 <= 160) ksplit = 2;
        }
    }
    COTR_CHECK(p.a_ln_cs == nullptr || (DLN && p.K == 256 && p.a_mode == A_ROWMAJOR && p.a_ln_part != nullptr),
               "gemm_tc: the deferred LayerNorm on A needs a row-major operand with K = 256 and its partial statistics");
    COTR_CHECK((p.res_ln_part == nullptr && p.ln_part_out == nullptr && p.sync.dep_mode == DEP_PDL && p.sync.sig == nullptr) || DLN,
               "gemm_tc: deferred-LayerNorm residual / statistics on an unsupported tile");
    COTR_CHECK(p.ln_part_out == nullptr || (p.N == 256 && !p.remap && p.out_f32 == nullptr), "gemm_tc: row statistics need a plain N = 256 output");
    grid.z = ksplit;
    const size_t smem = C::kSmemBytes + (size_t)(ksplit - 1) * (BM / ksplit) * C::kPartPitch;     // incoming partial rows
    if (g_launch_info) *g_launch_info = GemmLaunchInfo{(int)grid.x, (int)grid.y, ksplit};
    COTR_CHECK_CUDA(launch_kernel_cluster(gemm_tc_kernel<BN, LN, MODE, DLN>, grid, dim3(kThreads), smem, s, ksplit, p, npad, next_trace_block()));
    return 0;
}

template <int BN, bool LN>
int launch_mode(const GemmParams& p, cudaStream_t s) {
    const bool gather = (p.a_mode == A_ROWMAJOR || p.a_mode == A_TOKENS);
    if (gather && (p.K & 7) == 0 && (p.lda & 7) == 0) {
        if constexpr (!LN) {
            const bool dln = p.a_ln_cs != nullptr || p.res_ln_part != nullptr || p.ln_part_out != nullptr ||
                             p.sync.dep_mode != DEP_PDL || p.sync.sig != nullptr;
            if (dln) return launch_one<BN, LN, LD_GATHER, true>(p, s);
        }
        return launch_one<BN, LN, LD_GATHER>(p, s);
    }
    if constexpr (!LN && BN >= 32) {
        if (p.a_mode == A_CONV_NHWC && (p.C & 63) == 0) return launch_one<BN, LN, LD_CONV>(p, s);
    }
    if constexpr (!LN && BN == 64) {
        if (p.a_mode == A_STEM_NHWC4 && p.K == kStemK) return launch_one<64, false, LD_STEM4>(p, s);
    }
    set_error("gemm_tc: no kernel instantiation for a_mode %d, K %d, lda %d, C %d with tile N %d", p.a_mode, p.K, p.lda, p.C, BN);
    return 1;
}

inline uint16_t f32_to_f16_rn(float f) {     // round-to-nearest-even, saturating, subnormals supported
    uint32_t x;
    memcpy(&x, &f, 4);
    const uint16_t sign = (uint16_t)((x >> 16) & 0x8000u);
    x &= 0x7FFFFFFFu;
    if (x >= 0x47800000u) return sign | 0x7BFFu;                     // >= 65536 (or NaN): clamp to max finite
    if (x < 0x38800000u) {                                           // < 2^-14: fp16 subnormal, spacing 2^-24
        float af;
        memcpy(&af, &x, 4);
        const uint32_t m = (uint32_t)nearbyintf(af * 16777216.0f);   // <= 0x400 (== smallest normal when it rounds up)
        return sign | (uint16_t)m;
    }
    const uint32_t mant = x & 0x7FFFFFu;
    uint32_t h = (((x >> 23) - 112u) << 10) | (mant >> 13);
    const uint32_t rem = mant & 0x1FFFu;
    if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;
    if (h >= 0x7C00u) h = 0x7BFFu;
    return sign | (uint16_t)h;
}
inline float f16_to_f32(uint16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    const uint32_t e = (h >> 10) & 0x1Fu, m = h & 0x3FFu;
    float mag;
    if (e == 0) mag = (float)m * (1.0f / 16777216.0f);
    else {
        const uint32_t u = ((e + 112u) << 23) | (m << 13);
        memcpy(&mag, &u, 4);
    }
    uint32_t u;
    memcpy(&u, &mag, 4);
    u |= sign;
    float out;
    memcpy(&out, &u, 4);
    return out;
}

}  // namespace

size_t tc_weight_bytes(int N, int K) {
    const size_t kc = (K + BK - 1) / BK;
    return kc * 2 * (size_t)tc_npad(N) * 128;
}

// Image layout: [k chunk (64)][plane: hi, lo][row (npad)][128 bytes = 8 chunks of 8 halves], chunk c of row r stored
// at chunk position c ^ (r % 8) (SWIZZLE_128B); zero padded in N and K.  The matrix is multiplied by 2^e, e chosen so
// that max|w| * 2^e lies in [2^12, 2^13); returns 2^-e for the epilogue.
float tc_pack_weight(const float* w, int N, int K, void* dst_host) {
    const int npad = tc_npad(N);
    const int kc_n = (K + BK - 1) / BK;
    float amax = 0.f;
    for (size_t i = 0; i < (size_t)N * K; ++i) amax = fmaxf(amax, fabsf(w[i]));
    int e = 0;
    if (amax > 0.f && std::isfinite(amax)) {
        e = 12 - (int)floorf(log2f(amax));
        if (e > 24) e = 24;
        if (e < -24) e = -24;
    }
    const float scale = ldexpf(1.f, e);
    uint16_t* out = reinterpret_cast<uint16_t*>(dst_host);
    for (int kc = 0; kc < kc_n; ++kc)
        for (int r = 0; r < npad; ++r)
            for (int c = 0; c < 8; ++c)
                for (int el = 0; el < 8; ++el) {
                    const int k = kc * BK + c * 8 + el;
                    const float x = (r < N && k < K) ? w[(size_t)r * K + k] * scale : 0.f;
                    const uint16_t hi = f32_to_f16_rn(x);
                    const uint16_t lo = f32_to_f16_rn(x - f16_to_f32(hi));
                    const size_t pos = (size_t)r * 64 + (size_t)((c ^ (r & 7)) * 8) + el;      // in halves
                    out[((size_t)kc * 2 + 0) * npad * 64 + pos] = hi;
                    out[((size_t)kc * 2 + 1) * npad * 64 + pos] = lo;
                }
    return ldexpf(1.f, -e);
}

int launch_gemm_tc(const GemmParams& p, cudaStream_t s, GemmLaunchInfo* info) {
    struct InfoScope {          // launch_one fills *info through the thread-local pointer
        explicit InfoScope(GemmLaunchInfo* i) { g_launch_info = i; }
        ~InfoScope() { g_launch_info = nullptr; }
    } scope(info);
    COTR_CHECK(p.M > 0 && p.N > 0 && p.K > 0, "gemm_tc: empty problem %d x %d x %d", p.M, p.N, p.K);
    COTR_CHECK(p.Wtc != nullptr, "gemm_tc: weight has no tensor-core image");
    COTR_CHECK(p.out_f32 != nullptr || (p.N & 15) == 0, "gemm_tc: split16 outputs need N %% 16 == 0 (N=%d)", p.N);
    COTR_CHECK(p.res.hi == nullptr || ((p.ldr & 15) == 0 && (p.N & 15) == 0 && ((uintptr_t)p.res.hi & 31) == 0 && ((uintptr_t)p.res.lo & 31) == 0),
               "gemm_tc: residual needs ldr %% 16 == 0 and 32-byte aligned planes");
    COTR_CHECK(p.addmat == nullptr || ((p.ld_add & 3) == 0 && (p.N & 15) == 0), "gemm_tc: add-matrix needs ld %% 4 == 0");
    COTR_CHECK(p.out_f32 != nullptr || (p.ldc & 7) == 0, "gemm_tc: split16 output needs ldc %% 8 == 0");
    if (p.ln_gamma) {
        COTR_CHECK(p.N == 256 && p.relu == 0 && p.out_f32 == nullptr && !p.remap, "gemm_tc: LayerNorm epilogue needs N = 256");
        return launch_mode<256, true>(p, s);
    }
    if (p.N < 64) {
        COTR_CHECK(p.N <= 16, "gemm_tc: N between 17 and 63 is not instantiated");
        return launch_mode<16, false>(p, s);
    }
    // Tile width: at small batch most GEMMs of this network have a handful of 128-row tiles, so the widest tile
    // that still yields ~100 CTAs (148 SMs) wins; the narrow tiles trade tensor efficiency for parallelism and a
    // shorter per-CTA epilogue (the critical path of these latency-bound launches).  The tile width sets the number
    // of TMEM accumulators and so the summation order: it is chosen from the scheduling row count (M_sched).
    const long long mt = ((p.M_sched > 0 ? p.M_sched : p.M) + BM - 1) / BM;
    // bring-up knobs (cotr_debug_set_variant): bits 10-11 / 12-13 move the CTA-count thresholds of the 64 / 128 tiles
    static const long long kThr[4] = {96, 48, 64, 148};
    static const long long kThrWide[4] = {96, 48, 1 << 30, 148};
    const long long thr64 = kThr[(g_tc_variant >> 10) & 3], thr128 = kThrWide[(g_tc_variant >> 12) & 3];
    if ((p.N % 128) == 0 && mt * (p.N / 128) >= thr128) return launch_mode<128, false>(p, s);
    if (mt * ((p.N + 63) / 64) >= thr64 || p.a_mode == A_STEM_NHWC4 || (p.N % 32) != 0) return launch_mode<64, false>(p, s);
    return launch_mode<32, false>(p, s);
}

}  // namespace cotr
