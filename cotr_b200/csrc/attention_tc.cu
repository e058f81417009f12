// tcgen05 attention over the 512-token context (encoder self-attention and decoder cross-attention), split16 I/O.
//
// One CTA per (128-query tile, head, image pair).  The whole score tile S = Q K^T (128 x 512 fp32) fits TMEM exactly
// (512 columns), so the softmax is exact (no online rescaling):
//   warps 0-7  stage Q, K and V^T of this head with asynchronous 16-byte copies (cp.async -> LDGSTS, completion on an
//              mbarrier): the operands already live in HBM as fp16 hi/lo planes and V is stored transposed by the
//              projection GEMM's epilogue, so staging is pure data movement into the UMMA canonical layout.  They then
//              run the softmax straight out of TMEM.  A query row is shared by two threads (warps w and w + 4 read
//              the same TMEM lane quarter): each takes 32 of the 64 keys of every chunk, the row max and the row sum
//              are combined through shared memory on a 64-thread named barrier.  P (split to fp16 hi/lo) goes to the
//              MMA in 64-key chunks, double buffered;
//   warp 8     (one lane) issues the tcgen05 MMAs: 2 x (128x256x32) for S, then O = P V per 64-key chunk.  The hi and
//              lo planes of V^T sit next to each other in shared memory, so ONE MMA of N = 64 forms
//              P_hi * [V_hi; V_lo] (main | correction columns) and a second one of N = 32 adds P_lo * V_hi - an
//              M = 128 MMA this narrow costs the same ~60-80 cycles whatever its N.  The O accumulators re-use TMEM
//              columns of S chunks that have already been turned into P; because the tensor core's fp32 accumulate
//              truncates (profiles/r01_tc_precision.md) even / odd chunks accumulate into different column sets
//              ([0,64) and [64,128): main | correction), summed with RN adds at the end.
// q is expected pre-scaled by head_dim^-0.5 (folded into the projection weights).
#include "split16.cuh"
#include "tc_common.cuh"

namespace cotr {

namespace {

using namespace tc;

constexpr int kTile = 128;
constexpr int kSoftmaxThreads = 256;                     // warps 0-7
constexpr int kThreads = kSoftmaxThreads + 32;            // + the MMA warp
constexpr int kChunk = 64;                                // keys per P chunk
constexpr int kChunks = kTokens / kChunk;                 // 8
constexpr uint32_t kQLbo = kTile * 16;                    // Q tile  [4 K-groups][128 rows][16 B]
constexpr uint32_t kQPlane = 4 * kQLbo;                   // 8 KB
constexpr uint32_t kKLbo = kTokens * 16;                  // K tile  [4 K-groups][512 keys][16 B]
constexpr uint32_t kKPlane = 4 * kKLbo;                   // 32 KB
constexpr uint32_t kVLbo = 2 * kHeadDim * 16 + 16;        // V^T tile [64 key-groups][hi: 32 d | lo: 32 d][16 B], padded against bank conflicts
constexpr uint32_t kVBytes = (kTokens / 8) * kVLbo;       // 65 KB
constexpr uint32_t kVLoOff = kHeadDim * 16;               // the lo rows of a key group follow its hi rows
constexpr uint32_t kPLbo = kTile * 16;                    // P chunk [8 key-groups][128 rows][16 B]
constexpr uint32_t kPPlane = (kChunk / 8) * kPLbo;        // 16 KB
constexpr uint32_t kSbo = 128;

constexpr uint32_t kOffQ = 0;
constexpr uint32_t kOffK = kOffQ + 2 * kQPlane;
constexpr uint32_t kOffV = kOffK + 2 * kKPlane;
constexpr uint32_t kOffP = kOffV + kVBytes;               // 2 buffers x (hi, lo)
constexpr uint32_t kOffStat = kOffP + 4 * kPPlane;         // row max / row sum exchange: [2 halves][128 rows] floats
constexpr uint32_t kOffBar = kOffStat + 2 * kTile * 4;
constexpr uint32_t kSmemBytes = kOffBar + 128;
static_assert(kSmemBytes <= 227 * 1024, "attention tile does not fit shared memory");
// the operand images of common.cuh are byte-for-byte these shared-memory tiles
static_assert(2 * kKPlane == kAttnKImgBytes && kKPlane == kAttnKPlaneBytes && kVLbo == kAttnVGroupBytes && kVBytes == kAttnVImgBytes &&
              kOffV == kOffK + kAttnKImgBytes, "attention operand images and shared-memory tiles went out of step");

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// kSkipIdle (launches with nq < 32 only): softmax warps whose 32-row TMEM lane quarter holds no valid query row skip the
// TMEM reads, the exponentials and the P stores; they still wait on and arrive at every barrier like the others, so the
// arrival counts are unchanged.  The MMA then multiplies stale P rows of those lanes, whose output rows are never read.
// The rows of the other quarters run exactly the instructions of the default instantiation.  A separate instantiation
// because a flag-guarded path that never executes still slows a tcgen05 kernel down (DESIGN.md section 8).
template <bool kSkipIdle>
__global__ void __launch_bounds__(kThreads, 1) attention_tc_kernel(const AttnParams p, long long* __restrict__ ts) {
    // debug timeline (ts != null, cotr_debug_set_timestamps): 64 clock64() stamps per CTA, slots in tools/bringup.py
    long long* my_ts = ts ? ts + (size_t)((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 64 : nullptr;
    const long long t_start = ts ? clock64() : 0;
#define COTR_TS(slot) do { if (my_ts) my_ts[(slot)] = clock64() - t_start; } while (0)
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
    uint64_t* qk_full = bars + 0;
    uint64_t* v_full = bars + 1;
    uint64_t* s_full = bars + 2;
    uint64_t* o_full = bars + 3;
    uint64_t* p_full = bars + 4;     // [2]
    uint64_t* p_empty = bars + 6;    // [2]
    uint64_t* dep_ready = bars + 8;  // dataflow mode (common.cuh LaunchSync): the polling thread has seen the producer's counters
    uint64_t* k_img_full = bars + 9; // operand images: the bulk copy of K (hi + lo planes) has landed
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 10);
    const bool img = p.kv_img != nullptr;       // keys / values arrive as operand images by bulk TMA (tensor-core schedule)
    const bool dflow = p.sync.dep_mode != DEP_PDL;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int head = blockIdx.y;
    const int pair_local = blockIdx.z;
    const int row0 = blockIdx.x * kTile;
    const int sync_tile = (pair_local * p.nq + row0) / kTile;      // this CTA's 128-row tile of the launch's row space (nq % 128 == 0 in tile modes)

    if (threadIdx.x == 0) {
        mbar_init(qk_full, kSoftmaxThreads);
        mbar_init(v_full, img ? 1 : kSoftmaxThreads);
        mbar_init(s_full, 1);
        mbar_init(o_full, 1);
        mbar_init(&p_full[0], kSoftmaxThreads);
        mbar_init(&p_full[1], kSoftmaxThreads);
        mbar_init(&p_empty[0], 1);
        mbar_init(&p_empty[1], 1);
        mbar_init(dep_ready, 1);
        mbar_init(k_img_full, 1);
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(tmem_ptr, 512);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t sbase = smem_u32(smem);
    if (threadIdx.x == 0) COTR_TS(1);

    if (warp < 8) {
        const int t = threadIdx.x;
        const int quarter = warp & 3;                    // TMEM lane quarter
        const int half = warp >> 2;                      // which 32 keys of every 64-key chunk / which 16 output columns
        const int trow_i = quarter * 32 + lane;          // query row inside the tile == TMEM lane
        const int qi = row0 + trow_i;
        const bool row_ok = qi < p.nq;
        const bool idle = kSkipIdle && row0 + quarter * 32 >= p.nq;      // warp-uniform: no valid row in this lane quarter
        const size_t grow = (size_t)pair_local * p.nq + (row_ok ? qi : 0);
        const size_t kv_row0 = (size_t)(p.pair0 + pair_local) * kTokens;
        if (t == 0) {
            pdl_launch_dependents();                     // the next kernel may start its prologue on idle SMs
            if (dflow) { dep_wait_thread(p.sync, sync_tile); mbar_arrive(dep_ready); }
        }
        if (dflow) mbar_wait(dep_ready, 0); else pdl_wait();      // prologue above overlaps the previous kernel
        if (t == 0) COTR_TS(2);

        if (img && t == 0) {
            // keys and values of this (pair, head): two bulk-TMA copies (UBLKCP) of the operand images straight into the
            // tiles, issued by one thread before anything else; the 256 threads then only stage the 16 KB of Q
            const unsigned char* src = p.kv_img + (size_t)(p.pair0 + pair_local) * p.img_pair_stride + (size_t)head * kAttnHeadImgBytes;
            mbar_arrive_expect_tx(k_img_full, (uint32_t)kAttnKImgBytes);
            tma_bulk_g2s(smem + kOffK, src, (uint32_t)kAttnKImgBytes, k_img_full);
            mbar_arrive_expect_tx(v_full, (uint32_t)kAttnVImgBytes);
            tma_bulk_g2s(smem + kOffV, src + kAttnKImgBytes, (uint32_t)kAttnVImgBytes, v_full);
        }
        // ---- stage Q (row t % 128, two of the four 16-byte K groups per thread) and K (4 keys per thread) --------
        {
            const int r = t & 127, kg0 = (t >> 7) * 2;
            const int qr = row0 + r;
            const bool ok = qr < p.nq;
            const size_t qoff = ((size_t)pair_local * p.nq + (ok ? qr : 0)) * p.ldq + head * kHeadDim;
            const uint32_t bytes = ok ? 16u : 0u;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int kg = kg0 + j;
                const uint32_t dst = sbase + kOffQ + kg * kQLbo + r * 16;
                cp_async16(dst, p.q.hi + qoff + kg * 8, bytes);
                cp_async16(dst + kQPlane, p.q.lo + qoff + kg * 8, bytes);
            }
            if (!img) {
#pragma unroll
            for (int i = 0; i < kTokens / 128; ++i) {
                const int key = r + 128 * i;
                const size_t koff = (kv_row0 + key) * p.ldk + head * kHeadDim;
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int kg = kg0 + j;
                    const uint32_t dst = sbase + kOffK + kg * kKLbo + key * 16;
                    cp_async16(dst, p.k.hi + koff + kg * 8, 16u);
                    cp_async16(dst + kKPlane, p.k.lo + koff + kg * 8, 16u);
                }
            }
            }
        }
        cp_async_mbar_arrive_noinc(qk_full);

        // ---- stage V^T (already transposed in HBM): piece (key-group kg8, d) = 8 consecutive keys of row d ----
        if (!img) {
            const size_t vbase = (size_t)(p.pair0 + pair_local) * p.vt_pair_stride + (size_t)head * kHeadDim * kTokens;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int u = t + kSoftmaxThreads * i;
                const int kg8 = u & 63, d = u >> 6;
                const uint32_t dst = sbase + kOffV + kg8 * kVLbo + d * 16;
                const size_t voff = vbase + (size_t)d * kTokens + kg8 * 8;
                cp_async16(dst, p.vt.hi + voff, 16u);
                cp_async16(dst + kVLoOff, p.vt.lo + voff, 16u);
            }
            cp_async_mbar_arrive_noinc(v_full);
        }
        if (t == 0) COTR_TS(3);

        // ---- softmax out of TMEM ---------------------------------------------------------------------------
        float* stat = reinterpret_cast<float*>(smem + kOffStat);         // [half][row]
        mbar_wait(s_full, 0);
        tcgen05_fence_after();
        if (t == 0) COTR_TS(4);
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 32);
        float mx = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < (idle ? 0 : kTokens); c += 128) {
            uint32_t r[4][16];
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 4; ++h) tmem_ld16_issue(trow + c + (h >> 1) * 64 + (h & 1) * 16, r[h]);
#pragma unroll
            for (int h = 0; h < 4; ++h) tmem_ld16_fence(r[h]);
#pragma unroll
            for (int h = 0; h < 4; ++h)
#pragma unroll
                for (int j = 0; j < 16; ++j) mx = fmaxf(mx, __uint_as_float(r[h][j]));
        }
        if (!idle) {                                     // (both warps of a quarter skip together: the barrier is theirs alone)
            stat[half * kTile + trow_i] = mx;
            named_barrier_sync(1 + quarter, 64);
            mx = fmaxf(mx, stat[(half ^ 1) * kTile + trow_i]);
            named_barrier_sync(1 + quarter, 64);         // both have read: the slots are free for the row sums
        }
        if (t == 0) COTR_TS(5);
        const float kLog2e = 1.4426950408889634f;
        const float mxs = mx * kLog2e;
        float sum = 0.f;
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c) {
            const int buf = c & 1;
            if (idle) {                                  // keep the barrier protocol, skip the work
                if (c >= 2) mbar_wait(&p_empty[buf], (uint32_t)((c >> 1) - 1) & 1u);
                mbar_arrive(&p_full[buf]);
                continue;
            }
            uint32_t r[2][16];
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 2; ++h) tmem_ld16_issue(trow + c * kChunk + h * 16, r[h]);
#pragma unroll
            for (int h = 0; h < 2; ++h) tmem_ld16_fence(r[h]);
            if (c >= 2) mbar_wait(&p_empty[buf], (uint32_t)((c >> 1) - 1) & 1u);
            uint8_t* p_hi = smem + kOffP + buf * 2 * kPPlane + (half * 4) * kPLbo + trow_i * 16;
            uint8_t* p_lo = p_hi + kPPlane;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float v[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    v[j] = fast_exp2(fmaf(__uint_as_float(r[h][j]), kLog2e, -mxs));
                    sum += v[j];
                }
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    uint4 hi, lo;
                    split_f16x2(v[g * 8 + 0], v[g * 8 + 1], hi.x, lo.x);
                    split_f16x2(v[g * 8 + 2], v[g * 8 + 3], hi.y, lo.y);
                    split_f16x2(v[g * 8 + 4], v[g * 8 + 5], hi.z, lo.z);
                    split_f16x2(v[g * 8 + 6], v[g * 8 + 7], hi.w, lo.w);
                    *reinterpret_cast<uint4*>(p_hi + (h * 2 + g) * kPLbo) = hi;
                    *reinterpret_cast<uint4*>(p_lo + (h * 2 + g) * kPLbo) = lo;
                }
            }
            tcgen05_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(&p_full[buf]);
            if (t == 0) COTR_TS(6 + c);
        }
        if (!idle) {
            stat[half * kTile + trow_i] = sum;
            named_barrier_sync(1 + quarter, 64);
            sum += stat[(half ^ 1) * kTile + trow_i];
        }

        // ---- O / sum -> global (split16): this thread's 16 of the 32 head-dim columns ------------------------
        mbar_wait(o_full, 0);
        tcgen05_fence_after();
        if (t == 0) COTR_TS(14);
        if (!idle) {
            const float inv = 1.f / sum;
            const size_t ooff = grow * p.ldo + head * kHeadDim + half * 16;
            const uint32_t orow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 16);
            uint32_t r0[16], r1[16], r2[16], r3[16];
            __syncwarp();
            tmem_ld16_issue(orow, r0);            // main, even chunks
            tmem_ld16_issue(orow + 64, r1);       // main, odd chunks
            tmem_ld16_issue(orow + 32, r2);       // corrections
            tmem_ld16_issue(orow + 96, r3);
            tmem_ld16_fence(r0);
            tmem_ld16_fence(r1);
            tmem_ld16_fence(r2);
            tmem_ld16_fence(r3);
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)
                v[j] = ((__uint_as_float(r2[j]) + __uint_as_float(r3[j])) + (__uint_as_float(r0[j]) + __uint_as_float(r1[j]))) * inv;
            if (row_ok) {
                store8_split(p.out, ooff, v);
                store8_split(p.out, ooff + 8, v + 8);
            }
        }
        if (t == 0) COTR_TS(15);
    } else {
        // ================= MMA issuer =========================================================================
        if (lane == 0) {
            constexpr uint32_t idesc_s = make_idesc_f16_f32(128, 256);
            constexpr uint32_t idesc_o = make_idesc_f16_f32(128, kHeadDim);
            constexpr uint32_t idesc_o2 = make_idesc_f16_f32(128, 2 * kHeadDim);
            const uint32_t hi_word = desc_hi(kSbo);
            mbar_wait(qk_full, 0);
            if (img) mbar_wait(k_img_full, 0);
            tcgen05_fence_after();
            COTR_TS(20);
#pragma unroll
            for (int nh = 0; nh < 2; ++nh) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint32_t qa = sbase + kOffQ + ks * 2 * kQLbo;
                    const uint32_t ka = sbase + kOffK + nh * 256 * 16 + ks * 2 * kKLbo;
                    const uint64_t qh = make_desc(desc_lo(qa, kQLbo), hi_word), ql = make_desc(desc_lo(qa + kQPlane, kQLbo), hi_word);
                    const uint64_t kh = make_desc(desc_lo(ka, kKLbo), hi_word), kl = make_desc(desc_lo(ka + kKPlane, kKLbo), hi_word);
                    const uint32_t d = tmem_base + nh * 256;
                    umma_f16_ss(d, ql, kh, idesc_s, ks != 0);
                    umma_f16_ss(d, qh, kl, idesc_s, true);
                    umma_f16_ss(d, qh, kh, idesc_s, true);
                }
            }
            umma_commit(s_full);
            COTR_TS(21);
            mbar_wait(v_full, 0);
            COTR_TS(22);
#pragma unroll 1
            for (int c = 0; c < kChunks; ++c) {
                const int buf = c & 1;
                mbar_wait(&p_full[buf], (uint32_t)(c >> 1) & 1u);
                tcgen05_fence_after();
                COTR_TS(24 + 2 * c);
                // chunk c may only touch TMEM columns of S chunks <= c (already consumed by the softmax warps):
                // even chunks accumulate [main | P_hi V_lo] into [0,64), odd chunks into [64,128); P_lo V_hi goes to
                // the correction columns of the OTHER set (no other writer during this chunk), except in chunk 0
                // where columns >= 64 still hold scores
                const uint32_t o_set = tmem_base + ((c & 1) ? 64u : 0u);
                const uint32_t o_lo = tmem_base + ((c == 0 || (c & 1)) ? 32u : 96u);
#pragma unroll
                for (int ks = 0; ks < kChunk / 16; ++ks) {
                    const uint32_t pa = sbase + kOffP + buf * 2 * kPPlane + ks * 2 * kPLbo;
                    const uint32_t va = sbase + kOffV + (c * (kChunk / 8) + ks * 2) * kVLbo;
                    const uint64_t ph = make_desc(desc_lo(pa, kPLbo), hi_word), pl = make_desc(desc_lo(pa + kPPlane, kPLbo), hi_word);
                    const uint64_t vv = make_desc(desc_lo(va, kVLbo), hi_word);       // N = 64: hi rows then lo rows; N = 32: hi only
                    umma_f16_ss(o_set, ph, vv, idesc_o2, (c >= 2) || ks != 0);
                    umma_f16_ss(o_lo, pl, vv, idesc_o, true);
                }
                umma_commit(&p_empty[buf]);
                COTR_TS(25 + 2 * c);
            }
            umma_commit(o_full);
        }
        __syncwarp();
    }

    tcgen05_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) dep_signal_thread(p.sync, sync_tile);
    if (warp == 8) tmem_dealloc(tmem_base, 512);
    if (threadIdx.x == 0) COTR_TS(60);
    if (my_ts && threadIdx.x == 0) my_ts[62] = global_ns();
#undef COTR_TS
}

}  // namespace

int launch_attention_tc(const AttnParams& p, cudaStream_t s) {
    if (p.nq <= 0 || p.npairs <= 0) return 0;
    // a 128-row MMA tile would be > 75% padding: by default such launches run on the SIMT kernel; a scheduling count
    // of 32 or more (batch-invariant mode, the path-2 test hook) keeps them on the tensor cores
    if ((p.nq_sched > 0 ? p.nq_sched : p.nq) < 32) return launch_attention_simt(p, s);
    const bool skip_idle = p.nq < 32;
    static unsigned long long configured = 0;      // bit per device
    if (first_use_on_device(&configured)) {
        COTR_CHECK_CUDA(cudaFuncSetAttribute(attention_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
        COTR_CHECK_CUDA(cudaFuncSetAttribute(attention_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    }
    COTR_CHECK(p.npairs <= 65535, "attention: too many pairs in one launch (%d)", p.npairs);
    COTR_CHECK((p.ldq & 7) == 0 && (p.ldk & 7) == 0 && (p.ldo & 7) == 0 && (p.vt_pair_stride & 7) == 0,
               "attention_tc: leading dimensions must be multiples of 8 elements");
    dim3 grid((p.nq + kTile - 1) / kTile, kHeads, p.npairs);
    COTR_CHECK_CUDA(launch_kernel(skip_idle ? attention_tc_kernel<true> : attention_tc_kernel<false>, grid, dim3(kThreads), kSmemBytes, s, p,
                                  next_trace_block()));
    return 0;
}

}  // namespace cotr
