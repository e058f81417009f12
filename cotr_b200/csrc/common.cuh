// Shared declarations of the cotr_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

namespace cotr {

void set_error(const char* fmt, ...);

#define COTR_CHECK_CUDA(expr)                                                                      \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ::cotr::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e_)); \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)

#define COTR_CHECK(cond, ...)                                                                      \
    do {                                                                                           \
        if (!(cond)) {                                                                             \
            ::cotr::set_error(__VA_ARGS__);                                                        \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel of the forward is launched with the programmatic-stream-serialization
// attribute: it may start (barrier init, TMEM allocation, weight prefetch by TMA) while its predecessor in the
// stream / graph is still draining, and calls pdl_wait() before it first touches memory the predecessor produces
// (or still reads).  At batch 1 the forward is ~135 latency-bound launches, so hiding launch + prologue matters.
// ---------------------------------------------------------------------------------------------------------------
extern int g_use_pdl;
extern long long* g_tc_timestamps;   // debug timeline buffer of the tcgen05 kernels (cotr_debug_set_timestamps), else null
extern int g_tc_variant;
extern int g_tc_trace_idx;
// Trace mode (cotr_debug_set_variant bit 17 + a timestamp buffer): every tcgen05 launch gets its own block of
// 256 CTAs x 64 slots, so one forward (graph replay included) leaves a per-launch record; slots 61-63 hold %globaltimer.
inline long long* next_trace_block() {
    if (!g_tc_timestamps) return nullptr;
    if (!(g_tc_variant & (1 << 17))) return g_tc_timestamps;
    return g_tc_timestamps + (size_t)(g_tc_trace_idx++) * 64 * 256;
}
#ifdef __CUDACC__
__device__ __forceinline__ long long global_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// ---------------------------------------------------------------------------------------------------------------
// Launch-to-launch dependencies through counters in global memory ("dataflow" mode of the forward chain).
// griddepcontrol.wait releases a dependent grid only when the WHOLE producer grid has retired and its memory is flushed
// (measured 0.7-1.3 us after the producer's last CTA, plus the start skew of the producer's CTAs).  In dataflow mode
// every CTA announces its finished stores on a counter block of its launch (block[0]: all CTAs, block[1 + t]: the CTAs
// that wrote rows of the 128-row tile t) with a gpu-scope release, and a consumer CTA waits - one polling thread, then
// an mbarrier / __syncthreads for the rest of the CTA - only for what it reads:
//   DEP_ALL    every CTA of the producer                                   block[0]      >= dep_target
//   DEP_TILE   the producer CTAs of this CTA's own 128-row tile            block[1 + t]  >= dep_target
//   DEP_SPAN   the producer CTAs of dep_span consecutive tiles starting at (t / dep_span) * dep_span (attention: keys
//              and values of the whole image pair)
// The launches keep the programmatic-stream-serialization attribute (a consumer becomes resident early) but do not
// execute griddepcontrol.wait.  No deadlock: a grid is only launched once every CTA of its producer is resident or done.
// Counters are zeroed by one memset at the head of the forward.  dep_mode == DEP_PDL keeps the hardware wait.
// ---------------------------------------------------------------------------------------------------------------
enum DepMode : int { DEP_PDL = 0, DEP_ALL = 1, DEP_TILE = 2, DEP_SPAN = 3 };
constexpr int kSyncBlockInts = 256;        // ints per launch: [0] total, [1 .. 255] per 128-row tile
struct LaunchSync {
    const int* dep;       // counter block of the producer launch
    int dep_mode;
    int dep_target;       // signals expected on each counter that is waited for
    int dep_span;         // DEP_SPAN: tiles per group
    int* sig;             // counter block of this launch (null: no announcement)
    int sig_tiles;        // per-tile counters in use (0: only the total)
};

#ifdef __CUDACC__
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// One thread: spin until *p >= target.  A counter that never arrives would hang the GPU, so the spin is bounded
// (~2 s) and traps: the failure is loud and the device survives.
__device__ __forceinline__ void dep_spin(const int* p, int target) {
    long long t0 = 0;
    unsigned spins = 0;
    while (ld_acquire_gpu(p) < target) {
        if ((++spins & 0xFFFu) == 0) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) __trap();
        }
    }
}
// tile = this CTA's 128-row tile in the producer's row space
__device__ __forceinline__ void dep_wait_thread(const LaunchSync& y, int tile) {
    if (y.dep_mode == DEP_ALL) {
        dep_spin(y.dep, y.dep_target);
    } else if (y.dep_mode == DEP_TILE) {
        dep_spin(y.dep + 1 + tile, y.dep_target);
    } else if (y.dep_mode == DEP_SPAN) {
        const int t0 = (tile / y.dep_span) * y.dep_span;
        for (int t = 0; t < y.dep_span; ++t) dep_spin(y.dep + 1 + t0 + t, y.dep_target);
    }
}
// One thread, after a CTA-wide barrier that follows the CTA's last global store.
__device__ __forceinline__ void dep_signal_thread(const LaunchSync& y, int tile) {
    if (y.sig == nullptr) return;
    __threadfence();
    atomicAdd(y.sig, 1);
    if (y.sig_tiles > 0 && tile < y.sig_tiles) atomicAdd(y.sig + 1 + tile, 1);
}
#endif

// Function attributes (opt-in dynamic shared memory) are per device, and one process may hold one handle per device:
// remember per kernel on which devices it has been configured.  (Racing first uses merely set the attribute twice.)
inline bool first_use_on_device(unsigned long long* configured_mask) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (*configured_mask & bit) return false;
    *configured_mask |= bit;
    return true;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Same, with a thread-block cluster of (1, 1, cluster_z) CTAs (grid.z must equal cluster_z).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                         int cluster_z, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (g_use_pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster_z > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = 1;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = (unsigned)cluster_z;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

constexpr int kDModel = 256;
constexpr int kHeads = 8;
constexpr int kHeadDim = 32;
constexpr int kTokens = 512;   // 16 x 32 context grid
constexpr int kFF = 1024;
constexpr int kEncLayers = 6;
constexpr int kDecLayers = 6;

// Attention operand images (tensor-core path).  The keys and values of one (pair, slot, head) - slot = decoder layer, or 0
// for the encoder's own layer - are stored in HBM exactly as the attention kernel wants them in shared memory, so that
// staging them is two bulk-TMA copies issued by one thread (cp.async.bulk -> UBLKCP) instead of 8 192 16-byte cp.async:
//   K image  [plane hi | lo][4 groups of 8 head dims][512 keys][16 B]           = 2 x 32 KB  (UMMA K-major canonical layout)
//   V image  [64 groups of 8 keys][hi: 32 head dims x 16 B | lo: 32 x 16 B | 16 B pad]  = 64 x 1040 B
// written in that form by the epilogue of the projection GEMM (split16.cuh::store16).
constexpr size_t kAttnKPlaneBytes = 4 * 512 * 16;                         // 32 KB
constexpr size_t kAttnKImgBytes = 2 * kAttnKPlaneBytes;                   // 64 KB
constexpr size_t kAttnVGroupBytes = 2 * 32 * 16 + 16;                     // 1040 B
constexpr size_t kAttnVImgBytes = 64 * kAttnVGroupBytes;                  // 66 560 B
constexpr size_t kAttnHeadImgBytes = kAttnKImgBytes + kAttnVImgBytes;     // 132 096 B per (pair, slot, head)

// ---------------------------------------------------------------------------------------------------------------
// "split16" activations.  Every activation between kernels is stored as TWO fp16 planes, x ~= hi + lo (22 mantissa
// bits, same bytes as fp32): the tensor-core kernels need their operands in exactly that form (gemm_tc.cu), so the
// producer's epilogue splits once and every consumer stages its operand with plain asynchronous 16-byte copies.
// hi + lo is exactly representable in fp32, so reconstruct -> split round-trips are lossless.
// ---------------------------------------------------------------------------------------------------------------
struct Split16 {          // plain aggregates: they travel inside kernel parameter structs
    __half* hi;
    __half* lo;
};
struct CSplit16 {
    const __half* hi;
    const __half* lo;
};
inline CSplit16 cs(const Split16& s) { return CSplit16{s.hi, s.lo}; }
inline Split16 offset(const Split16& s, size_t elems) { return Split16{s.hi + elems, s.lo + elems}; }
inline CSplit16 offset(const CSplit16& s, size_t elems) { return CSplit16{s.hi + elems, s.lo + elems}; }

// The stem's input.  The network input is an fp32 (B,3,256,512) NCHW canvas, two 256x256 images side by side.  The 7x7
// stride-2 convolution reads it through a split16 copy made by one small kernel per forward (launch_stem_canvas): image
// n = 2*pair + half as [kStemCanvasRows][kStemCanvasPitch] pixels of 4 halves (r, g, b, 0), the image at rows / columns
// 3.., everything else zero (the convolution's padding, written once when the buffer is allocated).  A filter row of
// output pixel (oh, ow) is then 8 consecutive pixels = 64 contiguous, 16-byte aligned bytes per plane starting at pixel
// (2 oh + kh, 2 ow): no bounds checks, plain 16-byte cp.async like every other operand.  K = 7 rows x 8 pixel slots x 4
// channels = 224, the weights carry zeros for slot 7 and channel 3.
constexpr int kStemCanvasRows = 262, kStemCanvasPitch = 264;
constexpr size_t kStemCanvasElems = (size_t)kStemCanvasRows * kStemCanvasPitch * 4;      // halves per image and plane
constexpr int kStemK = 7 * 32;

// How a GEMM finds row m, column k of its A operand.
enum AMode : int {
    A_ROWMAJOR = 0,   // A[m * lda + k]
    A_CONV_NHWC = 1,  // implicit im2col over an NHWC activation: m -> (n, oh, ow), k -> (kh, kw, c)
    A_STEM_NHWC4 = 2, // 7x7 stride-2 stem: implicit im2col over the zero-bordered split16 NHWC4 copy of the canvas (below)
    A_TOKENS = 3,     // m = pair*512 + i*32 + j gathers row ((2*pair + (j>>4))*16 + i)*16 + (j&15)
};

// D[M,N] = epilogue( A[M,K] * W[N,K]^T ).
struct GemmParams {
    int M, N, K;
    // A operand: split16 activation (A_STEM_NHWC4: the stem canvas)
    CSplit16 a;
    int a_mode;
    int lda;
    int H, W, C;      // convolution geometry: input height / width / channels (per image)
    int OH, OW;       // output height / width
    int KH, KW, stride, pad;
    // weights: fp32 row-major [N, K] (K ordered (kh, kw, c) for convolutions) for the SIMT path; for the tensor-core
    // path the same matrix pre-scaled by a power of two, pre-split into fp16 hi/lo and pre-tiled (gemm_tc.cu).
    const float* Wt;
    const void* Wtc;
    float acc_scale;  // undoes the power of two on the accumulator
    // epilogue: v = acc * acc_scale + bias[n] + addmat[(m % add_period) * ld_add + n] + residual[m * ldr + n]; relu; LN
    const float* bias;
    const float* addmat;
    int add_period, ld_add;
    CSplit16 res;
    int ldr;
    int relu;
    const float* ln_gamma;   // optional LayerNorm over the N = 256 columns of each row (after the residual)
    const float* ln_beta;
    // Deferred LayerNorm (tcgen05 path, row-major A).  A LayerNorm output is never stored: the GEMM that produces the
    // PRE-norm rows x (N = 256) also leaves, per row and 16-column chunk, the chunk's (mean, M2) in `ln_part_out`
    // [M][16] float2 (from the fp32 values in its epilogue registers); every consumer merges the 16 pairs into the row's
    // (mean, rstd) in its own epilogue prologue and applies the norm on the fly:
    //   * as the A operand (K = 256): the weights carry gamma (W' = W diag(gamma), packed at model creation) and
    //         y[n] = rstd * (acc[n] - mean * a_ln_cs[n]) + bias[n],   a_ln_cs[n] = sum_k W'[n,k],  bias = beta W^T + b;
    //   * as the residual operand: res[n] = (r[n] - mean) rstd res_ln_gamma[n] + res_ln_beta[n].
    const float* a_ln_cs;          // [N]; null = A is used as it is stored
    const float2* a_ln_part;       // [M][16] partial statistics of the A rows
    const float2* res_ln_part;     // [M][16] partial statistics of the residual rows; null = plain residual
    const float* res_ln_gamma;
    const float* res_ln_beta;
    float2* ln_part_out;           // [M][16]; null = no statistics wanted
    LaunchSync sync;         // dataflow dependencies (all zero: hardware griddepcontrol.wait)
    // outputs
    float* out_f32;          // when non-null: plain fp32 row-major output (the final prediction, N = 2)
    Split16 out;             // otherwise split16, row-major with leading dimension ldc ...
    int ldc;
    // ... except that 256-column blocks of N can be redirected (K/V projections): blk_map[b] >= 0 -> the block is
    // stored at column offset blk_map[b] of `out`; blk_map[b] = -(v+1) -> the block is a value projection and is
    // stored TRANSPOSED as vt[((pair * n_vt + v) * 256 + c) * 512 + key] (row = pair*512 + key), the K-major B operand
    // the attention kernels need.
    // With kv_img set (tensor-core path) the key / value blocks go into the attention operand images instead:
    // blk_map[b] = -(v+1) -> value block of slot v, blk_map[b] = -1000 - s -> key block of slot s; the image of
    // (pair, slot, head) starts at kv_img + ((pair * n_vt + slot) * 8 + head) * kAttnHeadImgBytes.
    int remap;
    int blk_map[12];
    Split16 vt;
    int n_vt;
    unsigned char* kv_img;
    // Scheduling row count (host side only, never read by a kernel): tile width and split-K are chosen as if the launch
    // had M_sched rows; 0 = M.  The batch-invariant mode sets it to the row count of the same call site at the
    // headline shape, so a row's summation order does not depend on how many other rows share the launch.
    int M_sched;
};

// softmax(q k^T) v per head; q already carries the head_dim^-0.5 scale.
struct AttnParams {
    CSplit16 q; int ldq;         // rows: local row r = pair_local * nq + i
    CSplit16 k; int ldk;         // rows: (pair0 + pair_local) * 512 + key
    CSplit16 vt;                 // [(pair0 + pair_local) * vt_pair_stride + (head*32 + d) * 512 + key]
    size_t vt_pair_stride;
    // tensor-core path: keys and values as operand images (see kAttnHeadImgBytes); k / vt above are then unused.
    // image of (pair0 + pair_local, head) = kv_img + (pair0 + pair_local) * img_pair_stride + head * kAttnHeadImgBytes
    const unsigned char* kv_img;
    size_t img_pair_stride;
    Split16 out; int ldo;
    int nq;                      // query rows per pair in this launch
    int npairs;
    int pair0;
    LaunchSync sync;             // dataflow dependencies (all zero: hardware griddepcontrol.wait)
    // Scheduling query count (host side only): launch_attention_tc hands launches with nq_sched < 32 to the SIMT kernel;
    // 0 = nq.  The batch-invariant mode sets it to the headline's count, so every nq >= 1 runs on the tensor cores.
    int nq_sched;
};

int launch_gemm_simt(const GemmParams& p, cudaStream_t s);
int launch_gemm_simt_raw(const GemmParams& p, float* raw_out_f32, cudaStream_t s);   // result as plain fp32 [M,N]
int launch_layernorm_f32(const float* x, const float* gamma, const float* beta, Split16 out, int rows, cudaStream_t s);
struct GemmLaunchInfo { int row_tiles, col_tiles, ksplit; };      // the grid launch_gemm_tc chose (dataflow bookkeeping)
int launch_gemm_tc(const GemmParams& p, cudaStream_t s, GemmLaunchInfo* info = nullptr);
int launch_attention_simt(const AttnParams& p, cudaStream_t s);
int launch_attention_tc(const AttnParams& p, cudaStream_t s);
int launch_maxpool_3x3s2_nhwc(CSplit16 in, Split16 out, int N, int H, int W, int C, cudaStream_t s, LaunchSync sync = LaunchSync{});
int launch_layernorm(CSplit16 x, const float* gamma, const float* beta, Split16 out, int rows, cudaStream_t s);
// out = LN2(LN1(x)): the last decoder layer's norm3 followed by decoder.norm (transformer.py:110-111) in one pass
// part[row][c] = (mean, M2) of channels [16c, 16c+16) of a [rows][256] tensor (what GemmParams::ln_part_out holds)
int launch_ln_partials(CSplit16 x, float2* part, int rows, cudaStream_t s);
int launch_layernorm_twice(CSplit16 x, const float* g1, const float* b1, const float* g2, const float* b2, Split16 out, int rows, cudaStream_t s,
                           LaunchSync sync = LaunchSync{});
int launch_query_encode(const float* queries, Split16 qpos, int rows, cudaStream_t s, LaunchSync sync = LaunchSync{});
// fp32 (B,3,256,512) canvas -> the stem's bordered split16 NHWC4 operand (2B images of kStemCanvasElems halves per plane)
int launch_stem_canvas(const float* img, Split16 canvas, int n_img, cudaStream_t s, LaunchSync sync = LaunchSync{});
int launch_f32_to_split16(const float* in, Split16 out, size_t n, cudaStream_t s);
int launch_split16_to_f32(CSplit16 in, float* out, size_t n, cudaStream_t s);

// Device-side post-processing of the dense pass (dense_post.cu)
int dense_post_launch(const float* pred, float* out, int n, cudaStream_t s);

// Barycentric triangle rasteriser of triangulate_corr (engine_ops.cu)
int rasterize_triangles_launch(const float* tris, int n_tri, int H, int W, float* out, cudaStream_t s);

// Squad formation of the grouped scheduler (engine_ops.cu)
int group_tasks_launch(const double* pts, const double* box, int n, int batch_size, int max_load, int* squad, int* rank, int* n_squads, cudaStream_t s);

// Dense first guess: affine + Pillow-exact float resize + confidence merge of one tile (engine_ops.cu)
struct FlowMerger;
FlowMerger* flow_merger_create();
void flow_merger_destroy(FlowMerger* f);
int flow_tile_merge_launch(FlowMerger* f, const float* tile, int pitch, const double* affine, int px, int py, int pw, int ph, int ow, int oh,
                           float* flow, float* conf, int first, cudaStream_t s);

// Device-side crop + Pillow-exact resize + normalise (preprocess.cu)
struct Preprocessor;
Preprocessor* preprocessor_create();
void preprocessor_destroy(Preprocessor* p);
int preprocess_launch(Preprocessor* p, const unsigned char* img_from, int hf, int wf, const unsigned char* img_to, int ht, int wt,
                      const int* rects_host, int n, float* canvas_dev, cudaStream_t s);

// Bytes of the pre-tiled fp16 hi/lo image of an [N,K] weight matrix, and the host-side packer (returns acc_scale).
size_t tc_weight_bytes(int N, int K);
float tc_pack_weight(const float* w, int N, int K, void* dst_host);

}  // namespace cotr
