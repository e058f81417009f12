// Model state, weight packing, workspace and the forward schedule behind the C ABI (include/cotr_b200.h).
//
// Reference lines restated by each stage are cited inline (paths relative to the reference root).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "../../include/cotr_b200.h"
#include "common.cuh"

namespace cotr {

extern int g_tc_variant;
extern long long* g_tc_timestamps;
static thread_local char g_error[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

namespace {

constexpr int kDecodeChunkRows = 32768;   // decoder rows processed per pass (rows are independent, so chunking is exact)
constexpr int kKCols = kDecLayers * kDModel;         // 1536: K of all decoder layers, [layer][256]
constexpr int kQpCols = kDecLayers * kDModel;        // 1536
constexpr size_t kVtLayer = (size_t)kDModel * kTokens;   // one transposed value projection [256][512]

struct DevConv {
    float* w = nullptr;    // [cout][kh][kw][cin], FrozenBN scale folded in
    void* wtc = nullptr;   // tensor-core image of w
    float wtc_scale = 1.f; // accumulator scale that undoes the image's power-of-two pre-scaling
    float* b = nullptr;    // FrozenBN shift
    int cout = 0, cin = 0, kh = 1, kw = 1, stride = 1, pad = 0;
    bool stem = false;     // 7x7/2 stem over the bordered NHWC4 canvas: kw = 8 pixel slots, cin = 4 (common.cuh)
};

struct DevLinear {
    float* w = nullptr;    // [N][K]
    void* wtc = nullptr;
    float wtc_scale = 1.f;
    float* b = nullptr;    // [N] or null
    int n = 0, k = 0;
    // Deferred LayerNorm on the input (tensor-core path, GemmParams::a_ln_cs): wtc then holds W diag(gamma),
    // cs its column sums and b_tc = beta W^T + b; w / b stay the checkpoint's values for the fp32 SIMT path.
    float* cs = nullptr;
    float* b_tc = nullptr;
    void* wtc_plain = nullptr;       // tensor-core image of the un-folded W (explicit-LayerNorm schedule on the tensor-core path)
    float wtc_plain_scale = 1.f;
};

struct Block {
    DevConv c1, c2, c3, ds;
    bool has_ds = false;
};

struct EncLayer {
    DevLinear qkv;         // [768][256]; q rows pre-scaled by head_dim^-0.5; bias folded into add_qkv
    float* add_qkv = nullptr;   // [512][768] = [ (pos Wq^T + bq) s | pos Wk^T + bk | bv ]
    float* add_qkv_tc = nullptr;   // + beta W^T of the previous layer's norm2 (deferred LayerNorm, layers > 0)
    DevLinear o, l1, l2;
    float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
};
static_assert(sizeof(float2) == 8, "row statistics are (mean, rstd) pairs");

struct DecLayer {
    DevLinear q;           // [256][256] pre-scaled, no bias (bias lives in the qpos projection)
    DevLinear o, l1, l2;
    float *ln2_g, *ln2_b, *ln3_g, *ln3_b;
};

const Split16 kNoSplit = {nullptr, nullptr};

struct Workspace {
    int cap_pairs = 0;
    int cap_rows = 0;
    // backbone (per image sizes x 2*cap_pairs), all split16
    Split16 canvas = kNoSplit, stem = kNoSplit, bx = kNoSplit, by = kNoSplit, bt1 = kNoSplit, bt2 = kNoSplit, bds = kNoSplit;
    // encoder
    Split16 src = kNoSplit, xa = kNoSplit, xb = kNoSplit, qk = kNoSplit, vt = kNoSplit, ao = kNoSplit, ffh = kNoSplit;
    Split16 qk2 = kNoSplit, vt2 = kNoSplit;      // odd encoder layers: with tile-level dependencies layer l+1 projects while layer l still attends
    unsigned char *kvimg = nullptr, *kvimg2 = nullptr;      // [pairs][8 heads] attention operand images of the encoder's own k / v
    int* sync_ctr = nullptr;      // dataflow counter blocks (common.cuh LaunchSync): kSyncBlocks x kSyncBlockInts ints
    float* ln_tmp = nullptr;      // fp32 [tokens][256]: pre-LayerNorm rows of the SIMT cross-check path
    float2 *enc_st_a = nullptr, *enc_st_b = nullptr;     // [tokens][16] partial row statistics of xa / xb (deferred LayerNorms)
    // decoder
    Split16 qpos = kNoSplit, qp = kNoSplit, t = kNoSplit, qb = kNoSplit, dao = kNoSplit, dh = kNoSplit, hs = kNoSplit,
            hd1 = kNoSplit, hd2 = kNoSplit, t2 = kNoSplit;
    float* dln_tmp = nullptr;
    float2 *dec_st_a = nullptr, *dec_st_b = nullptr;
    // host-buffer entry point staging
    float *img_stage = nullptr, *q_stage = nullptr, *pred_stage = nullptr;
    size_t img_stage_elems = 0, q_stage_elems = 0;
};

}  // namespace
}  // namespace cotr

struct cotr_context {
    cotr_model* model = nullptr;
    cotr::Split16 k = cotr::kNoSplit;    // [max_pairs * 512][6 * 256]
    cotr::Split16 vt = cotr::kNoSplit;   // [max_pairs][6][256][512]  (value projections stored transposed)
    unsigned char* img = nullptr;        // [max_pairs][6][8 heads] attention operand images (common.cuh kAttnHeadImgBytes)
    bool holds_img = false;              // what the last encode wrote: images (tensor-core path) or k / vt (fp32 SIMT path)
    bool batch_invariant = false;        // the schedule policy the last encode ran under (cotr_set_batch_invariant)
    int max_pairs = 0;
    int pairs = 0;                       // pairs encoded by the last cotr_encode_context
};

struct cotr_model {
    int device = 0;
    int gemm_path = 0;          // 0 = tcgen05, 1 = fp32 SIMT
    bool batch_invariant = false;   // cotr_set_batch_invariant: every launch scheduled as at the headline shape
    int launches = 0;
    std::vector<void*> allocs;
    cotr::DevConv stem;
    std::vector<cotr::Block> blocks;
    cotr::DevLinear proj;
    cotr::EncLayer enc[cotr::kEncLayers];
    cotr::DevLinear kv_all;     // [3072][256] rows [l*512, l*512+256) = Wk_l, [l*512+256, l*512+512) = Wv_l
    float* add_kv = nullptr;    // [512][3072]
    float* add_kv_tc = nullptr; // + beta W^T of the last encoder norm2 (deferred LayerNorm)
    cotr::DevLinear qpos_all;   // [1536][256] pre-scaled, bias pre-scaled
    cotr::DecLayer dec[cotr::kDecLayers];
    float *dec_norm_g = nullptr, *dec_norm_b = nullptr;
    cotr::DevLinear head[3];
    float* pos = nullptr;       // [512][256] grid position embedding (fp32, debug / tests)
    cotr::Workspace ws;
    cotr_context* own_ctx = nullptr;
    cudaStream_t host_stream = nullptr;
    cotr::Split16 last_feat = cotr::kNoSplit;
    cotr::Split16 last_mem = cotr::kNoSplit;
    bool last_mem_pre_ln = false;   // tensor-core path: last_mem holds the rows BEFORE the last encoder norm2
    int last_pairs = 0, last_rows = 0;
    // per-launch profiler (cotr_profile_begin / cotr_profile_end): CUDA event pairs on the launching stream
    // CUDA-graph replay of cotr_forward, one executable graph per (B, Q) shape (captured on the second call)
    bool graph_mode = true;
    std::map<long long, cudaGraphExec_t> graphs;
    std::map<long long, int> graph_launches;
    std::set<long long> shapes_seen;
    cotr::Preprocessor* pre = nullptr;         // device-side crop / resize / normalise (cotr_preprocess)
    cotr::FlowMerger* merger = nullptr;        // device-side tail of the dense first guess (cotr_flow_tile_merge)
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_events;      // 2 per record
    std::vector<cotr_launch_record> prof_records;
    int prof_max = 0;
    // The workspace, the staging buffers and own_ctx are shared by every entry point: consecutive calls on different
    // streams are ordered with this event (recorded at the end of each call, waited for by the next call's stream).
    cudaEvent_t order_event = nullptr;
    cudaStream_t order_stream = nullptr;
    bool order_valid = false;
};

namespace cotr {
namespace {

// ----------------------------------------------------------------------------------------------
// weight lookup / upload helpers
// ----------------------------------------------------------------------------------------------
struct TensorMap {
    std::map<std::string, const cotr_tensor*> m;
    const cotr_tensor* get(const std::string& name, std::initializer_list<int64_t> shape) const {
        auto it = m.find(name);
        if (it == m.end()) { set_error("cotr_create: missing tensor '%s'", name.c_str()); return nullptr; }
        const cotr_tensor* t = it->second;
        if (t->ndim != (int)shape.size()) { set_error("cotr_create: '%s' has ndim %d, expected %zu", name.c_str(), t->ndim, shape.size()); return nullptr; }
        int i = 0;
        for (int64_t s : shape) {
            if (t->shape[i] != s) { set_error("cotr_create: '%s' dim %d is %lld, expected %lld", name.c_str(), i, (long long)t->shape[i], (long long)s); return nullptr; }
            ++i;
        }
        if (!t->data) { set_error("cotr_create: '%s' has a null data pointer", name.c_str()); return nullptr; }
        return t;
    }
};

int dev_alloc(cotr_model* m, void** p, size_t bytes) {
    COTR_CHECK_CUDA(cudaMalloc(p, bytes ? bytes : 4));
    m->allocs.push_back(*p);
    return 0;
}

int upload(cotr_model* m, const std::vector<float>& h, float** d) {
    if (dev_alloc(m, (void**)d, h.size() * sizeof(float))) return 1;
    COTR_CHECK_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

int upload_tc(cotr_model* m, const std::vector<float>& w, int N, int K, void** d, float* acc_scale) {
    const size_t bytes = tc_weight_bytes(N, K);
    std::vector<uint8_t> img(bytes);
    *acc_scale = tc_pack_weight(w.data(), N, K, img.data());
    if (dev_alloc(m, d, bytes)) return 1;
    COTR_CHECK_CUDA(cudaMemcpy(*d, img.data(), bytes, cudaMemcpyHostToDevice));
    return 0;
}

int make_linear(cotr_model* m, const std::vector<float>& w, const std::vector<float>* b, int N, int K, DevLinear* out) {
    out->n = N; out->k = K;
    if (upload(m, w, &out->w)) return 1;
    if (upload_tc(m, w, N, K, &out->wtc, &out->wtc_scale)) return 1;
    if (b) { if (upload(m, *b, &out->b)) return 1; }
    return 0;
}

// Linear layer whose input is a deferred LayerNorm (gamma, beta): tensor-core image of W diag(gamma), its column sums
// and the folded bias beta W^T + b (see GemmParams::a_ln_cs).
int make_linear_ln(cotr_model* m, const std::vector<float>& w, const std::vector<float>* b, int N, int K,
                   const float* gamma, const float* beta, DevLinear* out, std::vector<float>* folded_bias = nullptr) {
    out->n = N; out->k = K;
    if (upload(m, w, &out->w)) return 1;
    if (b) { if (upload(m, *b, &out->b)) return 1; }
    std::vector<float> wg((size_t)N * K), cs(N), cb(N);
    for (int n = 0; n < N; ++n) {
        double s = 0.0, c = b ? (double)(*b)[n] : 0.0;
        for (int k = 0; k < K; ++k) {
            const float v = w[(size_t)n * K + k] * gamma[k];
            wg[(size_t)n * K + k] = v;
            s += (double)v;
            c += (double)w[(size_t)n * K + k] * (double)beta[k];
        }
        cs[n] = (float)s;
        cb[n] = (float)c;
    }
    if (upload_tc(m, wg, N, K, &out->wtc, &out->wtc_scale)) return 1;
    if (upload_tc(m, w, N, K, &out->wtc_plain, &out->wtc_plain_scale)) return 1;
    if (upload(m, cs, &out->cs) || upload(m, cb, &out->b_tc)) return 1;
    if (folded_bias) *folded_bias = cb;
    return 0;
}

// backbone.py:46-56 folded into the conv: w' = w * s[o], shift = b - rm * s, s = weight * (rv + 1e-5)^-1/2.
// [cout][7][7][3] (kh, kw, c) -> [cout][7][8][4]: the K order of A_STEM_NHWC4 (common.cuh), zero weights for pixel slot 7 / channel 3
std::vector<float> stem_weight_order(const std::vector<float>& w, int cout) {
    std::vector<float> o((size_t)cout * kStemK, 0.f);
    for (int n = 0; n < cout; ++n)
        for (int y = 0; y < 7; ++y)
            for (int x = 0; x < 7; ++x)
                for (int c = 0; c < 3; ++c)
                    o[(size_t)n * kStemK + y * 32 + x * 4 + c] = w[(((size_t)n * 7 + y) * 7 + x) * 3 + c];
    return o;
}

int make_conv(cotr_model* m, const TensorMap& tm, const std::string& conv, const std::string& bn,
              int cout, int cin, int kh, int kw, int stride, int pad, DevConv* out) {
    const cotr_tensor* w = tm.get(conv + ".weight", {cout, cin, kh, kw});
    const cotr_tensor* g = tm.get(bn + ".weight", {cout});
    const cotr_tensor* b = tm.get(bn + ".bias", {cout});
    const cotr_tensor* rm = tm.get(bn + ".running_mean", {cout});
    const cotr_tensor* rv = tm.get(bn + ".running_var", {cout});
    if (!w || !g || !b || !rm || !rv) return 1;
    std::vector<float> wf((size_t)cout * kh * kw * cin), bf(cout);
    for (int o = 0; o < cout; ++o) {
        const double s = (double)g->data[o] / std::sqrt((double)rv->data[o] + 1e-5);
        bf[o] = (float)((double)b->data[o] - (double)rm->data[o] * s);
        for (int c = 0; c < cin; ++c)
            for (int y = 0; y < kh; ++y)
                for (int x = 0; x < kw; ++x)
                    wf[(((size_t)o * kh + y) * kw + x) * cin + c] =
                        (float)((double)w->data[(((size_t)o * cin + c) * kh + y) * kw + x] * s);
    }
    out->cout = cout; out->cin = cin; out->kh = kh; out->kw = kw; out->stride = stride; out->pad = pad;
    if (kh == 7 && cin == 3) {      // the stem reads the bordered NHWC4 canvas: K = (kh, 8 pixel slots, 4 channels), zeros in the padding
        wf = stem_weight_order(wf, cout);
        out->kw = 8; out->cin = 4; out->stem = true;
    }
    if (upload(m, wf, &out->w)) return 1;
    if (upload_tc(m, wf, cout, out->kh * out->kw * out->cin, &out->wtc, &out->wtc_scale)) return 1;
    if (upload(m, bf, &out->b)) return 1;
    return 0;
}

std::vector<float> to_vec(const cotr_tensor* t, size_t n, size_t offset = 0) {
    return std::vector<float>(t->data + offset, t->data + offset + n);
}

int upload_vec(cotr_model* m, const TensorMap& tm, const std::string& name, int n, float** d) {
    const cotr_tensor* t = tm.get(name, {n});
    if (!t) return 1;
    return upload(m, to_vec(t, n), d);
}

// position_encoding.py:60-72 for the all-False mask of the 16x32 grid, evaluated like the reference in fp32.
std::vector<float> grid_position_table() {
    std::vector<float> pos((size_t)kTokens * kDModel);
    for (int i = 0; i < 16; ++i)
        for (int j = 0; j < 32; ++j) {
            const float y = ((float)(i + 1) - 0.5f) / ((float)16 + 1e-6f);
            const float x = ((float)(j + 1) - 0.5f) / ((float)32 + 1e-6f);
            float* row = pos.data() + (size_t)(i * 32 + j) * kDModel;
            for (int k = 1; k <= 64; ++k) {
                const float kpi = (float)((double)k * 3.14159265358979323846);
                const float ax = kpi * x, ay = kpi * y;
                row[2 * (k - 1) + 0] = (float)std::sin((double)ax);
                row[2 * (k - 1) + 1] = (float)std::sin((double)ay);
                row[128 + 2 * (k - 1) + 0] = (float)std::cos((double)ax);
                row[128 + 2 * (k - 1) + 1] = (float)std::cos((double)ay);
            }
        }
    return pos;
}

// ----------------------------------------------------------------------------------------------
// launch helpers (all kernel launches of the forward go through these, so they can be counted / profiled)
// ----------------------------------------------------------------------------------------------
// Dataflow dependencies between the launches of one call (common.cuh LaunchSync): the planner hands every launch the
// counter block of its predecessor (what to wait for) and a fresh block of its own (where to announce its tiles).
struct SyncPlan {
    int* base = nullptr;       // counter blocks of this call (zeroed by the caller)
    int cap_blocks = 0;
    int next = 0;
    bool on = false;
    const int* prev = nullptr;             // the previous launch's block; null: it announced nothing -> hardware wait
    int prev_total = 0, prev_tile_target = 0, prev_tiles = 0, prev_rows = -1;
};

struct Run {
    cotr_model* m;
    cudaStream_t s;
    SyncPlan* sp = nullptr;
    // batch-invariant schedule (tensor-core path): a launch of M rows is scheduled as if it had sched_rows rows (decoder)
    // or M / sched_pairs rows (encoder of sched_pairs pairs, i.e. one pair's rows); both 0 = as M rows
    int sched_pairs = 0;
    int sched_rows = 0;
};

// The batch-invariant mode schedules every launch as the same call site at the headline shape (B = 1, Q = 1024): the
// backbone and encoder as for one pair, the decoder, query projection and head as for 1024 query rows.
constexpr int kHeadlineQueries = 1024;
inline bool invariant_schedule(const cotr_model* m) { return m->batch_invariant && m->gemm_path == 0; }

// Row count every schedule decision of a launch with M rows reads (tile width, split-K, LayerNorm placement).
inline int sched_rows(const Run& r, int M) {
    if (r.sched_rows > 0) return r.sched_rows;
    if (r.sched_pairs > 0) return M / r.sched_pairs;
    return M;
}

// mode: what this launch would like to wait for (degraded to DEP_ALL when the producer's row tiling does not match);
// rows: size of this launch's row space; returns the LaunchSync with the dependency part and the signal block filled.
LaunchSync plan_dep(const Run& r, int mode, int rows, int span = 0) {
    LaunchSync y;
    memset(&y, 0, sizeof(y));
    SyncPlan* sp = r.sp;
    if (!sp || !sp->on) return y;
    if (sp->prev) {
        const bool tile_ok = sp->prev_tiles > 0 && sp->prev_rows == rows;
        y.dep = sp->prev;
        if (mode == DEP_TILE && tile_ok) { y.dep_mode = DEP_TILE; y.dep_target = sp->prev_tile_target; }
        else if (mode == DEP_SPAN && tile_ok && span > 0 && sp->prev_tiles % span == 0) { y.dep_mode = DEP_SPAN; y.dep_span = span; y.dep_target = sp->prev_tile_target; }
        else { y.dep_mode = DEP_ALL; y.dep_target = sp->prev_total; }
    }
    if (sp->next < sp->cap_blocks) {
        y.sig = sp->base + (size_t)sp->next * kSyncBlockInts;
        sp->next++;
    }
    return y;
}
// after the launch: what the NEXT launch may wait for
void plan_done(const Run& r, const LaunchSync& y, int total, int tile_target, int rows) {
    SyncPlan* sp = r.sp;
    if (!sp || !sp->on) return;
    sp->prev = y.sig;
    sp->prev_total = total;
    sp->prev_tile_target = tile_target;
    sp->prev_tiles = y.sig ? y.sig_tiles : 0;
    sp->prev_rows = rows;
}
inline int sync_tiles_for(int rows) {          // per-tile counters only while they fit the block
    const int t = (rows + 127) / 128;
    return t <= kSyncBlockInts - 1 ? t : 0;
}

enum KernelId { K_GEMM_TC = 0, K_GEMM_SIMT = 1, K_ATTN_TC = 2, K_ATTN_SIMT = 3, K_LAYERNORM = 4, K_MAXPOOL = 5, K_QENC = 6, K_STEM_CANVAS = 7 };

// Counts the launch and, when the profiler is on, brackets it with two events on the launching stream.
struct LaunchScope {
    cotr_model* m;
    cudaStream_t s;
    int slot = -1;
    LaunchScope(const Run& r, int kernel, int M, int N, int K) : m(r.m), s(r.s) {
        m->launches++;
        if (!m->prof_on || (int)m->prof_records.size() >= m->prof_max) return;
        slot = (int)m->prof_records.size();
        while ((int)m->prof_events.size() < 2 * (slot + 1)) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) { slot = -1; return; }
            m->prof_events.push_back(e);
        }
        cotr_launch_record rec;
        rec.kernel = kernel; rec.M = M; rec.N = N; rec.K = K; rec.ms = 0.f;
        m->prof_records.push_back(rec);
        cudaEventRecord(m->prof_events[2 * slot], s);
    }
    ~LaunchScope() {
        if (slot >= 0) cudaEventRecord(m->prof_events[2 * slot + 1], s);
    }
};

GemmParams gemm_base(int M, int N, int K, CSplit16 A, int lda, const float* W, const void* Wtc, float wtc_scale,
                     Split16 out, int ldc) {
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = N; p.K = K;
    p.a = A; p.a_mode = A_ROWMAJOR; p.lda = lda;
    p.Wt = W; p.Wtc = Wtc; p.acc_scale = wtc_scale;
    p.out = out; p.ldc = ldc;
    p.add_period = 1;
    return p;
}

// One tcgen05 GEMM launch with its dataflow bookkeeping.  dep_mode: DEP_ALL / DEP_TILE (the A rows of a CTA's tile come
// from the same 128-row tile of the previous launch, and nothing this launch overwrites is still read by other tiles).
int launch_tc(const Run& r, GemmParams& p, int dep_mode = DEP_ALL) {
    // only the row-major operand kernels exist in a dataflow-capable form (gemm_tc.cu, DLN instantiations): convolutions
    // keep the hardware wait and announce nothing, so their successor falls back to the hardware wait as well
    const bool flow_ok = (p.a_mode == A_ROWMAJOR || p.a_mode == A_TOKENS) && (p.K & 7) == 0 && (p.lda & 7) == 0;
    p.M_sched = sched_rows(r, p.M);
    if (flow_ok) p.sync = plan_dep(r, dep_mode, p.M);
    else if (r.sp) r.sp->prev = nullptr;
    p.sync.sig_tiles = p.sync.sig ? sync_tiles_for(p.M) : 0;
    GemmLaunchInfo info{0, 0, 1};
    LaunchScope scope(r, K_GEMM_TC, p.M, p.N, p.K);
    if (launch_gemm_tc(p, r.s, &info)) return 1;
    if (flow_ok) plan_done(r, p.sync, info.row_tiles * info.col_tiles * info.ksplit, info.col_tiles * info.ksplit, p.M);
    return 0;
}

// ln_scratch: fp32 [M][256] staging for the SIMT path (the tensor-core GEMM fuses LayerNorm into its epilogue).
int run_gemm(const Run& r, GemmParams p, float* ln_scratch, int dep_mode = DEP_ALL) {
    if (r.m->gemm_path == 0 && p.ln_gamma == nullptr) return launch_tc(r, p, dep_mode);
    if (r.m->gemm_path == 0) {
        // The fused LayerNorm epilogue needs the whole 256-wide row in one CTA (128 x 256 tile): with few rows that is
        // a handful of CTAs doing a long serial epilogue while the other SMs idle.  Below ~64 row tiles the GEMM runs
        // with narrow tiles across many SMs and LayerNorm follows as its own (in-place, one warp per row) kernel.
        // The batch-invariant schedule decides from its scheduling row count (<= 1024 rows: always separate).
        p.M_sched = sched_rows(r, p.M);
        const bool defuse = p.ln_gamma != nullptr && (p.M_sched + 127) / 128 < 64;
        const float* g = p.ln_gamma;
        const float* b = p.ln_beta;
        if (defuse) { p.ln_gamma = nullptr; p.ln_beta = nullptr; }
        // (legacy schedule, not used by the deferred-LayerNorm forward: no dataflow announcements)
        if (r.sp) r.sp->prev = nullptr;
        {
            LaunchScope scope(r, K_GEMM_TC, p.M, p.N, p.K);
            if (launch_gemm_tc(p, r.s)) return 1;
        }
        if (defuse) {
            LaunchScope scope(r, K_LAYERNORM, p.M, kDModel, 0);
            if (launch_layernorm(cs(p.out), g, b, p.out, p.M, r.s)) return 1;
        }
        return 0;
    }
    const float* g = p.ln_gamma;
    const float* b = p.ln_beta;
    if (g) {
        COTR_CHECK(p.N == kDModel && ln_scratch != nullptr, "run_gemm: LayerNorm epilogue needs N = 256");
        p.ln_gamma = nullptr; p.ln_beta = nullptr;
    }
    {
        LaunchScope scope(r, K_GEMM_SIMT, p.M, p.N, p.K);
        if (launch_gemm_simt_raw(p, g ? ln_scratch : nullptr, r.s)) return 1;
    }
    if (g) {
        LaunchScope scope(r, K_LAYERNORM, p.M, kDModel, 0);
        if (launch_layernorm_f32(ln_scratch, g, b, Split16{p.out.hi, p.out.lo}, p.M, r.s)) return 1;
    }
    return 0;
}

int run_linear(const Run& r, const DevLinear& L, int M, CSplit16 A, int lda, Split16 out, int ldc, bool relu,
               CSplit16 residual = CSplit16{nullptr, nullptr}, int ldr = 0, const float* ln_g = nullptr,
               const float* ln_b = nullptr, float* ln_scratch = nullptr, int dep_mode = DEP_ALL) {
    // explicit-LayerNorm schedule: layers that also exist in a gamma-folded form use their plain image here
    GemmParams p = gemm_base(M, L.n, L.k, A, lda, L.w, L.wtc_plain ? L.wtc_plain : L.wtc, L.wtc_plain ? L.wtc_plain_scale : L.wtc_scale, out, ldc);
    p.bias = L.b;
    p.relu = relu ? 1 : 0;
    p.res = residual; p.ldr = ldr;
    p.ln_gamma = ln_g; p.ln_beta = ln_b;
    return run_gemm(r, p, ln_scratch, dep_mode);
}

// Tensor-core path only: linear layer with deferred LayerNorms (GemmParams::a_ln_cs / res_ln_part / ln_part_out).
//   a_part     non-null: A holds pre-LayerNorm rows with these partial statistics; L was built by make_linear_ln
//   part_out   non-null: the output rows are pre-LayerNorm rows of a later norm - leave their partial statistics here
//   res_part   non-null: the residual operand is a deferred LayerNorm (res_g, res_b) of the stored rows
int run_linear_dln(const Run& r, const DevLinear& L, int M, CSplit16 A, int lda, Split16 out, int ldc, bool relu,
                   const float2* a_part, float2* part_out, CSplit16 residual = CSplit16{nullptr, nullptr}, int ldr = 0,
                   const float2* res_part = nullptr, const float* res_g = nullptr, const float* res_b = nullptr, int dep_mode = DEP_TILE) {
    GemmParams p = gemm_base(M, L.n, L.k, A, lda, L.w, L.wtc, L.wtc_scale, out, ldc);
    p.bias = a_part ? L.b_tc : L.b;
    p.relu = relu ? 1 : 0;
    p.res = residual; p.ldr = ldr;
    if (a_part) { p.a_ln_cs = L.cs; p.a_ln_part = a_part; }
    p.ln_part_out = part_out;
    p.res_ln_part = res_part; p.res_ln_gamma = res_g; p.res_ln_beta = res_b;
    return launch_tc(r, p, dep_mode);
}

int run_conv(const Run& r, const DevConv& c, int n_img, CSplit16 in, int H, int W, Split16 out, bool relu, CSplit16 residual) {
    const int OH = c.stem ? H / 2 : (H + 2 * c.pad - c.kh) / c.stride + 1;
    const int OW = c.stem ? W / 2 : (W + 2 * c.pad - c.kw) / c.stride + 1;
    GemmParams p = gemm_base(n_img * OH * OW, c.cout, c.kh * c.kw * c.cin, in, c.cin, c.w, c.wtc, c.wtc_scale, out, c.cout);
    if (c.stem) {
        p.a_mode = A_STEM_NHWC4;        // `in` is the bordered canvas (launch_stem_canvas)
    } else if (c.kh == 1 && c.kw == 1 && c.stride == 1) {
        p.a_mode = A_ROWMAJOR;          // NHWC 1x1 convolution is a plain GEMM over pixels
    } else {
        p.a_mode = A_CONV_NHWC;
    }
    p.H = H; p.W = W; p.C = c.cin; p.OH = OH; p.OW = OW;
    p.KH = c.kh; p.KW = c.kw; p.stride = c.stride; p.pad = c.pad;
    p.bias = c.b;
    p.relu = relu ? 1 : 0;
    p.res = residual; p.ldr = c.cout;
    return run_gemm(r, p, nullptr);
}

// dep_mode / span: DEP_TILE (decoder: a CTA reads only its own 128 query rows from the previous launch) or DEP_SPAN
// (encoder: the keys and values of the whole pair, `span` row tiles); both need query tiles aligned with 128-row tiles
int run_attention(const Run& r, AttnParams p, int dep_mode = DEP_ALL, int span = 0) {
    // recorded as M = query rows, N = 512 keys, K = 32 x 8 heads
    const int rows = p.nq * p.npairs;
    if (r.sched_rows > 0) p.nq_sched = r.sched_rows;       // batch-invariant decoder: tcgen05 for every nq >= 1
    // launch_attention_tc hands launches with fewer than 32 (scheduling) query rows to the SIMT kernel
    const bool simt = r.m->gemm_path != 0 || (p.nq_sched > 0 ? p.nq_sched : p.nq) < 32;
    LaunchScope scope(r, simt ? K_ATTN_SIMT : K_ATTN_TC, rows, kTokens, kDModel);
    if (r.m->gemm_path != 0) return launch_attention_simt(p, r.s);
    if (simt || p.nq < 32) {                  // SIMT, or a partial tile: hardware wait, no announcements
        if (r.sp) r.sp->prev = nullptr;
        return launch_attention_tc(p, r.s);
    }
    const bool aligned = (p.nq % 128) == 0;
    p.sync = plan_dep(r, aligned ? dep_mode : DEP_ALL, rows, span);
    p.sync.sig_tiles = (p.sync.sig && aligned) ? sync_tiles_for(rows) : 0;
    if (launch_attention_tc(p, r.s)) return 1;
    plan_done(r, p.sync, ((p.nq + 127) / 128) * kHeads * p.npairs, kHeads, rows);
    return 0;
}

// ----------------------------------------------------------------------------------------------
// workspace
// ----------------------------------------------------------------------------------------------
constexpr size_t kStemElems = 128 * 128 * 64;      // per image
constexpr size_t kBigElems = 64 * 64 * 256;        // largest block input / output per image
constexpr size_t kT1Elems = 64 * 64 * 128;         // largest conv1 output per image (layer2.0)
constexpr size_t kT2Elems = 64 * 64 * 64;          // largest conv2 output per image (layer1)

size_t encode_ws_elems(int B) {
    const size_t img = 2 * (size_t)B;
    const size_t tok = (size_t)B * kTokens;
    return img * (kStemCanvasElems + kStemElems + 3 * kBigElems + kT1Elems + kT2Elems) + tok * (kDModel * 4 + 4 * kDModel + kFF) +
           2 * (size_t)B * kVtLayer + tok * kDModel /* fp32 LN scratch */ + tok * 64 /* row statistics */;
}
size_t decode_ws_elems(int rows) {
    return (size_t)rows * (kDModel * 8 + kQpCols + kFF) + (size_t)rows * kDModel /* fp32 LN scratch */ + (size_t)rows * 64 /* row statistics */;
}

// split16 buffer of `elems` elements: one allocation, hi plane first (elems is always a multiple of 8)
int ws_alloc(Split16* t, size_t elems) {
    __half* base = nullptr;
    COTR_CHECK_CUDA(cudaMalloc((void**)&base, elems * 2 * sizeof(__half)));
    t->hi = base;
    t->lo = base + elems;
    return 0;
}
void ws_free(Split16* t) { if (t->hi) { cudaFree(t->hi); } t->hi = nullptr; t->lo = nullptr; }
int ws_alloc_f32(float** p, size_t elems) {
    COTR_CHECK_CUDA(cudaMalloc((void**)p, elems * sizeof(float)));
    return 0;
}
void ws_free_f32(float** p) { if (*p) { cudaFree(*p); *p = nullptr; } }

// Dataflow counters: kSyncEncodeBlocks for cotr_encode_context, kSyncChunkBlocks per decoder chunk behind them.
constexpr int kSyncEncodeBlocks = 128;
constexpr int kSyncChunkBlocks = 48;
constexpr int kSyncBlocks = 1024;

int ensure_sync_ctr(cotr_model* m) {
    if (m->ws.sync_ctr) return 0;
    COTR_CHECK_CUDA(cudaMalloc((void**)&m->ws.sync_ctr, (size_t)kSyncBlocks * kSyncBlockInts * sizeof(int)));
    return 0;
}
// bring-up switch: cotr_debug_set_variant bit 18 turns the dataflow dependencies off (hardware griddepcontrol.wait everywhere)
// Schedule selection (profiles/r02_deferred_layernorm.md has the measurements behind it).
// Deferred LayerNorm (no LayerNorm launches; consumers normalise on the fly) removes 12 launches from the encoder and
// 12 from each decoder chunk but makes its consumer GEMMs a little longer: on B200 it loses 2.4% on the 512-token /
// 1024-row chains of the headline shape and wins 3-5% once a section has thousands of rows, so each section picks it
// by its row count.  cotr_debug_set_variant overrides: bit 19 = always deferred, bit 16 = never.  Bits 19 + 18 together
// additionally swap griddepcontrol.wait for the counter-based dataflow dependencies of common.cuh - measured slower
// everywhere, opt-in only.
constexpr int kDeferredLnMinRows = 2048;
inline bool deferred_ln_enabled(const cotr_model* m, int rows) {
    if (m->gemm_path != 0 || (g_tc_variant & (1 << 16))) return false;
    return (g_tc_variant & (1 << 19)) != 0 || rows >= kDeferredLnMinRows;
}
inline bool dataflow_enabled(const cotr_model* m) {
    return m->gemm_path == 0 && (g_tc_variant & (1 << 18)) != 0 && (g_tc_variant & (1 << 19)) != 0 && !(g_tc_variant & (1 << 16)) && g_use_pdl;
}

// Captured graphs embed workspace / staging / context addresses: whenever one of those is reallocated every graph is
// stale.  The shapes stay "seen", so the next call of each shape re-captures against the new buffers.
void drop_graphs(cotr_model* m) {
    for (auto& kv : m->graphs) cudaGraphExecDestroy(kv.second);
    m->graphs.clear();
    m->graph_launches.clear();
}

// Cross-stream ordering of the entry points (see cotr_model::order_event).  Same-stream calls need no wait.
struct CallOrder {
    cotr_model* m;
    cudaStream_t s;
    CallOrder(cotr_model* m_, cudaStream_t s_) : m(m_), s(s_) {
        if (m->order_valid && m->order_stream != s && m->order_event) cudaStreamWaitEvent(s, m->order_event, 0);
    }
    ~CallOrder() {
        if (!m->order_event && cudaEventCreateWithFlags(&m->order_event, cudaEventDisableTiming) != cudaSuccess) {
            m->order_event = nullptr;
            return;
        }
        if (cudaEventRecord(m->order_event, s) == cudaSuccess) { m->order_stream = s; m->order_valid = true; }
    }
};

int ensure_encode_ws(cotr_model* m, int B) {
    Workspace& w = m->ws;
    if (B <= w.cap_pairs) return 0;
    COTR_CHECK_CUDA(cudaDeviceSynchronize());
    drop_graphs(m);
    Split16* bufs[] = {&w.canvas, &w.stem, &w.bx, &w.by, &w.bt1, &w.bt2, &w.bds, &w.src, &w.xa, &w.xb, &w.qk, &w.vt, &w.ao, &w.ffh, &w.qk2, &w.vt2};
    for (Split16* b : bufs) ws_free(b);
    ws_free_f32(&w.ln_tmp);
    if (w.kvimg) { cudaFree(w.kvimg); w.kvimg = nullptr; }
    if (w.kvimg2) { cudaFree(w.kvimg2); w.kvimg2 = nullptr; }
    ws_free_f32(reinterpret_cast<float**>(&w.enc_st_a));
    ws_free_f32(reinterpret_cast<float**>(&w.enc_st_b));
    const size_t img = 2 * (size_t)B, tok = (size_t)B * kTokens;
    if (ws_alloc(&w.canvas, img * kStemCanvasElems) || ws_alloc(&w.stem, img * kStemElems) || ws_alloc(&w.bx, img * kBigElems) || ws_alloc(&w.by, img * kBigElems) ||
        ws_alloc(&w.bds, img * kBigElems) || ws_alloc(&w.bt1, img * kT1Elems) || ws_alloc(&w.bt2, img * kT2Elems) ||
        ws_alloc(&w.src, tok * kDModel) || ws_alloc(&w.xa, tok * kDModel) || ws_alloc(&w.xb, tok * kDModel) ||
        ws_alloc(&w.qk, tok * 2 * kDModel) || ws_alloc(&w.vt, (size_t)B * kVtLayer) || ws_alloc(&w.ao, tok * kDModel) ||
        ws_alloc(&w.qk2, tok * 2 * kDModel) || ws_alloc(&w.vt2, (size_t)B * kVtLayer) ||
        ws_alloc(&w.ffh, tok * kFF) || ws_alloc_f32(&w.ln_tmp, tok * kDModel) ||
        ws_alloc_f32(reinterpret_cast<float**>(&w.enc_st_a), tok * 32) || ws_alloc_f32(reinterpret_cast<float**>(&w.enc_st_b), tok * 32))
        return 1;
    COTR_CHECK_CUDA(cudaMalloc((void**)&w.kvimg, (size_t)B * kHeads * kAttnHeadImgBytes));
    COTR_CHECK_CUDA(cudaMalloc((void**)&w.kvimg2, (size_t)B * kHeads * kAttnHeadImgBytes));
    // the 16 pad bytes of every value key group are copied by the bulk TMA: keep them defined
    COTR_CHECK_CUDA(cudaMemset(w.kvimg, 0, (size_t)B * kHeads * kAttnHeadImgBytes));
    COTR_CHECK_CUDA(cudaMemset(w.kvimg2, 0, (size_t)B * kHeads * kAttnHeadImgBytes));
    // the border of the stem canvas is the convolution's zero padding: written here, never again
    COTR_CHECK_CUDA(cudaMemset(w.canvas.hi, 0, img * kStemCanvasElems * 2 * sizeof(__half)));
    w.cap_pairs = B;
    return 0;
}

int ensure_decode_ws(cotr_model* m, int rows) {
    Workspace& w = m->ws;
    if (rows <= w.cap_rows) return 0;
    COTR_CHECK_CUDA(cudaDeviceSynchronize());
    drop_graphs(m);
    Split16* bufs[] = {&w.qpos, &w.qp, &w.t, &w.qb, &w.dao, &w.dh, &w.hs, &w.hd1, &w.hd2, &w.t2};
    for (Split16* b : bufs) ws_free(b);
    ws_free_f32(&w.dln_tmp);
    ws_free_f32(reinterpret_cast<float**>(&w.dec_st_a));
    ws_free_f32(reinterpret_cast<float**>(&w.dec_st_b));
    const size_t R = ((size_t)rows + 7) & ~(size_t)7;
    if (ws_alloc(&w.qpos, R * kDModel) || ws_alloc(&w.qp, R * kQpCols) || ws_alloc(&w.t, R * kDModel) ||
        ws_alloc(&w.qb, R * kDModel) || ws_alloc(&w.dao, R * kDModel) || ws_alloc(&w.dh, R * kFF) ||
        ws_alloc(&w.hs, R * kDModel) || ws_alloc(&w.hd1, R * kDModel) || ws_alloc(&w.hd2, R * kDModel) ||
        ws_alloc(&w.t2, R * kDModel) || ws_alloc_f32(&w.dln_tmp, R * kDModel) ||
        ws_alloc_f32(reinterpret_cast<float**>(&w.dec_st_a), R * 32) || ws_alloc_f32(reinterpret_cast<float**>(&w.dec_st_b), R * 32))
        return 1;
    w.cap_rows = rows;
    return 0;
}

// ----------------------------------------------------------------------------------------------
// forward schedule
// ----------------------------------------------------------------------------------------------
int encode_impl(cotr_model* m, const float* img, int B, cotr_context* ctx, cudaStream_t s) {
    COTR_CHECK(B >= 1, "cotr_encode_context: B must be >= 1 (got %d)", B);
    COTR_CHECK(ctx && ctx->model == m, "cotr_encode_context: context does not belong to this model");
    COTR_CHECK(B <= ctx->max_pairs, "cotr_encode_context: B = %d exceeds the context capacity %d", B, ctx->max_pairs);
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    if (ensure_encode_ws(m, B) || ensure_sync_ctr(m)) return 1;
    Workspace& w = m->ws;
    SyncPlan plan;
    plan.on = dataflow_enabled(m);
    plan.base = w.sync_ctr;
    plan.cap_blocks = kSyncEncodeBlocks;
    if (plan.on) COTR_CHECK_CUDA(cudaMemsetAsync(w.sync_ctr, 0, (size_t)kSyncEncodeBlocks * kSyncBlockInts * sizeof(int), s));
    Run r{m, s, &plan};
    if (invariant_schedule(m)) r.sched_pairs = B;
    const int n_img = 2 * B;
    const CSplit16 none{nullptr, nullptr};

    // backbone.py:81-82: the two 256x256 halves go through the ResNet body as independent images.
    // Stem: conv 7x7/2 (+FrozenBN folded) + ReLU, then MaxPool 3x3/2  (torchvision resnet.py _forward_impl).
    {
        LaunchScope scope(r, K_STEM_CANVAS, n_img * 256 * 256, 4, 0);
        LaunchSync y = plan_dep(r, DEP_ALL, n_img * 256 * 256);
        if (launch_stem_canvas(img, w.canvas, n_img, s, y)) return 1;
        const size_t blocks = ((size_t)n_img * 256 * 256 + 255) / 256;
        plan_done(r, y, (int)(blocks < 148 * 16 ? blocks : 148 * 16), 0, n_img * 256 * 256);
    }
    if (run_conv(r, m->stem, n_img, cs(w.canvas), 256, 256, w.stem, true, none)) return 1;
    {
        LaunchScope scope(r, K_MAXPOOL, n_img * 64 * 64, 64, 0);
        LaunchSync y = plan_dep(r, DEP_ALL, n_img * 64 * 64);
        if (launch_maxpool_3x3s2_nhwc(cs(w.stem), w.bx, n_img, 128, 128, 64, s, y)) return 1;
        const size_t total = (size_t)n_img * 64 * 64 * 8;
        const size_t blocks = (total + 255) / 256;
        plan_done(r, y, (int)(blocks < 148 * 16 ? blocks : 148 * 16), 0, n_img * 64 * 64);
    }

    Split16 x = w.bx;
    Split16 y = w.by;
    int H = 64, W = 64;
    for (const Block& b : m->blocks) {
        // torchvision Bottleneck (v1.5): 1x1 -> 3x3(stride) -> 1x1, + identity | downsample, ReLU
        if (run_conv(r, b.c1, n_img, cs(x), H, W, w.bt1, true, none)) return 1;
        if (run_conv(r, b.c2, n_img, cs(w.bt1), H, W, w.bt2, true, none)) return 1;
        const int OH = H / b.c2.stride, OW = W / b.c2.stride;
        CSplit16 identity = cs(x);
        if (b.has_ds) {
            if (run_conv(r, b.ds, n_img, cs(x), H, W, w.bds, false, none)) return 1;
            identity = cs(w.bds);
        }
        if (run_conv(r, b.c3, n_img, cs(w.bt2), OH, OW, y, true, identity)) return 1;
        Split16 t = x; x = y; y = t;
        H = OH; W = OW;
    }
    m->last_feat = x;   // (2B,16,16,1024) NHWC

    // cotr_model.py:37 input_proj (1x1 conv 1024 -> 256) fused with the left|right concat (backbone.py:85)
    // and the flatten to token-major (transformer.py:50): row = pair*512 + i*32 + j.
    const int T = B * kTokens;
    {
        GemmParams p = gemm_base(T, kDModel, 1024, cs(x), 1024, m->proj.w, m->proj.wtc, m->proj.wtc_scale, w.src, kDModel);
        p.a_mode = A_TOKENS;
        p.bias = m->proj.b;
        if (run_gemm(r, p, nullptr)) return 1;
    }

    // transformer.py:143-159 x6 (post-LN).  q = k = x + pos is folded into the constant add_qkv matrix.
    // q | k land row-major in qk [T][512]; v lands transposed in vt [pair][256][512] (what P V needs as its B operand).
    Split16 xin = w.src;      // layer input
    if (deferred_ln_enabled(m, sched_rows(r, T))) {
        // Tensor-core path: no LayerNorm kernel and no LayerNorm epilogue.  A LayerNorm output is never stored; its
        // producer writes the pre-norm rows (xa: x + attention, xb: x1 + FFN) and every consumer applies the norm on
        // the fly (GemmParams::a_ln_cs for GEMM inputs, res_ln_part for residual operands) from the partial row
        // statistics the producer's epilogue leaves behind: enc_st_a belongs to xa (norm1), enc_st_b to xb (norm2).
        const int n_enc_dbg = (g_tc_variant >> 20) & 7;        // bring-up: stop after this many encoder layers (0 = all)
        for (int l = 0; l < (n_enc_dbg ? n_enc_dbg : kEncLayers); ++l) {
            const EncLayer& e = m->enc[l];
            const bool ln_in = l > 0;          // the layer input is LN2_{l-1}(xb), deferred
            // q|k and v^T alternate between two buffers: with tile-level dependencies the next layer's projection of a
            // row tile may run while other tiles of this layer still attend to the old keys / values
            const Split16 qk_l = (l & 1) ? w.qk2 : w.qk, vt_l = (l & 1) ? w.vt2 : w.vt;
            unsigned char* const kvimg_l = (l & 1) ? w.kvimg2 : w.kvimg;
            {
                GemmParams p = gemm_base(T, 3 * kDModel, kDModel, cs(xin), kDModel, e.qkv.w, e.qkv.wtc, e.qkv.wtc_scale, qk_l, 2 * kDModel);
                p.addmat = e.add_qkv_tc; p.add_period = kTokens; p.ld_add = 3 * kDModel;
                p.remap = 1;
                p.blk_map[0] = 0; p.blk_map[1] = kDModel; p.blk_map[2] = -1;
                p.vt = vt_l; p.n_vt = 1;
                p.kv_img = kvimg_l; p.blk_map[1] = -1000;           // keys and values go straight into the attention operand images
                if (ln_in) { p.a_ln_cs = e.qkv.cs; p.a_ln_part = w.enc_st_b; }
                if (launch_tc(r, p, DEP_TILE)) return 1;
            }
            AttnParams a{};
            a.q = cs(qk_l); a.ldq = 2 * kDModel;
            a.k = offset(cs(qk_l), kDModel); a.ldk = 2 * kDModel;
            a.vt = cs(vt_l); a.vt_pair_stride = kVtLayer;
            a.kv_img = kvimg_l; a.img_pair_stride = kHeads * kAttnHeadImgBytes;
            a.out = w.ao; a.ldo = kDModel;
            a.nq = kTokens; a.npairs = B; a.pair0 = 0;
            if (run_attention(r, a, DEP_SPAN, kTokens / 128)) return 1;
            // xa = x + out_proj(attn)                                   (transformer.py:149-154, norm1 deferred)
            if (run_linear_dln(r, e.o, T, cs(w.ao), kDModel, w.xa, kDModel, false, nullptr, w.enc_st_a, cs(xin), kDModel,
                               ln_in ? w.enc_st_b : nullptr, ln_in ? m->enc[l - 1].ln2_g : nullptr, ln_in ? m->enc[l - 1].ln2_b : nullptr)) return 1;
            // h = relu(W1 norm1(xa) + b1)                               (transformer.py:155)
            if (run_linear_dln(r, e.l1, T, cs(w.xa), kDModel, w.ffh, kFF, true, w.enc_st_a, nullptr)) return 1;
            // xb = norm1(xa) + W2 h + b2                                (transformer.py:155-157, norm2 deferred)
            if (run_linear_dln(r, e.l2, T, cs(w.ffh), kFF, w.xb, kDModel, false, nullptr, w.enc_st_b, cs(w.xa), kDModel,
                               w.enc_st_a, e.ln1_g, e.ln1_b)) return 1;
            xin = w.xb;
        }
        m->last_mem = xin;
        m->last_mem_pre_ln = true;
        // K / V projections of all 6 decoder layers from norm2(xb) of the last encoder layer (deferred as well)
        {
            GemmParams p = gemm_base(T, 2 * kKCols, kDModel, cs(xin), kDModel, m->kv_all.w, m->kv_all.wtc, m->kv_all.wtc_scale, ctx->k, kKCols);
            p.addmat = m->add_kv_tc; p.add_period = kTokens; p.ld_add = 2 * kKCols;
            p.remap = 1;
            for (int l = 0; l < kDecLayers; ++l) {
                p.blk_map[2 * l] = l * kDModel;
                p.blk_map[2 * l + 1] = -(l + 1);
            }
            p.vt = ctx->vt; p.n_vt = kDecLayers;
            p.kv_img = ctx->img;
            for (int l = 0; l < kDecLayers; ++l) p.blk_map[2 * l] = -1000 - l;
            p.a_ln_cs = m->kv_all.cs; p.a_ln_part = w.enc_st_b;
            if (launch_tc(r, p, DEP_TILE)) return 1;
        }
        ctx->pairs = B;
        ctx->holds_img = true;
        ctx->batch_invariant = m->batch_invariant;
        m->last_pairs = B;
        return 0;
    }
    // default schedule (and the fp32 SIMT cross-check path): explicit LayerNorm launches, the checkpoint's weights as they are
    m->last_mem_pre_ln = false;
    const bool tc = m->gemm_path == 0;      // tensor-core path: keys / values are written as attention operand images
    const int n_enc_dbg = (g_tc_variant >> 20) & 7;
    for (int l = 0; l < (n_enc_dbg ? n_enc_dbg : kEncLayers); ++l) {
        const EncLayer& e = m->enc[l];
        {
            GemmParams p = gemm_base(T, 3 * kDModel, kDModel, cs(xin), kDModel, e.qkv.w, e.qkv.wtc_plain ? e.qkv.wtc_plain : e.qkv.wtc, e.qkv.wtc_plain ? e.qkv.wtc_plain_scale : e.qkv.wtc_scale, w.qk, 2 * kDModel);
            p.addmat = e.add_qkv; p.add_period = kTokens; p.ld_add = 3 * kDModel;
            p.remap = 1;
            p.blk_map[0] = 0; p.blk_map[1] = kDModel; p.blk_map[2] = -1;
            p.vt = w.vt; p.n_vt = 1;
            if (tc) { p.kv_img = w.kvimg; p.blk_map[1] = -1000; }
            if (run_gemm(r, p, nullptr)) return 1;
        }
        AttnParams a{};
        a.q = cs(w.qk); a.ldq = 2 * kDModel;
        a.k = offset(cs(w.qk), kDModel); a.ldk = 2 * kDModel;
        a.vt = cs(w.vt); a.vt_pair_stride = kVtLayer;
        if (tc) { a.kv_img = w.kvimg; a.img_pair_stride = kHeads * kAttnHeadImgBytes; }
        a.out = w.ao; a.ldo = kDModel;
        a.nq = kTokens; a.npairs = B; a.pair0 = 0;
        if (run_attention(r, a)) return 1;
        // x1 = LN1(x + out_proj(attn))
        if (run_linear(r, e.o, T, cs(w.ao), kDModel, w.xa, kDModel, false, cs(xin), kDModel, e.ln1_g, e.ln1_b, w.ln_tmp)) return 1;
        // x2 = LN2(x1 + W2 relu(W1 x1 + b1) + b2)
        if (run_linear(r, e.l1, T, cs(w.xa), kDModel, w.ffh, kFF, true)) return 1;
        if (run_linear(r, e.l2, T, cs(w.ffh), kFF, w.xb, kDModel, false, cs(w.xa), kDModel, e.ln2_g, e.ln2_b, w.ln_tmp)) return 1;
        xin = w.xb;
    }
    m->last_mem = xin;

    // transformer.py:192-195: K_l = (mem + pos) Wk_l^T + bk_l, V_l = mem Wv_l^T + bv_l for all 6 decoder layers in ONE
    // GEMM (N = 3072): K blocks go row-major into ctx->k [T][1536], V blocks transposed into ctx->vt [pair][6][256][512].
    {
        GemmParams p = gemm_base(T, 2 * kKCols, kDModel, cs(xin), kDModel, m->kv_all.w, m->kv_all.wtc_plain ? m->kv_all.wtc_plain : m->kv_all.wtc, m->kv_all.wtc_plain ? m->kv_all.wtc_plain_scale : m->kv_all.wtc_scale, ctx->k, kKCols);
        p.addmat = m->add_kv; p.add_period = kTokens; p.ld_add = 2 * kKCols;
        p.remap = 1;
        for (int l = 0; l < kDecLayers; ++l) {
            p.blk_map[2 * l] = l * kDModel;
            p.blk_map[2 * l + 1] = -(l + 1);
        }
        p.vt = ctx->vt; p.n_vt = kDecLayers;
        if (tc) {
            p.kv_img = ctx->img;
            for (int l = 0; l < kDecLayers; ++l) p.blk_map[2 * l] = -1000 - l;
        }
        if (run_gemm(r, p, nullptr)) return 1;
    }
    ctx->pairs = B;
    ctx->holds_img = tc;
    ctx->batch_invariant = m->batch_invariant;
    m->last_pairs = B;
    return 0;
}

int decode_chunk(cotr_model* m, const cotr_context* ctx, const float* queries, float* pred, int pair0, int npairs,
                 int nq, cudaStream_t s, int chunk_index) {
    Workspace& w = m->ws;
    // dataflow counters of this chunk (zeroed by decode_impl); the chunk's first launch has no announced producer and
    // falls back to the hardware wait, which also orders it behind the previous chunk / the encoder
    SyncPlan plan;
    plan.on = dataflow_enabled(m) && kSyncEncodeBlocks + (chunk_index + 1) * kSyncChunkBlocks <= kSyncBlocks;
    plan.base = w.sync_ctr + (size_t)(kSyncEncodeBlocks + chunk_index * kSyncChunkBlocks) * kSyncBlockInts;
    plan.cap_blocks = kSyncChunkBlocks;
    Run r{m, s, &plan};
    if (invariant_schedule(m)) r.sched_rows = kHeadlineQueries;
    const int R = npairs * nq;
    const CSplit16 none{nullptr, nullptr};
    // cotr_model.py:34-35 query_proj (lin_sine, depth 64)
    {
        LaunchScope scope(r, K_QENC, R, kDModel, 0);
        LaunchSync y = plan_dep(r, DEP_ALL, R);
        y.sig_tiles = (y.sig && (R % 128) == 0) ? sync_tiles_for(R) : 0;      // one block per row: whole tiles only
        if (launch_query_encode(queries, w.qpos, R, s, y)) return 1;
        plan_done(r, y, R, 128, R);
    }
    // q-side of transformer.py:192: ((t + qpos) Wq^T + bq) s  =  t (s Wq)^T + [qpos (s Wq)^T + s bq]; the bracket for
    // all 6 layers is one GEMM.
    if (run_linear(r, m->qpos_all, R, cs(w.qpos), kDModel, w.qp, kQpCols, false, none, 0, nullptr, nullptr, nullptr, DEP_TILE)) return 1;

    if (deferred_ln_enabled(m, sched_rows(r, R))) {
        // Tensor-core path with deferred LayerNorms (see encode_impl): w.t = t + attention (norm2 deferred),
        // w.t2 = t1 + FFN (norm3 deferred); dec_st_a = partial row statistics of w.t (norm2), dec_st_b of w.t2 (norm3).
        for (int l = 0; l < kDecLayers; ++l) {
            const DecLayer& d = m->dec[l];
            const bool ln_in = l > 0;
            CSplit16 q = cs(w.qp);      // layer 0: tgt = 0 (transformer.py:54), so q is the qpos projection alone
            int ldq = kQpCols;
            if (ln_in) {
                if (run_linear_dln(r, d.q, R, cs(w.t2), kDModel, w.qb, kDModel, false, w.dec_st_b, nullptr,
                                   offset(cs(w.qp), (size_t)l * kDModel), kQpCols)) return 1;
                q = cs(w.qb); ldq = kDModel;
            }
            AttnParams a{};
            a.q = q; a.ldq = ldq;
            a.k = offset(cs(ctx->k), (size_t)l * kDModel); a.ldk = kKCols;
            a.vt = offset(cs(ctx->vt), (size_t)l * kVtLayer); a.vt_pair_stride = kDecLayers * kVtLayer;
            if (ctx->holds_img) { a.kv_img = ctx->img + (size_t)l * kHeads * kAttnHeadImgBytes; a.img_pair_stride = (size_t)kDecLayers * kHeads * kAttnHeadImgBytes; }
            a.out = w.dao; a.ldo = kDModel;
            a.nq = nq; a.npairs = npairs; a.pair0 = pair0;
            if (run_attention(r, a, DEP_TILE)) return 1;
            // transformer.py:196-197: t = t + out_proj(attn)   (norm2 deferred; t = norm3_{l-1}(t2), deferred, or 0)
            if (run_linear_dln(r, d.o, R, cs(w.dao), kDModel, w.t, kDModel, false, nullptr, w.dec_st_a, ln_in ? cs(w.t2) : none, kDModel,
                               ln_in ? w.dec_st_b : nullptr, ln_in ? m->dec[l - 1].ln3_g : nullptr, ln_in ? m->dec[l - 1].ln3_b : nullptr)) return 1;
            // transformer.py:198-200: t2 = norm2(t) + linear2(relu(linear1(norm2(t))))   (norm3 deferred)
            if (run_linear_dln(r, d.l1, R, cs(w.t), kDModel, w.dh, kFF, true, w.dec_st_a, nullptr)) return 1;
            if (run_linear_dln(r, d.l2, R, cs(w.dh), kFF, w.t2, kDModel, false, nullptr, w.dec_st_b, cs(w.t), kDModel,
                               w.dec_st_a, d.ln2_g, d.ln2_b)) return 1;
        }
        // norm3 of the last layer, then transformer.py:110-111 decoder.norm, in one pass over the rows
        {
            const DecLayer& d = m->dec[kDecLayers - 1];
            LaunchScope scope(r, K_LAYERNORM, R, kDModel, 0);
            LaunchSync y = plan_dep(r, DEP_TILE, R);
            y.sig_tiles = (y.sig && (R % 128) == 0) ? sync_tiles_for(R) : 0;      // 8 rows per block: whole tiles only
            if (launch_layernorm_twice(cs(w.t2), d.ln3_g, d.ln3_b, m->dec_norm_g, m->dec_norm_b, w.hs, R, s, y)) return 1;
            plan_done(r, y, (R + 7) / 8, 16, R);
        }
    } else {
        for (int l = 0; l < kDecLayers; ++l) {
            const DecLayer& d = m->dec[l];
            CSplit16 q = cs(w.qp);      // layer 0: tgt = 0 (transformer.py:54), so q is the qpos projection alone
            int ldq = kQpCols;
            if (l > 0) {
                if (run_linear(r, d.q, R, cs(w.t), kDModel, w.qb, kDModel, false, offset(cs(w.qp), (size_t)l * kDModel), kQpCols)) return 1;
                q = cs(w.qb); ldq = kDModel;
            }
            AttnParams a{};
            a.q = q; a.ldq = ldq;
            a.k = offset(cs(ctx->k), (size_t)l * kDModel); a.ldk = kKCols;
            a.vt = offset(cs(ctx->vt), (size_t)l * kVtLayer); a.vt_pair_stride = kDecLayers * kVtLayer;
            if (ctx->holds_img) { a.kv_img = ctx->img + (size_t)l * kHeads * kAttnHeadImgBytes; a.img_pair_stride = (size_t)kDecLayers * kHeads * kAttnHeadImgBytes; }
            a.out = w.dao; a.ldo = kDModel;
            a.nq = nq; a.npairs = npairs; a.pair0 = pair0;
            if (run_attention(r, a)) return 1;
            // transformer.py:196-197: t = norm2(t + out_proj(attn))
            if (run_linear(r, d.o, R, cs(w.dao), kDModel, w.t, kDModel, false, l > 0 ? cs(w.t) : none, kDModel, d.ln2_g, d.ln2_b, w.dln_tmp)) return 1;
            // transformer.py:198-200: t = norm3(t + linear2(relu(linear1(t))))
            if (run_linear(r, d.l1, R, cs(w.t), kDModel, w.dh, kFF, true)) return 1;
            if (run_linear(r, d.l2, R, cs(w.dh), kFF, w.t, kDModel, false, cs(w.t), kDModel, d.ln3_g, d.ln3_b, w.dln_tmp)) return 1;
        }
        // transformer.py:110-111 decoder.norm on the last level; cotr_model.py:38-39 corr_embed on that level only.
        {
            LaunchScope scope(r, K_LAYERNORM, R, kDModel, 0);
            if (launch_layernorm(cs(w.t), m->dec_norm_g, m->dec_norm_b, w.hs, R, s)) return 1;
        }
    }
    if (run_linear(r, m->head[0], R, cs(w.hs), kDModel, w.hd1, kDModel, true, none, 0, nullptr, nullptr, nullptr, DEP_TILE)) return 1;
    if (run_linear(r, m->head[1], R, cs(w.hd1), kDModel, w.hd2, kDModel, true, none, 0, nullptr, nullptr, nullptr, DEP_TILE)) return 1;
    {
        GemmParams p = gemm_base(R, 2, kDModel, cs(w.hd2), kDModel, m->head[2].w, m->head[2].wtc, m->head[2].wtc_scale, kNoSplit, 2);
        p.bias = m->head[2].b;
        p.out_f32 = pred;
        if (run_gemm(r, p, nullptr, DEP_TILE)) return 1;
    }
    return 0;
}

int decode_impl(cotr_model* m, const cotr_context* ctx, const float* queries, int B, int Q, float* pred, cudaStream_t s) {
    COTR_CHECK(ctx && ctx->model == m, "cotr_decode: context does not belong to this model");
    COTR_CHECK(B >= 1 && B == ctx->pairs, "cotr_decode: B = %d but the context holds %d pairs", B, ctx ? ctx->pairs : -1);
    COTR_CHECK(Q >= 0, "cotr_decode: negative Q");
    COTR_CHECK(ctx->holds_img == (m->gemm_path == 0), "cotr_decode: the context was encoded under the other matrix-multiply path "
               "(cotr_set_gemm_path): re-encode it");
    COTR_CHECK(ctx->batch_invariant == m->batch_invariant, "cotr_decode: the context was encoded with batch-invariant mode %s and the "
               "model now has it %s (cotr_set_batch_invariant): re-encode it", ctx->batch_invariant ? "on" : "off",
               m->batch_invariant ? "on" : "off");
    if (Q == 0) return 0;
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    const long long total = (long long)B * Q;
    const int cap = (int)(total < kDecodeChunkRows ? total : kDecodeChunkRows);
    if (ensure_decode_ws(m, cap) || ensure_sync_ctr(m)) return 1;
    int n_chunks = 0;
    if (Q <= kDecodeChunkRows) {
        const int pairs_per = kDecodeChunkRows / Q;
        n_chunks = (B + pairs_per - 1) / pairs_per;
    } else {
        n_chunks = B * ((Q + kDecodeChunkRows - 1) / kDecodeChunkRows);
    }
    if (dataflow_enabled(m)) {
        const int blocks = std::min(kSyncBlocks - kSyncEncodeBlocks, n_chunks * kSyncChunkBlocks);
        COTR_CHECK_CUDA(cudaMemsetAsync(m->ws.sync_ctr + (size_t)kSyncEncodeBlocks * kSyncBlockInts, 0,
                                        (size_t)blocks * kSyncBlockInts * sizeof(int), s));
    }
    int chunk = 0;
    if (Q <= kDecodeChunkRows) {
        const int pairs_per = kDecodeChunkRows / Q;
        for (int b0 = 0; b0 < B; b0 += pairs_per) {
            const int nb = (B - b0 < pairs_per) ? B - b0 : pairs_per;
            if (decode_chunk(m, ctx, queries + (size_t)b0 * Q * 2, pred + (size_t)b0 * Q * 2, b0, nb, Q, s, chunk++)) return 1;
        }
    } else {
        for (int b = 0; b < B; ++b)
            for (int q0 = 0; q0 < Q; q0 += kDecodeChunkRows) {
                const int nq = (Q - q0 < kDecodeChunkRows) ? Q - q0 : kDecodeChunkRows;
                const size_t off = ((size_t)b * Q + q0) * 2;
                if (decode_chunk(m, ctx, queries + off, pred + off, b, 1, nq, s, chunk++)) return 1;
            }
    }
    m->last_rows = (total <= kDecodeChunkRows) ? (int)total : 0;
    return 0;
}

// ----------------------------------------------------------------------------------------------
// model construction
// ----------------------------------------------------------------------------------------------
int build_model(cotr_model* m, const TensorMap& tm) {
    const std::string body = "backbone.0.body";
    if (make_conv(m, tm, body + ".conv1", body + ".bn1", 64, 3, 7, 7, 2, 3, &m->stem)) return 1;
    struct LayerCfg { const char* name; int n, planes, stride; };
    const LayerCfg layers[3] = {{"layer1", 3, 64, 1}, {"layer2", 4, 128, 2}, {"layer3", 6, 256, 2}};
    int inplanes = 64;
    for (const LayerCfg& L : layers) {
        for (int i = 0; i < L.n; ++i) {
            const std::string p = body + "." + L.name + "." + std::to_string(i);
            Block b;
            const int stride = (i == 0) ? L.stride : 1;
            if (make_conv(m, tm, p + ".conv1", p + ".bn1", L.planes, inplanes, 1, 1, 1, 0, &b.c1)) return 1;
            if (make_conv(m, tm, p + ".conv2", p + ".bn2", L.planes, L.planes, 3, 3, stride, 1, &b.c2)) return 1;
            if (make_conv(m, tm, p + ".conv3", p + ".bn3", L.planes * 4, L.planes, 1, 1, 1, 0, &b.c3)) return 1;
            b.has_ds = (i == 0);
            if (b.has_ds && make_conv(m, tm, p + ".downsample.0", p + ".downsample.1", L.planes * 4, inplanes, 1, 1, stride, 0, &b.ds)) return 1;
            m->blocks.push_back(b);
            inplanes = L.planes * 4;
        }
    }
    {
        const cotr_tensor* w = tm.get("input_proj.weight", {kDModel, 1024, 1, 1});
        const cotr_tensor* b = tm.get("input_proj.bias", {kDModel});
        if (!w || !b) return 1;
        std::vector<float> bv = to_vec(b, kDModel);
        if (make_linear(m, to_vec(w, (size_t)kDModel * 1024), &bv, kDModel, 1024, &m->proj)) return 1;
    }
    if (upload(m, grid_position_table(), &m->pos)) return 1;

    const float qscale = 1.0f / std::sqrt((float)kHeadDim);   // F.multi_head_attention_forward: q * head_dim^-0.5
    const size_t DD = (size_t)kDModel * kDModel;

    auto linear_from = [&](const std::string& prefix, int N, int K, DevLinear* out) -> int {
        const cotr_tensor* w = tm.get(prefix + ".weight", {N, K});
        const cotr_tensor* b = tm.get(prefix + ".bias", {N});
        if (!w || !b) return 1;
        std::vector<float> bv = to_vec(b, N);
        return make_linear(m, to_vec(w, (size_t)N * K), &bv, N, K, out);
    };

    // same, for a layer whose input is a deferred LayerNorm `norm` (weight / bias in the checkpoint)
    auto linear_ln_from = [&](const std::string& prefix, int N, int K, const std::string& norm, DevLinear* out) -> int {
        const cotr_tensor* w = tm.get(prefix + ".weight", {N, K});
        const cotr_tensor* b = tm.get(prefix + ".bias", {N});
        const cotr_tensor* g = tm.get(norm + ".weight", {K});
        const cotr_tensor* be = tm.get(norm + ".bias", {K});
        if (!w || !b || !g || !be) return 1;
        std::vector<float> bv = to_vec(b, N);
        return make_linear_ln(m, to_vec(w, (size_t)N * K), &bv, N, K, g->data, be->data, out);
    };

    // constant position-bias matrices, produced with the fp32 SIMT GEMM once per model
    struct PosBiasJob { std::vector<float> w_masked; std::vector<float> bias; int N; float** dst; };
    std::vector<PosBiasJob> jobs;

    for (int l = 0; l < kEncLayers; ++l) {
        const std::string p = "transformer.encoder.layers." + std::to_string(l);
        EncLayer& e = m->enc[l];
        const cotr_tensor* w = tm.get(p + ".self_attn.in_proj_weight", {3 * kDModel, kDModel});
        const cotr_tensor* b = tm.get(p + ".self_attn.in_proj_bias", {3 * kDModel});
        if (!w || !b) return 1;
        std::vector<float> wv = to_vec(w, 3 * DD), bv = to_vec(b, 3 * kDModel);
        for (size_t i = 0; i < DD; ++i) wv[i] *= qscale;
        for (int i = 0; i < kDModel; ++i) bv[i] *= qscale;
        std::vector<float> wm = wv;                               // value rows see x only, not x + pos
        std::fill(wm.begin() + 2 * DD, wm.end(), 0.f);
        jobs.push_back({wm, bv, 3 * kDModel, &e.add_qkv});
        if (l == 0) {
            if (make_linear(m, wv, nullptr, 3 * kDModel, kDModel, &e.qkv)) return 1;
        } else {
            // the layer input is norm2 of the previous layer, applied on the fly by this GEMM (tensor-core path)
            const std::string prev = "transformer.encoder.layers." + std::to_string(l - 1) + ".norm2";
            const cotr_tensor* g = tm.get(prev + ".weight", {kDModel});
            const cotr_tensor* be = tm.get(prev + ".bias", {kDModel});
            if (!g || !be) return 1;
            std::vector<float> cb;
            if (make_linear_ln(m, wv, nullptr, 3 * kDModel, kDModel, g->data, be->data, &e.qkv, &cb)) return 1;
            std::vector<float> bv_tc = bv;
            for (int i = 0; i < 3 * kDModel; ++i) bv_tc[i] += cb[i];
            jobs.push_back({wm, bv_tc, 3 * kDModel, &e.add_qkv_tc});
        }
        if (linear_from(p + ".self_attn.out_proj", kDModel, kDModel, &e.o)) return 1;
        if (linear_ln_from(p + ".linear1", kFF, kDModel, p + ".norm1", &e.l1)) return 1;
        if (linear_from(p + ".linear2", kDModel, kFF, &e.l2)) return 1;
        if (upload_vec(m, tm, p + ".norm1.weight", kDModel, &e.ln1_g) || upload_vec(m, tm, p + ".norm1.bias", kDModel, &e.ln1_b) ||
            upload_vec(m, tm, p + ".norm2.weight", kDModel, &e.ln2_g) || upload_vec(m, tm, p + ".norm2.bias", kDModel, &e.ln2_b))
            return 1;
    }

    const int kKvN = 2 * kKCols;   // 3072
    std::vector<float> kv_w((size_t)kKvN * kDModel), kv_wm((size_t)kKvN * kDModel, 0.f), kv_b(kKvN);
    std::vector<float> qp_w((size_t)kQpCols * kDModel), qp_b(kQpCols);
    for (int l = 0; l < kDecLayers; ++l) {
        const std::string p = "transformer.decoder.layers." + std::to_string(l);
        DecLayer& d = m->dec[l];
        const cotr_tensor* w = tm.get(p + ".multihead_attn.in_proj_weight", {3 * kDModel, kDModel});
        const cotr_tensor* b = tm.get(p + ".multihead_attn.in_proj_bias", {3 * kDModel});
        if (!w || !b) return 1;
        std::vector<float> wq = to_vec(w, DD);
        for (float& v : wq) v *= qscale;
        if (l == 0) {
            if (make_linear(m, wq, nullptr, kDModel, kDModel, &d.q)) return 1;       // (never run: tgt = 0 in layer 0)
        } else {
            const std::string prev = "transformer.decoder.layers." + std::to_string(l - 1) + ".norm3";
            const cotr_tensor* g = tm.get(prev + ".weight", {kDModel});
            const cotr_tensor* be = tm.get(prev + ".bias", {kDModel});
            if (!g || !be) return 1;
            if (make_linear_ln(m, wq, nullptr, kDModel, kDModel, g->data, be->data, &d.q)) return 1;
        }
        memcpy(qp_w.data() + (size_t)l * DD, wq.data(), DD * sizeof(float));
        for (int i = 0; i < kDModel; ++i) qp_b[l * kDModel + i] = b->data[i] * qscale;
        // K rows then V rows of layer l
        memcpy(kv_w.data() + (size_t)l * 2 * DD, w->data + DD, 2 * DD * sizeof(float));
        memcpy(kv_wm.data() + (size_t)l * 2 * DD, w->data + DD, DD * sizeof(float));   // only K sees pos
        memcpy(kv_b.data() + (size_t)l * 2 * kDModel, b->data + kDModel, 2 * kDModel * sizeof(float));
        if (linear_from(p + ".multihead_attn.out_proj", kDModel, kDModel, &d.o)) return 1;
        if (linear_ln_from(p + ".linear1", kFF, kDModel, p + ".norm2", &d.l1)) return 1;
        if (linear_from(p + ".linear2", kDModel, kFF, &d.l2)) return 1;
        if (upload_vec(m, tm, p + ".norm2.weight", kDModel, &d.ln2_g) || upload_vec(m, tm, p + ".norm2.bias", kDModel, &d.ln2_b) ||
            upload_vec(m, tm, p + ".norm3.weight", kDModel, &d.ln3_g) || upload_vec(m, tm, p + ".norm3.bias", kDModel, &d.ln3_b))
            return 1;
        // decoder.layers.N.norm1.* exists in the checkpoint but transformer.py:185-201 never uses it.
    }
    {
        const std::string last = "transformer.encoder.layers." + std::to_string(kEncLayers - 1) + ".norm2";
        const cotr_tensor* g = tm.get(last + ".weight", {kDModel});
        const cotr_tensor* be = tm.get(last + ".bias", {kDModel});
        if (!g || !be) return 1;
        std::vector<float> cb;
        if (make_linear_ln(m, kv_w, nullptr, kKvN, kDModel, g->data, be->data, &m->kv_all, &cb)) return 1;
        std::vector<float> kv_b_tc = kv_b;
        for (int i = 0; i < kKvN; ++i) kv_b_tc[i] += cb[i];
        jobs.push_back({kv_wm, kv_b_tc, kKvN, &m->add_kv_tc});
    }
    jobs.push_back({kv_wm, kv_b, kKvN, &m->add_kv});
    if (make_linear(m, qp_w, &qp_b, kQpCols, kDModel, &m->qpos_all)) return 1;
    if (upload_vec(m, tm, "transformer.decoder.norm.weight", kDModel, &m->dec_norm_g) ||
        upload_vec(m, tm, "transformer.decoder.norm.bias", kDModel, &m->dec_norm_b))
        return 1;
    if (linear_from("corr_embed.layers.0", kDModel, kDModel, &m->head[0])) return 1;
    if (linear_from("corr_embed.layers.1", kDModel, kDModel, &m->head[1])) return 1;
    if (linear_from("corr_embed.layers.2", 2, kDModel, &m->head[2])) return 1;

    // add matrices: pos [512,256] x Wmasked^T + bias  (fp32 SIMT GEMM on the split16 pos table, fp32 result)
    Split16 pos16 = kNoSplit;
    if (ws_alloc(&pos16, (size_t)kTokens * kDModel)) return 1;
    if (launch_f32_to_split16(m->pos, pos16, (size_t)kTokens * kDModel, 0)) return 1;
    for (PosBiasJob& j : jobs) {
        float *wd = nullptr, *bd = nullptr;
        COTR_CHECK_CUDA(cudaMalloc((void**)&wd, j.w_masked.size() * sizeof(float)));
        COTR_CHECK_CUDA(cudaMalloc((void**)&bd, j.bias.size() * sizeof(float)));
        COTR_CHECK_CUDA(cudaMemcpy(wd, j.w_masked.data(), j.w_masked.size() * sizeof(float), cudaMemcpyHostToDevice));
        COTR_CHECK_CUDA(cudaMemcpy(bd, j.bias.data(), j.bias.size() * sizeof(float), cudaMemcpyHostToDevice));
        if (dev_alloc(m, (void**)j.dst, (size_t)kTokens * j.N * sizeof(float))) return 1;
        GemmParams p = gemm_base(kTokens, j.N, kDModel, cs(pos16), kDModel, wd, nullptr, 1.f, kNoSplit, j.N);
        p.bias = bd;
        if (launch_gemm_simt_raw(p, *j.dst, 0)) return 1;
        COTR_CHECK_CUDA(cudaDeviceSynchronize());
        cudaFree(wd);
        cudaFree(bd);
    }
    ws_free(&pos16);
    if (!m->enc[0].add_qkv_tc) m->enc[0].add_qkv_tc = m->enc[0].add_qkv;     // layer 0 reads the un-normalised input projection
    return 0;
}

}  // namespace
}  // namespace cotr

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
using namespace cotr;

extern "C" {

const char* cotr_last_error(void) { return g_error; }
const char* cotr_version(void) { return "cotr_b200 0.2 (sm_100a)"; }

int cotr_create(int device, const cotr_tensor* tensors, int n_tensors, cotr_model** out) {
    COTR_CHECK(out != nullptr && tensors != nullptr && n_tensors > 0, "cotr_create: bad arguments");
    *out = nullptr;
    int n_dev = 0;
    COTR_CHECK_CUDA(cudaGetDeviceCount(&n_dev));
    COTR_CHECK(device >= 0 && device < n_dev, "cotr_create: CUDA device %d not available (%d visible)", device, n_dev);
    COTR_CHECK_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    COTR_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
    COTR_CHECK(prop.major == 10, "cotr_create: this library is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    TensorMap tm;
    for (int i = 0; i < n_tensors; ++i) {
        COTR_CHECK(tensors[i].name != nullptr, "cotr_create: tensor %d has no name", i);
        tm.m[tensors[i].name] = &tensors[i];
    }
    cotr_model* m = new cotr_model();
    m->device = device;
    g_error[0] = 0;
    if (build_model(m, tm) || cotr_context_create(m, 1, &m->own_ctx) ||
        cudaStreamCreateWithFlags(&m->host_stream, cudaStreamNonBlocking) != cudaSuccess) {
        if (g_error[0] == 0) set_error("cotr_create: stream creation failed");
        cotr_destroy(m);
        return 1;
    }
    *out = m;
    return 0;
}

void cotr_destroy(cotr_model* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    if (m->own_ctx) cotr_context_destroy(m->own_ctx);
    for (void* p : m->allocs) cudaFree(p);
    Workspace& w = m->ws;
    Split16* bufs[] = {&w.canvas, &w.stem, &w.bx, &w.by, &w.bt1, &w.bt2, &w.bds, &w.src, &w.xa, &w.xb, &w.qk, &w.vt, &w.ao, &w.ffh,
                       &w.qpos, &w.qp, &w.t, &w.qb, &w.dao, &w.dh, &w.hs, &w.hd1, &w.hd2, &w.t2, &w.qk2, &w.vt2};
    for (Split16* b : bufs) ws_free(b);
    if (w.sync_ctr) cudaFree(w.sync_ctr);
    if (w.kvimg) cudaFree(w.kvimg);
    if (w.kvimg2) cudaFree(w.kvimg2);
    float** fbufs[] = {&w.ln_tmp, &w.dln_tmp, &w.img_stage, &w.q_stage, &w.pred_stage,
                       reinterpret_cast<float**>(&w.enc_st_a), reinterpret_cast<float**>(&w.enc_st_b),
                       reinterpret_cast<float**>(&w.dec_st_a), reinterpret_cast<float**>(&w.dec_st_b)};
    for (float** b : fbufs) ws_free_f32(b);
    if (m->host_stream) cudaStreamDestroy(m->host_stream);
    for (auto& kv : m->graphs) cudaGraphExecDestroy(kv.second);
    preprocessor_destroy(m->pre);
    flow_merger_destroy(m->merger);
    for (cudaEvent_t e : m->prof_events) cudaEventDestroy(e);
    if (m->order_event) cudaEventDestroy(m->order_event);
    delete m;
}

int cotr_context_create(cotr_model* m, int max_pairs, cotr_context** out) {
    COTR_CHECK(m && out && max_pairs >= 1, "cotr_context_create: bad arguments");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    cotr_context* c = new cotr_context();
    c->model = m;
    c->max_pairs = max_pairs;
    const size_t img_bytes = (size_t)max_pairs * kDecLayers * kHeads * kAttnHeadImgBytes;
    if (ws_alloc(&c->k, (size_t)max_pairs * kTokens * kKCols) || ws_alloc(&c->vt, (size_t)max_pairs * kDecLayers * kVtLayer) ||
        cudaMalloc((void**)&c->img, img_bytes) != cudaSuccess || cudaMemset(c->img, 0, img_bytes) != cudaSuccess) {
        set_error("cotr_context_create: out of device memory for %d pairs", max_pairs);
        cotr_context_destroy(c);
        return 1;
    }
    *out = c;
    return 0;
}

void cotr_context_destroy(cotr_context* c) {
    if (!c) return;
    ws_free(&c->k);
    ws_free(&c->vt);
    if (c->img) cudaFree(c->img);
    delete c;
}

int cotr_encode_context(cotr_model* m, const float* img_dev, int B, cotr_context* ctx, void* cuda_stream) {
    COTR_CHECK(m && img_dev, "cotr_encode_context: null argument");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    CallOrder order(m, (cudaStream_t)cuda_stream);
    m->launches = 0;
    return encode_impl(m, img_dev, B, ctx, (cudaStream_t)cuda_stream);
}

int cotr_decode(cotr_model* m, const cotr_context* ctx, const float* queries_dev, int B, int Q, float* pred_dev, void* cuda_stream) {
    COTR_CHECK(m && (Q == 0 || (queries_dev && pred_dev)), "cotr_decode: null argument");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    CallOrder order(m, (cudaStream_t)cuda_stream);
    m->launches = 0;
    return decode_impl(m, ctx, queries_dev, B, Q, pred_dev, (cudaStream_t)cuda_stream);
}

namespace {

int ensure_stage(cotr_model* m, int B, int Q) {
    Workspace& w = m->ws;
    const size_t img_elems = (size_t)B * 3 * COTR_CANVAS_H * COTR_CANVAS_W;
    const size_t q_elems = (size_t)B * Q * 2;
    if (img_elems > w.img_stage_elems) {
        COTR_CHECK_CUDA(cudaDeviceSynchronize());
        drop_graphs(m);
        ws_free_f32(&w.img_stage);
        if (ws_alloc_f32(&w.img_stage, img_elems)) return 1;
        w.img_stage_elems = img_elems;
    }
    if (q_elems > w.q_stage_elems) {
        COTR_CHECK_CUDA(cudaDeviceSynchronize());
        drop_graphs(m);
        ws_free_f32(&w.q_stage); ws_free_f32(&w.pred_stage);
        if (ws_alloc_f32(&w.q_stage, q_elems ? q_elems : 2) || ws_alloc_f32(&w.pred_stage, q_elems ? q_elems : 2)) return 1;
        w.q_stage_elems = q_elems;
    }
    return 0;
}

int forward_eager(cotr_model* m, const float* img, const float* queries, int B, int Q, float* pred, cudaStream_t s) {
    if (m->own_ctx->max_pairs < B) {
        COTR_CHECK_CUDA(cudaDeviceSynchronize());
        drop_graphs(m);
        cotr_context_destroy(m->own_ctx);
        m->own_ctx = nullptr;
        if (cotr_context_create(m, B, &m->own_ctx)) return 1;
    }
    m->launches = 0;
    if (encode_impl(m, img, B, m->own_ctx, s)) return 1;
    return decode_impl(m, m->own_ctx, queries, B, Q, pred, s);
}

// Forward on the staging buffers (img_stage, q_stage -> pred_stage): graph replay when a graph exists for the shape.
int forward_staged(cotr_model* m, int B, int Q, cudaStream_t s) {
    Workspace& w = m->ws;
    const bool graphable = m->graph_mode && !m->prof_on && (g_tc_timestamps == nullptr || (g_tc_variant & (1 << 17)));
    const long long key = ((long long)B << 32) | (unsigned)Q;
    if (graphable) {
        auto it = m->graphs.find(key);
        if (it != m->graphs.end()) {
            COTR_CHECK_CUDA(cudaGraphLaunch(it->second, s));
            m->launches = m->graph_launches[key];
            return 0;
        }
        if (m->shapes_seen.count(key) && m->graphs.size() < 256) {
            // second call with this shape: workspace, contexts and kernel attributes are in place -> capture
            cudaGraph_t graph = nullptr;
            // the legacy default stream (what torch hands over by default) cannot be captured: record on ours,
            // the resulting graph is launched on the caller's stream either way
            cudaStream_t cs = (s == nullptr || s == cudaStreamLegacy || s == cudaStreamPerThread) ? m->host_stream : s;
            COTR_CHECK_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            const int rc = forward_eager(m, w.img_stage, w.q_stage, B, Q, w.pred_stage, cs);
            const cudaError_t e = cudaStreamEndCapture(cs, &graph);
            if (rc || e != cudaSuccess || graph == nullptr) {
                if (graph) cudaGraphDestroy(graph);
                if (!rc) set_error("cotr_forward: stream capture failed: %s", cudaGetErrorString(e));
                return 1;
            }
            cudaGraphExec_t exec = nullptr;
            const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            COTR_CHECK(ei == cudaSuccess, "cotr_forward: cudaGraphInstantiate failed: %s", cudaGetErrorString(ei));
            m->graphs[key] = exec;
            m->graph_launches[key] = m->launches;
            COTR_CHECK_CUDA(cudaGraphLaunch(exec, s));
            return 0;
        }
        m->shapes_seen.insert(key);
    }
    return forward_eager(m, w.img_stage, w.q_stage, B, Q, w.pred_stage, s);
}

}  // namespace

int cotr_forward(cotr_model* m, const float* img_dev, const float* queries_dev, int B, int Q, float* pred_dev, void* cuda_stream) {
    COTR_CHECK(m && img_dev && (Q == 0 || (queries_dev && pred_dev)), "cotr_forward: null argument");
    COTR_CHECK(B >= 1 && Q >= 0, "cotr_forward: B must be >= 1 and Q >= 0");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    CallOrder order(m, s);
    const bool graphable = m->graph_mode && !m->prof_on && (g_tc_timestamps == nullptr || (g_tc_variant & (1 << 17))) && Q > 0;
    if (!graphable) return forward_eager(m, img_dev, queries_dev, B, Q, pred_dev, s);
    // graph replay needs fixed addresses: go through the staging buffers (two small device-to-device copies in, one out)
    if (ensure_stage(m, B, Q)) return 1;
    Workspace& w = m->ws;
    const size_t img_bytes = (size_t)B * 3 * COTR_CANVAS_H * COTR_CANVAS_W * sizeof(float), q_bytes = (size_t)B * Q * 2 * sizeof(float);
    COTR_CHECK_CUDA(cudaMemcpyAsync(w.img_stage, img_dev, img_bytes, cudaMemcpyDeviceToDevice, s));
    COTR_CHECK_CUDA(cudaMemcpyAsync(w.q_stage, queries_dev, q_bytes, cudaMemcpyDeviceToDevice, s));
    if (forward_staged(m, B, Q, s)) return 1;
    COTR_CHECK_CUDA(cudaMemcpyAsync(pred_dev, w.pred_stage, q_bytes, cudaMemcpyDeviceToDevice, s));
    return 0;
}

int cotr_forward_host(cotr_model* m, const float* img_host, const float* queries_host, int B, int Q, float* pred_host) {
    COTR_CHECK(m && img_host && (Q == 0 || (queries_host && pred_host)), "cotr_forward_host: null argument");
    COTR_CHECK(B >= 1 && Q >= 0, "cotr_forward_host: B must be >= 1 and Q >= 0");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    if (ensure_stage(m, B, Q)) return 1;
    Workspace& w = m->ws;
    const size_t img_bytes = (size_t)B * 3 * COTR_CANVAS_H * COTR_CANVAS_W * sizeof(float), q_bytes = (size_t)B * Q * 2 * sizeof(float);
    cudaStream_t s = m->host_stream;
    CallOrder order(m, s);
    COTR_CHECK_CUDA(cudaMemcpyAsync(w.img_stage, img_host, img_bytes, cudaMemcpyHostToDevice, s));
    if (q_bytes) COTR_CHECK_CUDA(cudaMemcpyAsync(w.q_stage, queries_host, q_bytes, cudaMemcpyHostToDevice, s));
    if (Q > 0) {
        if (forward_staged(m, B, Q, s)) return 1;
        COTR_CHECK_CUDA(cudaMemcpyAsync(pred_host, w.pred_stage, q_bytes, cudaMemcpyDeviceToHost, s));
    }
    COTR_CHECK_CUDA(cudaStreamSynchronize(s));
    return 0;
}

int cotr_preprocess(cotr_model* m, const uint8_t* img_from_dev, int h_from, int w_from, const uint8_t* img_to_dev, int h_to,
                    int w_to, const int32_t* rects_host, int n, float* canvas_dev, void* cuda_stream) {
    COTR_CHECK(m != nullptr, "cotr_preprocess: null model");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    if (!m->pre) m->pre = preprocessor_create();
    CallOrder order(m, (cudaStream_t)cuda_stream);
    return preprocess_launch(m->pre, img_from_dev, h_from, w_from, img_to_dev, h_to, w_to, rects_host, n, canvas_dev,
                             (cudaStream_t)cuda_stream);
}

int cotr_dense_postprocess(cotr_model* m, const float* pred_dev, int n, float* out_dev, void* cuda_stream) {
    COTR_CHECK(m != nullptr, "cotr_dense_postprocess: null model");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    return dense_post_launch(pred_dev, out_dev, n, (cudaStream_t)cuda_stream);
}

int cotr_flow_tile_merge(cotr_model* m, const float* tile_dev, int pitch_floats, const double* affine_host, int px, int py, int pw, int ph,
                         int ow, int oh, float* flow_dev, float* conf_dev, int first, void* cuda_stream) {
    COTR_CHECK(m != nullptr, "cotr_flow_tile_merge: null model");
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    if (!m->merger) m->merger = flow_merger_create();
    CallOrder order(m, (cudaStream_t)cuda_stream);
    return flow_tile_merge_launch(m->merger, tile_dev, pitch_floats, affine_host, px, py, pw, ph, ow, oh, flow_dev, conf_dev, first,
                                  (cudaStream_t)cuda_stream);
}

int cotr_group_tasks(int device, const double* pts_dev, const double* box_dev, int n, int batch_size, int max_load, int32_t* squad_dev,
                     int32_t* rank_dev, int32_t* n_squads_dev, void* cuda_stream) {
    COTR_CHECK_CUDA(cudaSetDevice(device));
    return group_tasks_launch(pts_dev, box_dev, n, batch_size, max_load, squad_dev, rank_dev, n_squads_dev, (cudaStream_t)cuda_stream);
}

int cotr_rasterize_triangles(int device, const float* tris_dev, int n_tri, int H, int W, float* out_dev, void* cuda_stream) {
    COTR_CHECK_CUDA(cudaSetDevice(device));
    return rasterize_triangles_launch(tris_dev, n_tri, H, W, out_dev, (cudaStream_t)cuda_stream);
}

int cotr_set_graph_mode(cotr_model* m, int enabled) {
    COTR_CHECK(m != nullptr, "cotr_set_graph_mode: null model");
    m->graph_mode = enabled != 0;
    return 0;
}

size_t cotr_workspace_bytes(int B, int Q) {
    if (B < 1 || Q < 0) return 0;
    const long long total = (long long)B * Q;
    const int rows = (int)(total < kDecodeChunkRows ? total : kDecodeChunkRows);
    return (encode_ws_elems(B) + decode_ws_elems(rows)) * sizeof(float);
}

int cotr_last_launch_count(const cotr_model* m) { return m ? m->launches : -1; }

int cotr_profile_begin(cotr_model* m, int max_records) {
    COTR_CHECK(m && max_records > 0, "cotr_profile_begin: bad arguments");
    m->prof_records.clear();
    m->prof_records.reserve(max_records);
    m->prof_max = max_records;
    m->prof_on = true;
    return 0;
}

int cotr_profile_end(cotr_model* m, cotr_launch_record* out, int max_records) {
    COTR_CHECK(m && out, "cotr_profile_end: bad arguments");
    m->prof_on = false;
    COTR_CHECK_CUDA(cudaSetDevice(m->device));
    COTR_CHECK_CUDA(cudaDeviceSynchronize());
    int n = (int)m->prof_records.size();
    if (n > max_records) n = max_records;
    for (int i = 0; i < n; ++i) {
        float ms = 0.f;
        COTR_CHECK_CUDA(cudaEventElapsedTime(&ms, m->prof_events[2 * i], m->prof_events[2 * i + 1]));
        m->prof_records[i].ms = ms;
        out[i] = m->prof_records[i];
    }
    return -n - 1;     // see header: success is encoded as -(count + 1)
}

namespace {
struct TmpSplitDbg {
    Split16 t = kNoSplit;
    ~TmpSplitDbg() { ws_free(&t); }
};
}  // namespace

int64_t cotr_debug_read(cotr_model* m, const char* name, float* out_host, int64_t max_elems) {
    if (!m || !name || !out_host) return -1;
    cudaSetDevice(m->device);
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    CSplit16 src{nullptr, nullptr};
    const float* src_f32 = nullptr;
    int64_t n = 0;
    const std::string s(name);
    if (s == "feat") { src = cs(m->last_feat); n = (int64_t)m->last_pairs * 2 * 16 * 16 * 1024; }
    else if (s == "src") { src = cs(m->ws.src); n = (int64_t)m->last_pairs * kTokens * kDModel; }
    else if (s == "mem") { src = cs(m->last_mem); n = (int64_t)m->last_pairs * kTokens * kDModel; }
    TmpSplitDbg mem_ln;
    if (s == "mem" && m->last_mem_pre_ln && src.hi && n > 0) {
        // tensor-core path: the encoder output exists only before its last (deferred) LayerNorm - apply it here
        const EncLayer& e = m->enc[kEncLayers - 1];
        if (ws_alloc(&mem_ln.t, (size_t)n) || launch_layernorm(src, e.ln2_g, e.ln2_b, mem_ln.t, (int)(n / kDModel), 0) ||
            cudaDeviceSynchronize() != cudaSuccess)
            return -1;
        src = cs(mem_ln.t);
    }
    else if (s == "hs") { src = cs(m->ws.hs); n = (int64_t)m->last_rows * kDModel; }
    else if (s == "pos") { src_f32 = m->pos; n = (int64_t)kTokens * kDModel; }
    // bring-up: raw workspace buffers of the last forward (tokens = pairs * 512, rows = the decoder rows of the last chunk)
    else if (s == "ws.xa") { src = cs(m->ws.xa); n = (int64_t)m->last_pairs * kTokens * kDModel; }
    else if (s == "ws.xb") { src = cs(m->ws.xb); n = (int64_t)m->last_pairs * kTokens * kDModel; }
    else if (s == "ws.ao") { src = cs(m->ws.ao); n = (int64_t)m->last_pairs * kTokens * kDModel; }
    else if (s == "ws.qk") { src = cs(m->ws.qk); n = (int64_t)m->last_pairs * kTokens * 2 * kDModel; }
    else if (s == "ws.ffh") { src = cs(m->ws.ffh); n = (int64_t)m->last_pairs * kTokens * kFF; }
    else if (s == "ws.t") { src = cs(m->ws.t); n = (int64_t)m->last_rows * kDModel; }
    else if (s == "ws.t2") { src = cs(m->ws.t2); n = (int64_t)m->last_rows * kDModel; }
    else if (s == "ws.dao") { src = cs(m->ws.dao); n = (int64_t)m->last_rows * kDModel; }
    else if (s == "ws.st_a") { src_f32 = reinterpret_cast<const float*>(m->ws.enc_st_a); n = (int64_t)m->last_pairs * kTokens * 32; }
    else if (s == "ws.st_b") { src_f32 = reinterpret_cast<const float*>(m->ws.enc_st_b); n = (int64_t)m->last_pairs * kTokens * 32; }
    if ((!src.hi && !src_f32) || n <= 0 || n > max_elems) return -1;
    float* tmp = nullptr;
    if (!src_f32) {
        if (cudaMalloc((void**)&tmp, n * sizeof(float)) != cudaSuccess) return -1;
        if (launch_split16_to_f32(src, tmp, (size_t)n, 0) || cudaDeviceSynchronize() != cudaSuccess) { cudaFree(tmp); return -1; }
        src_f32 = tmp;
    }
    const cudaError_t e = cudaMemcpy(out_host, src_f32, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (tmp) cudaFree(tmp);
    return e == cudaSuccess ? n : -1;
}

int cotr_set_gemm_path(cotr_model* m, int path) {
    COTR_CHECK(m && (path == 0 || path == 1), "cotr_set_gemm_path: path must be 0 (tcgen05) or 1 (fp32 SIMT)");
    if (m->gemm_path != path) {          // captured graphs embed the kernels of the old path
        cudaSetDevice(m->device);
        cudaDeviceSynchronize();
        drop_graphs(m);
        m->shapes_seen.clear();
    }
    m->gemm_path = path;
    return 0;
}

int cotr_set_batch_invariant(cotr_model* m, int enabled) {
    COTR_CHECK(m != nullptr, "cotr_set_batch_invariant: null model");
    const bool on = enabled != 0;
    if (m->batch_invariant != on) {      // a graph captured under one policy must never replay under the other
        cudaSetDevice(m->device);
        cudaDeviceSynchronize();
        drop_graphs(m);
        m->shapes_seen.clear();
    }
    m->batch_invariant = on;
    return 0;
}

void cotr_debug_set_variant(int variant) { g_tc_variant = variant; g_use_pdl = (variant & 256) ? 0 : 1; }
void cotr_debug_set_timestamps(void* dev_buffer) {
    g_tc_timestamps = reinterpret_cast<long long*>(dev_buffer);
    g_tc_trace_idx = 0;
}

// ---- kernel-level test hooks: fp32 device tensors in / out, converted to split16 around the kernel under test -------
namespace {
struct TmpSplit {
    Split16 t = kNoSplit;
    ~TmpSplit() { ws_free(&t); }
    int from_f32(const float* src, size_t n) {
        const size_t padded = (n + 7) & ~(size_t)7;
        if (ws_alloc(&t, padded)) return 1;
        return launch_f32_to_split16(src, t, n, 0);
    }
    int empty(size_t n) { return ws_alloc(&t, (n + 7) & ~(size_t)7); }
};
}  // namespace

int cotr_test_gemm(const cotr_test_gemm_desc* d, const float* A_dev, const float* w_host, const float* bias_dev,
                   const float* addmat_dev, const float* residual_dev, const float* ln_gamma_dev,
                   const float* ln_beta_dev, float* out_dev, float* part_out_dev) {
    COTR_CHECK(d && A_dev && w_host && out_dev, "cotr_test_gemm: null argument");
    COTR_CHECK(d->ldc == d->N, "cotr_test_gemm: ldc must equal N");
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = d->M; p.N = d->N; p.K = d->K;
    p.a_mode = d->a_mode; p.lda = d->lda;
    p.H = d->H; p.W = d->W; p.C = d->C; p.OH = d->OH; p.OW = d->OW;
    p.KH = d->KH; p.KW = d->KW; p.stride = d->stride; p.pad = d->pad;
    p.bias = bias_dev; p.addmat = addmat_dev; p.add_period = d->add_period > 0 ? d->add_period : 1; p.ld_add = d->ld_add;
    p.ldr = d->ldr; p.relu = d->relu;
    const bool dln = d->a_ln != 0 || d->res_ln != 0;
    COTR_CHECK(!dln || (d->path == 0 && ln_gamma_dev && ln_beta_dev), "cotr_test_gemm: deferred LayerNorm needs path 0 and gamma / beta");
    if (!dln) { p.ln_gamma = ln_gamma_dev; p.ln_beta = ln_beta_dev; }
    p.ldc = d->ldc;
    TmpSplit a16, res16, out16;
    int K = d->K;
    std::vector<float> w_stem;
    if (d->a_mode == A_STEM_NHWC4) {
        // the stem as the model runs it: A_dev is the fp32 (B,3,256,512) canvas, w_host [N][7][7][3]; the hook builds the
        // bordered NHWC4 operand and the matching weight order (K = 224)
        COTR_CHECK(d->K == 147 && d->OH == 128 && d->OW == 128 && d->M % (128 * 128) == 0, "cotr_test_gemm: the stem mode expects K = 147, 128 x 128 outputs per image");
        const int n_img = d->M / (128 * 128);
        if (a16.empty((size_t)n_img * kStemCanvasElems)) return 1;
        COTR_CHECK_CUDA(cudaMemset(a16.t.hi, 0, (size_t)n_img * kStemCanvasElems * 2 * sizeof(__half)));
        if (launch_stem_canvas(A_dev, a16.t, n_img, 0)) return 1;
        p.a = cs(a16.t);
        w_stem = stem_weight_order(std::vector<float>(w_host, w_host + (size_t)d->N * 147), d->N);
        w_host = w_stem.data();
        K = kStemK; p.K = K; p.KW = 8; p.C = 4;
    } else {
        COTR_CHECK(d->a_elems > 0, "cotr_test_gemm: a_elems missing");
        if (a16.from_f32(A_dev, (size_t)d->a_elems)) return 1;
        p.a = cs(a16.t);
    }
    if (residual_dev) {
        if (res16.from_f32(residual_dev, (size_t)d->M * d->ldr)) return 1;
        p.res = cs(res16.t);
    }
    const bool f32_out = (d->N & 15) != 0;
    if (f32_out) p.out_f32 = out_dev;
    else { if (out16.empty((size_t)d->M * d->N)) return 1; p.out = out16.t; }
    float* wd = nullptr;
    void* wtc = nullptr;
    float* scratch = nullptr;
    const size_t wn = (size_t)d->N * K;
    COTR_CHECK_CUDA(cudaMalloc((void**)&wd, wn * sizeof(float)));
    COTR_CHECK_CUDA(cudaMemcpy(wd, w_host, wn * sizeof(float), cudaMemcpyHostToDevice));
    // deferred LayerNorm of A: the packed weights carry gamma, column sums and beta W^T + bias go to the epilogue
    std::vector<float> w_fold;
    float *cs_dev = nullptr, *cb_dev = nullptr;
    float2 *stats_dev = nullptr, *res_stats_dev = nullptr;
    if (d->a_ln) {
        COTR_CHECK(d->K == 256 && d->a_mode == A_ROWMAJOR, "cotr_test_gemm: a_ln needs K = 256, row-major A");
        std::vector<float> g(d->K), be(d->K), bias_h(d->N, 0.f), cs(d->N), cb(d->N);
        COTR_CHECK_CUDA(cudaMemcpy(g.data(), ln_gamma_dev, d->K * sizeof(float), cudaMemcpyDeviceToHost));
        COTR_CHECK_CUDA(cudaMemcpy(be.data(), ln_beta_dev, d->K * sizeof(float), cudaMemcpyDeviceToHost));
        if (bias_dev) COTR_CHECK_CUDA(cudaMemcpy(bias_h.data(), bias_dev, d->N * sizeof(float), cudaMemcpyDeviceToHost));
        w_fold.resize(wn);
        for (int n = 0; n < d->N; ++n) {
            double sum = 0.0, c = bias_h[n];
            for (int k = 0; k < d->K; ++k) {
                const float v = w_host[(size_t)n * d->K + k] * g[k];
                w_fold[(size_t)n * d->K + k] = v;
                sum += v;
                c += (double)w_host[(size_t)n * d->K + k] * be[k];
            }
            cs[n] = (float)sum; cb[n] = (float)c;
        }
        COTR_CHECK_CUDA(cudaMalloc((void**)&cs_dev, d->N * sizeof(float)));
        COTR_CHECK_CUDA(cudaMalloc((void**)&cb_dev, d->N * sizeof(float)));
        COTR_CHECK_CUDA(cudaMemcpy(cs_dev, cs.data(), d->N * sizeof(float), cudaMemcpyHostToDevice));
        COTR_CHECK_CUDA(cudaMemcpy(cb_dev, cb.data(), d->N * sizeof(float), cudaMemcpyHostToDevice));
        p.a_ln_cs = cs_dev; p.bias = cb_dev;
        w_host = w_fold.data();
    }
    if (d->a_ln) {
        COTR_CHECK_CUDA(cudaMalloc((void**)&stats_dev, (size_t)d->M * 16 * sizeof(float2)));
        if (launch_ln_partials(p.a, stats_dev, d->M, 0)) return 1;
        p.a_ln_part = stats_dev;
    }
    if (d->res_ln) {
        COTR_CHECK(residual_dev && d->ldr == 256 && d->N == 256, "cotr_test_gemm: res_ln needs a [M,256] residual");
        COTR_CHECK_CUDA(cudaMalloc((void**)&res_stats_dev, (size_t)d->M * 16 * sizeof(float2)));
        if (launch_ln_partials(p.res, res_stats_dev, d->M, 0)) return 1;
        p.res_ln_part = res_stats_dev; p.res_ln_gamma = ln_gamma_dev; p.res_ln_beta = ln_beta_dev;
    }
    if (d->emit_part) {
        COTR_CHECK(d->path == 0 && part_out_dev != nullptr && d->N == 256, "cotr_test_gemm: emit_part needs path 0, N = 256 and an output buffer");
        p.ln_part_out = reinterpret_cast<float2*>(part_out_dev);
    }
    const size_t tcb = tc_weight_bytes(d->N, K);
    std::vector<uint8_t> img(tcb);
    p.acc_scale = tc_pack_weight(w_host, d->N, K, img.data());
    COTR_CHECK_CUDA(cudaMalloc(&wtc, tcb));
    COTR_CHECK_CUDA(cudaMemcpy(wtc, img.data(), tcb, cudaMemcpyHostToDevice));
    p.Wt = wd; p.Wtc = wtc;
    int rc;
    if (d->path == 0) {
        rc = launch_gemm_tc(p, 0);
    } else {
        const float* g = p.ln_gamma; const float* b = p.ln_beta;
        p.ln_gamma = nullptr; p.ln_beta = nullptr;
        if (g) {
            rc = cudaMalloc((void**)&scratch, (size_t)d->M * d->N * sizeof(float)) != cudaSuccess;
            if (!rc) rc = launch_gemm_simt_raw(p, scratch, 0);
            if (!rc) rc = launch_layernorm_f32(scratch, g, b, p.out, p.M, 0);
        } else {
            rc = launch_gemm_simt(p, 0);
        }
    }
    if (!rc && !f32_out) rc = launch_split16_to_f32(cs(out16.t), out_dev, (size_t)d->M * d->N, 0);
    cudaError_t e = cudaDeviceSynchronize();
    cudaFree(wd);
    cudaFree(wtc);
    if (scratch) cudaFree(scratch);
    if (cs_dev) cudaFree(cs_dev);
    if (cb_dev) cudaFree(cb_dev);
    if (stats_dev) cudaFree(stats_dev);
    if (res_stats_dev) cudaFree(res_stats_dev);
    if (rc) return rc;
    COTR_CHECK(e == cudaSuccess, "cotr_test_gemm: kernel failed: %s", cudaGetErrorString(e));
    return 0;
}

// q (npairs*nq,256), k / v (npairs*512,256) fp32 row-major; v is transposed into the [pair][256][512] layout first.
int cotr_test_attention(int path, const float* q_dev, const float* k_dev, const float* v_dev, float* out_dev,
                        int nq, int npairs) {
    COTR_CHECK(q_dev && k_dev && v_dev && out_dev, "cotr_test_attention: null argument");
    COTR_CHECK(path >= 0 && path <= 2, "cotr_test_attention: path must be 0, 1 or 2");
    TmpSplit q16, k16, vt16, o16;
    const size_t qn = (size_t)npairs * nq * kDModel, kn = (size_t)npairs * kTokens * kDModel;
    if (q16.from_f32(q_dev, qn) || k16.from_f32(k_dev, kn) || vt16.empty(kn) || o16.empty(qn)) return 1;
    {   // transpose V with an identity "GEMM": vt = (V * I^T) stored through the transposed-block epilogue
        std::vector<float> eye((size_t)kDModel * kDModel, 0.f);
        for (int i = 0; i < kDModel; ++i) eye[(size_t)i * kDModel + i] = 1.f;
        float* ed = nullptr;
        COTR_CHECK_CUDA(cudaMalloc((void**)&ed, eye.size() * sizeof(float)));
        COTR_CHECK_CUDA(cudaMemcpy(ed, eye.data(), eye.size() * sizeof(float), cudaMemcpyHostToDevice));
        TmpSplit v16;
        if (v16.from_f32(v_dev, kn)) { cudaFree(ed); return 1; }
        GemmParams p;
        memset(&p, 0, sizeof(p));
        p.M = npairs * kTokens; p.N = kDModel; p.K = kDModel;
        p.a = cs(v16.t); p.a_mode = A_ROWMAJOR; p.lda = kDModel;
        p.Wt = ed; p.acc_scale = 1.f; p.add_period = 1;
        p.remap = 1; p.blk_map[0] = -1; p.vt = vt16.t; p.n_vt = 1; p.ldc = kDModel;
        const int rc = launch_gemm_simt(p, 0);
        cudaDeviceSynchronize();
        cudaFree(ed);
        if (rc) return rc;
    }
    AttnParams a{};
    a.q = cs(q16.t); a.ldq = kDModel; a.k = cs(k16.t); a.ldk = kDModel;
    a.vt = cs(vt16.t); a.vt_pair_stride = kVtLayer;
    a.out = o16.t; a.ldo = kDModel; a.nq = nq; a.npairs = npairs; a.pair0 = 0;
    if (path == 2) a.nq_sched = kHeadlineQueries;      // tcgen05 whatever nq (as in the batch-invariant schedule)
    int rc = path == 1 ? launch_attention_simt(a, 0) : launch_attention_tc(a, 0);
    if (!rc) rc = launch_split16_to_f32(cs(o16.t), out_dev, qn, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (rc) return rc;
    COTR_CHECK(e == cudaSuccess, "cotr_test_attention: kernel failed: %s", cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
