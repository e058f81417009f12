/*
 * cotr_b200 - C ABI of the B200-native COTR correspondence-inference hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The
 * reference (ubc-vision/COTR) is pure Python, so "what its FFI would bind" is
 * the L4->L3 call of the inference loop and the model construction protocol:
 *
 *   cotr_create            <- COTR/models/__init__.py:9-10  build_model(args)  +
 *                             COTR/utils/utils.py:164-193   safe_load_weights(model, state_dict)
 *                             (tensors are named by the reference's state_dict keys, SURVEY.md app. C)
 *   cotr_forward           <- COTR/models/cotr_model.py:26-40  COTR.forward(samples, queries)
 *                             as called by sparse_engine.py:52,281 and inference_helper.py:126,134,197-198
 *   cotr_encode_context    <- the query-independent part of COTR.forward: backbone.py:79-92,
 *                             cotr_model.py:37 (input_proj), transformer.py:55 (encoder) and the K/V
 *                             in-projections inside transformer.py:192-195
 *   cotr_decode            <- the per-query part: cotr_model.py:34-36 (query_proj), transformer.py:56-57
 *                             (decoder), cotr_model.py:38-39 (corr_embed, last level only)
 *   cotr_forward_host      <- the same call with HOST buffers, i.e. including the .to(device) /
 *                             .cpu() copies of sparse_engine.py:50-53
 *
 * All device pointers are fp32, contiguous.  Every call returns 0 on success; on failure it returns
 * non-zero and cotr_last_error() describes the problem (the Python wrapper raises the exception type
 * the reference would: AssertionError for a wrong canvas size, RuntimeError otherwise).
 *
 * Threading: one caller thread per model handle; one handle per device.  A model's workspace, staging buffers and
 * internal context are shared by all its entry points: calls may use different streams (each call makes its stream
 * wait for the previous call's work through an internal event), but they execute one after the other, and a
 * cotr_context must not be re-encoded while a decode on it is still in flight on another stream.  No hidden host syncs in the
 * device-pointer calls (work is enqueued on the caller's stream) except when the internal workspace has
 * to grow (first call / larger B or Q than seen before).
 */
#ifndef COTR_B200_H_
#define COTR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COTR_CANVAS_H 256          /* COTR/utils/constants.py:2  MAX_SIZE            */
#define COTR_CANVAS_W 512          /* backbone.py:80             2 * MAX_SIZE        */
#define COTR_CONTEXT_TOKENS 512    /* 16 x 32 layer3 grid                            */
#define COTR_D_MODEL 256

typedef struct cotr_model cotr_model;       /* opaque: packed weights + workspace, bound to one device */
typedef struct cotr_context cotr_context;   /* opaque: per-pair decoder K/V cache (6 layers)           */

/* One named host tensor of the reference checkpoint (fp32, C-contiguous). */
typedef struct cotr_tensor {
    const char* name;        /* reference state_dict key, e.g. "transformer.encoder.layers.0.linear1.weight" */
    const float* data;       /* host pointer                                                                  */
    int32_t ndim;
    int64_t shape[4];
} cotr_tensor;

/* Build a model on CUDA device `device` from the 381 tensors of the reference state_dict
 * (FrozenBN buffers included; the unused decoder norm1.* entries may be present and are ignored).
 * Folds FrozenBN (backbone.py:46-56) into the conv kernels, repacks everything into kernel-native
 * layouts and uploads.  Fails if a required key is missing or has the wrong shape. */
int cotr_create(int device, const cotr_tensor* tensors, int n_tensors, cotr_model** out);
void cotr_destroy(cotr_model* m);

/* A context holds the K/V projections of all 6 decoder layers for up to `max_pairs` image pairs. */
int cotr_context_create(cotr_model* m, int max_pairs, cotr_context** out);
void cotr_context_destroy(cotr_context* c);

/* img_dev: (B,3,256,512) NCHW fp32, ImageNet-normalised, the two 256x256 images side by side. */
int cotr_encode_context(cotr_model* m, const float* img_dev, int B, cotr_context* ctx, void* cuda_stream);

/* queries_dev: (B,Q,2) fp32 (x over the 512-wide canvas, y over 256, both normalised to [0,1]);
 * pred_dev: (B,Q,2) fp32.  B must equal the B of the last cotr_encode_context on `ctx`. */
int cotr_decode(cotr_model* m, const cotr_context* ctx, const float* queries_dev, int B, int Q,
                float* pred_dev, void* cuda_stream);

/* cotr_encode_context + cotr_decode on an internal context. */
int cotr_forward(cotr_model* m, const float* img_dev, const float* queries_dev, int B, int Q,
                 float* pred_dev, void* cuda_stream);

/* Same with host buffers (pinned or pageable): H2D, forward, D2H, stream synchronised on return. */
int cotr_forward_host(cotr_model* m, const float* img_host, const float* queries_host, int B, int Q,
                      float* pred_host);

/* Device-side replacement of the host work of RefinementTask.get_task (COTR/inference/refinement_task.py:105-120) and
 * of the canvas construction in inference_helper.py:108-113: for each of the n tasks crop a square patch out of the
 * "from" image and one out of the "to" image (uint8 HWC, 3 channels, DEVICE memory, uploaded once per engine call),
 * resize both to 256x256 with Pillow's antialiased bilinear filter (bit-exact), put them side by side and apply
 * to_tensor + normalize(mean (0.485,0.456,0.406), std (0.229,0.224,0.225)).  rects_host: n x 6 int32 HOST array
 * [x_from, y_from, size_from, x_to, y_to, size_to]; canvas_dev: (n,3,256,512) fp32 DEVICE output. */
int cotr_preprocess(cotr_model* m, const uint8_t* img_from_dev, int h_from, int w_from, const uint8_t* img_to_dev, int h_to,
                    int w_to, const int32_t* rects_host, int n, float* canvas_dev, void* cuda_stream);

/* Device-side post-processing of the dense first guess (COTR/inference/inference_helper.py:131-145, the host work of
 * cotr_patch_flow_exhaustive after the 131 072-query forward): pred_dev holds n x (256*512) x 2 fp32 predictions for the
 * grid queries (j/512, i/256) in row-major (i, j) order; out_dev receives n x 256 x 512 x 3 fp32
 * [x in the other image's [-1,1] frame, y in [-1,1], cycle-consistency confidence] exactly as the reference's
 * `corr` array before it is split into its two halves (grid_sample: bilinear, zero padding, align_corners = False). */
int cotr_dense_postprocess(cotr_model* m, const float* pred_dev, int n, float* out_dev, void* cuda_stream);

/* Device-side tail of the dense first guess for ONE (tile of a, tile of b) answer (inference_helper.py:155-160, :61-75,
 * COTR/utils/utils.py:69-83): tile_dev is a 256 x 256 x 3 fp32 block [x, y, confidence] (row pitch `pitch_floats`, e.g.
 * one half of cotr_dense_postprocess' output).  (x, y) are mapped by the 2x3 affine `affine_host` (row-major doubles:
 * x' = a0 x + a1 y + a2, y' = a3 x + a4 y + a5, what cv2.getAffineTransform gives the reference), the three channels are
 * resized to ph x pw with Pillow's mode-'F' bilinear filter (bit-exact restatement) and merged into the oh x ow canvases
 * flow_dev (oh, ow, 2) / conf_dev (oh, ow) at (px, py): a pixel takes the tile's value when the tile's confidence is <=
 * the stored one (ties go to the later tile).  first != 0 initialises the canvases (flow 0, confidence 100) beforehand. */
int cotr_flow_tile_merge(cotr_model* m, const float* tile_dev, int pitch_floats, const double* affine_host, int px, int py, int pw, int ph,
                         int ow, int oh, float* flow_dev, float* conf_dev, int first, void* cuda_stream);

/* Squad formation of the grouped scheduler (FasterSparseEngine.form_grouped_batch / form_squad,
 * COTR/inference/sparse_engine.py:295-369) on the device.  pts_dev: n x 4 fp64 [x_from, y_from, x_to, y_to] of the open
 * tasks of one zoom level in the engine's (already shuffled) order; box_dev: n x 8 fp64, the central-half boxes
 * [f_l, f_r, f_u, f_d, t_l, t_r, t_u, t_d] of the two crops task i would impose as a pilot.  In list order every still
 * free task becomes the pilot of a new squad and takes along the first max_load free tasks strictly inside both of its
 * boxes, until batch_size squads exist.  squad_dev[i] = squad of task i or -1, rank_dev[i] = position inside the squad
 * (0 = pilot, members in list order), *n_squads_dev = squads formed.  All arrays DEVICE memory. */
int cotr_group_tasks(int device, const double* pts_dev, const double* box_dev, int n, int batch_size, int max_load, int32_t* squad_dev,
                     int32_t* rank_dev, int32_t* n_squads_dev, void* cuda_stream);

/* The rendering half of triangulate_corr (COTR/inference/inference_helper.py:293-308; the reference rasterises the
 * Delaunay triangles of the source points with OpenGL through vispy, vertex colour = target coordinates).
 * tris_dev: n_tri x 3 vertices x 4 fp32 [x, y, u, v] (DEVICE; x, y in pixels of the H x W source image, u, v the values
 * to interpolate); out_dev: H x W x 2 fp32 (DEVICE) = barycentric interpolation of (u, v) at every pixel centre
 * (x + 0.5, y + 0.5) covered by a triangle (top-left fill rule), zero elsewhere.  `device` is the CUDA device index. */
int cotr_rasterize_triangles(int device, const float* tris_dev, int n_tri, int H, int W, float* out_dev, void* cuda_stream);

/* ---- result exchange between the GPUs of one node over NVLink peer memory -------------------------------------------
 * The reference has no multi-GPU inference; its closest call site is the loop over independent pairs of
 * demo_reconstruction.py:44-49, which BASELINE.json configs[3] / configs[4] spread over 8 GPUs.  Pairs shard, weights are
 * replicated, and the only exchange is the all-gather of every rank's block of predictions.  cotr_exchange does that
 * gather with this library's own kernels instead of a collective: a push writes the block straight into every peer's
 * symmetric buffer (nobody waits in order to send), a wait polls the local arrival flags of one step and copies the
 * gathered blocks out.  One process per GPU:
 *     cotr_exchange_create(dev, rank, world, block_bytes, slots, &ex);  cotr_exchange_handle(ex, my_handle);
 *     <all-gather the 64-byte handles with whatever the host program has: torch.distributed, MPI, a file>
 *     cotr_exchange_connect(ex, all_handles);
 *     seq = cotr_exchange_push(ex, pred_dev, bytes, stream);  ...  cotr_exchange_wait(ex, seq, gathered_dev, NULL, stream);
 * Every rank must push the same sequence of steps.  `slots` (2..64) steps are kept; a wait for a step that a faster
 * peer has meanwhile overwritten is detected (cotr_exchange_status == 2), a peer that never publishes the step within
 * ~3 s gives status 1 instead of a hang.  A rank that alternates push and wait can never be overwritten.  Sizes and device
 * addresses are multiples of 16 bytes.  One stream at a time per exchange. */
typedef struct cotr_exchange cotr_exchange;
#define COTR_EXCHANGE_HANDLE_BYTES 64
int cotr_exchange_create(int device, int rank, int world, size_t block_bytes, int slots, cotr_exchange** out);
/* handle_out: COTR_EXCHANGE_HANDLE_BYTES bytes (a cudaIpcMemHandle_t of this rank's buffer) */
int cotr_exchange_handle(cotr_exchange* ex, void* handle_out);
/* handles: world x COTR_EXCHANGE_HANDLE_BYTES bytes in rank order (the own entry is ignored) */
int cotr_exchange_connect(cotr_exchange* ex, const void* handles);
/* the same for exchanges that live in ONE process (one thread per GPU, or tests): all[r] = the exchange of rank r */
int cotr_exchange_connect_local(cotr_exchange* ex, cotr_exchange* const* all);
/* returns the step number (1, 2, ...) or -1 */
long long cotr_exchange_push(cotr_exchange* ex, const void* block_dev, size_t bytes, void* cuda_stream);
/* gathered_dev: the blocks of step `seq` concatenated in rank order (NULL: only wait); bytes_per_rank: world entries
 * (HOST), NULL = every rank pushed block_bytes */
int cotr_exchange_wait(cotr_exchange* ex, long long seq, void* gathered_dev, const size_t* bytes_per_rank, void* cuda_stream);
/* 0 ok, 1 a peer never arrived, 2 a waited step was overwritten; meaningful after the stream of the wait synchronised */
int cotr_exchange_status(const cotr_exchange* ex);
void cotr_exchange_destroy(cotr_exchange* ex);

/* cotr_forward / cotr_forward_host replay a CUDA graph per (B,Q) shape (captured on the second call with that shape;
 * inputs / outputs pass through internal staging buffers so the graph's addresses stay fixed).  0 disables it. */
int cotr_set_graph_mode(cotr_model* m, int enabled);

/* Bytes of device workspace a (B,Q) call needs (activations only, excluding weights and contexts). */
size_t cotr_workspace_bytes(int B, int Q);

/* Number of kernels the last cotr_forward / encode / decode call launched (for bench.py's gpu_launches). */
int cotr_last_launch_count(const cotr_model* m);

/* Per-launch profiler.  Between cotr_profile_begin and cotr_profile_end every kernel the library launches is bracketed
 * by two CUDA events recorded on the launching stream.  cotr_profile_end synchronises the device, fills `out` with
 * one record per launch in launch order and returns -(count + 1) on success (so 0 records -> -1), > 0 on failure.
 * kernel ids: 0 gemm_tc (tcgen05), 1 gemm_simt, 2 attention_tc, 3 attention_simt (the fp32 path, and the default
 * schedule's attention of launches with fewer than 32 queries per pair), 4 layernorm, 5 maxpool, 6 query_encode, 7 stem_canvas.  For GEMMs M,N,K are the problem size; for attention M = query rows, N = 512, K = 256. */
typedef struct cotr_launch_record {
    int32_t kernel;
    int32_t M, N, K;
    float ms;
} cotr_launch_record;
int cotr_profile_begin(cotr_model* m, int max_records);
int cotr_profile_end(cotr_model* m, cotr_launch_record* out, int max_records);

/* Test hook: copy an intermediate of the LAST forward to the host.  name is one of
 * "feat" (2B,16,16,1024 NHWC, image n = 2*pair + half), "src" / "mem" (B*512,256 token-major),
 * "hs" (B*Q,256, final decoder LayerNorm output; only valid if B*Q fits in one decode chunk).
 * Returns the element count copied, or -1. */
int64_t cotr_debug_read(cotr_model* m, const char* name, float* out_host, int64_t max_elems);

/* Select the matrix-multiply path: 0 = tcgen05 tensor-core kernels (default), 1 = fp32 SIMT kernels
 * (debug / numerical cross-check only). */
int cotr_set_gemm_path(cotr_model* m, int path);

/* Batch-invariant inference mode (0 = off, the default).  By default each launch picks its schedule - GEMM tile width,
 * split-K, fused or separate LayerNorm, deferred LayerNorm, tensor-core or SIMT attention - from its own row count, so
 * a pair's predictions move in the last bits with the batch size, the query count and the decode chunking.  With the
 * mode on, every pair and every query is computed by the kernel sequence of the headline forward (B = 1, Q = 1024)
 * whatever B, Q, chunking or entry point the call has: the backbone and encoder are scheduled as for one pair, the
 * decoder, query projection and head as for 1024 query rows, LayerNorms run as separate launches and attention runs on
 * the tensor cores for any query count.  Consequences, all bitwise:
 *   - pair p alone gives the same predictions as pair p inside any batch;
 *   - a query gives the same prediction alone or among any others, at any position, across decode chunks and next to
 *     zero-padded queries;
 *   - cotr_forward, cotr_encode_context + any split of the queries over cotr_decode calls, cotr_forward_host, graph
 *     replay and eager execution agree;
 *   - at B = 1, Q = 1024 both modes launch the same kernels and produce the same bits.
 * Larger calls may be slower in this mode (narrow split-K tiles on big grids, separate LayerNorm launches).  The flag
 * belongs to the model handle.  Toggling it synchronises the device and drops captured graphs, like
 * cotr_set_gemm_path.  A context records the mode it was encoded under; cotr_decode refuses a context encoded under
 * the other mode.  The fp32 SIMT path (cotr_set_gemm_path 1) ignores the flag.  Bring-up switches of
 * cotr_debug_set_variant apply to every launch alike, so the guarantees hold under any fixed variant value. */
int cotr_set_batch_invariant(cotr_model* m, int enabled);

/* ---- kernel-level test hooks (used by tests/ only) ------------------------------------------------------ */
typedef struct cotr_test_gemm_desc {
    int32_t path;                 /* 0 = tcgen05, 1 = fp32 SIMT                                               */
    int32_t M, N, K;
    int32_t a_mode;               /* 0 row-major [M,K]; 1 implicit im2col over NHWC; 2 7x7/2 stem (A_dev = the fp32 (B,3,256,512) canvas, w_host [N][7][7][3]); 3 token gather */
    int32_t lda;
    int32_t H, W, C, OH, OW, KH, KW, stride, pad;   /* convolution geometry for a_mode 1 / 2                  */
    int32_t relu;
    int32_t add_period, ld_add, ldr, ldc;
    int32_t a_ln;                 /* 1: A holds PRE-LayerNorm rows (K = 256); ln_gamma / ln_beta are the norm of A,
                                     applied on the fly (deferred LayerNorm, tcgen05 path only) instead of an output norm */
    int32_t res_ln;               /* 1: the residual (ldr = N = 256) is a deferred LayerNorm too, same gamma / beta   */
    int32_t emit_part;            /* 1: also write the [M][16] (mean, M2) partial row statistics of the output (N = 256) */
    int32_t reserved;
    int64_t a_elems;              /* element count of the A activation tensor (a_mode 0 / 1 / 3)                 */
} cotr_test_gemm_desc;
/* out = epilogue(A * W^T): A/bias/addmat/residual/ln_* /out are fp32 DEVICE pointers (may be NULL where optional) -
 * the hook converts activations to / from the library's split16 storage around the kernel under test; w_host is a HOST
 * [N,K] matrix (packed for the tensor-core path internally). */
int cotr_test_gemm(const cotr_test_gemm_desc* d, const float* A_dev, const float* w_host, const float* bias_dev,
                   const float* addmat_dev, const float* residual_dev, const float* ln_gamma_dev,
                   const float* ln_beta_dev, float* out_dev, float* part_out_dev /* [M][16][2] or NULL */);
/* out[(p*nq+i), h*32+d] = softmax(q k^T) v per head; q (npairs*nq,256), k/v (npairs*512,256), all DEVICE, ld 256.
 * path: 0 = tcgen05 as the default schedule runs it (nq < 32 goes to the SIMT kernel), 1 = SIMT, 2 = tcgen05 for any
 * nq >= 1 (the batch-invariant schedule). */
int cotr_test_attention(int path, const float* q_dev, const float* k_dev, const float* v_dev, float* out_dev,
                        int nq, int npairs);
/* bring-up / A-B switches (0 = production): bit 8 (256) disables programmatic dependent launch, bit 9 (512) disables
 * split-K, bits 10-11 / 12-13 move the CTA-count thresholds of the 64- / 128-wide GEMM tiles, bits 14-15 lower the
 * minimum K of split-K (16 >> n chunks of 64), bit 17 selects trace mode for cotr_debug_set_timestamps, bits 20-22 stop
 * the encoder after n layers.  Schedule: by default a transformer section with >= 2048 rows runs the deferred-LayerNorm
 * schedule (no LayerNorm launches), smaller ones the explicit one; bit 19 forces deferred everywhere, bit 16 never;
 * bits 19 + 18 add the counter-based dataflow dependencies (experimental, slower - profiles/r02_deferred_layernorm.md).
 * Process-wide; graphs captured under another value are NOT dropped (call cotr_set_gemm_path twice to drop them). */
void cotr_debug_set_variant(int variant);
/* debug timeline of the tcgen05 kernels: DEVICE buffer of 64 int64 per CTA receiving clock64() deltas of the pipeline
 * events of every following GEMM / attention launch (NULL switches it off; graph replay is off while it is set).
 * Slot layout: tools/bringup.py::gemm_timeline / attn_timeline.  Trace mode (variant bit 17): the buffer holds
 * 256 x 64 slots PER LAUNCH (launch counter reset by this call), slot 62 receives %globaltimer at CTA exit, and graph
 * replay stays on - tools/bringup.py::forward_trace reconstructs a per-launch schedule of one forward from it. */
void cotr_debug_set_timestamps(void* dev_buffer);

const char* cotr_last_error(void);
const char* cotr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* COTR_B200_H_ */
