/* libmmee — C ABI of the B200 (sm_100a) early-exit LayoutLMv3 inference engine.
 *
 * The reference (Jordy-VL/multi-modal-early-exit) has no FFI of its own: its boundary for this path is two
 * Python call sites (SURVEY.md §8b):
 *   (1) outputs = model.forward(**batch)                       EE/utils.py:179
 *       -> LayoutLMv3EEForSequenceClassification.forward       EE/models/LayoutLMv3.py:696-896
 *   (2) Policy(logits, config).max_confidence_global_thresholding_policy()   EE/eval.py:91-98, EE/policy.py:12-53
 * The entry points below are what a binding for those two call sites needs; the Python mirror of the
 * reference interface (multi-modal-early-exit_b200/mmee/model.py) binds them with ctypes.
 * Plain pointers and sizes only; return code 0 = ok, < 0 = error (text via mmee_last_error()).
 * One engine per (device, model).  Calls on one engine are stream-ordered and NOT thread-safe.
 */
#ifndef MMEE_H_
#define MMEE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMEE_MAX_EXITS 64
/* embedding-level exits in exit_after_layer (EE/models/LayoutLMv3.py:465-483, 519-534, 581-606) */
#define MMEE_EXIT_VISION_AVG (-2)   /* mean of the visual embeddings */
#define MMEE_EXIT_TEXT_AVG   (-1)   /* mean of the text embeddings */
#define MMEE_EXIT_CONCAT       0    /* mean of the fused [text | visual] embeddings */

typedef struct mmee_engine mmee_engine;

/* Model description: HF LayoutLMv3Config fields (configuration_layoutlmv3.py) + the reference's ExitConfig
 * (EE/models/EE_modules.py:175-195). */
typedef struct {
  int hidden, layers, heads, inter;
  int n_text;               /* text tokens per document (512) */
  int image, patch, channels;
  int n_labels;
  int coord, shape;         /* coordinate_size, shape_size: 4*coord + 2*shape == hidden */
  int vocab, max_pos, max_2d;
  int rel_bins, max_rel, rel2d_bins, max_rel2d;
  int pad_id;
  float ln_eps, vis_ln_eps;
  int n_exits;                             /* E early exits, final classifier not counted */
  int exit_after_layer[MMEE_MAX_EXITS];    /* ascending; -2 / -1 / 0 = vision_avg / text_avg / text_visual_concat
                                              (embedding-level, see above), 1..layers = after that encoder layer */
  int head_kind;                           /* 0 ramp (EarlyExitHead.RAMP), 1 gate (EarlyExitHead.GATE) */
  int head_layers;                         /* exit_head_num_layers: 1 | 2 */
  int compute_dtype;                       /* MMEE_DTYPE_BF16 (default) | MMEE_DTYPE_FP32, see below */
} mmee_model_desc;

/* Arithmetic of the dense contractions (QKV / output / MLP projections, patch embedding, attention).  Everything else
 * (embedding sums, LayerNorm, GELU, softmax, exit heads, criteria) is fp32 in both modes.
 *   MMEE_DTYPE_BF16  bf16 tensor-core operands, fp32 accumulation: logits within 1e-2 of the reference's fp32 forward
 *   MMEE_DTYPE_FP32  fp32-parity mode (the reference computes in fp32, EE/utils.py:160-164): every operand is a
 *                    split-bf16 pair (hi + lo = 16 mantissa bits) and each product runs as hi*hi + lo*hi + hi*lo on
 *                    the same tensor cores with fp32 accumulation: logits within 1e-4 (measured ~5e-6), ~3x the
 *                    tensor work of the bf16 mode. */
#define MMEE_DTYPE_BF16 0
#define MMEE_DTYPE_FP32 1

/* Exit policy: EarlyExitInference criterion + sign (EE/models/EE_modules.py:116-146), per-exit thresholds
 * (EE/policy.py:17, :71-79) and per-exit temperatures (EE/generic_scaling.py:54-61, EE/eval.py:312-327). */
#define MMEE_CRIT_MAX_CONFIDENCE 0
#define MMEE_CRIT_ENTROPY        1
#define MMEE_CRIT_LTE            2

typedef struct {
  int criterion;              /* 0 max_confidence: exit iff crit > thr ; 1 entropy: exit iff crit < thr ;
                                 2 LTE (EE_config["use_lte"], EE/models/LayoutLMv3.py:142-149, 231-268): crit =
                                 sigmoid(lte_classifier(exit input row)), exit iff crit < thr, taken only at encoder
                                 exits after layer l < number of encoder exits (the reference's `i + 1 <
                                 self.num_layers`); embedding-level exits are scored but never taken.  Temperatures
                                 do not enter the LTE score.  Needs layoutlmv3.encoder.lte_classifier.{weight,bias}. */
  int mode;                   /* 0 dense: every exit head for every document (what the reference computes);
                                 1 early-exit: exiting documents leave, deeper layers run on survivors only */
  const float* thresholds;    /* [n_exits]   (host) */
  const float* temperatures;  /* [n_exits+1] (host) or NULL for T = 1 */
} mmee_policy;

/* Result buffers.  All nullable except logits / exit_index.  Shapes use B = batch, K = n_labels, E = n_exits.
 * In early-exit mode rows of all_* for exits a document never reached are NaN. */
typedef struct {
  float*   logits;          /* [B, K]     class logits of the exit each document took (Policy `predictions`) */
  int32_t* exit_index;      /* [B]        index into the E+1 exits (Policy `exits_store`) */
  float*   criterion;       /* [B]        criterion value at that exit (after temperature) */
  float*   all_exit_logits; /* [E+1, B, K]  per-exit class logits (what EE/utils.py:182-193 stores) */
  float*   all_head_logits; /* [E+1, B, K]  raw head outputs = exit_states[j][0] (first 2 cols in gate mode) */
  float*   all_criteria;    /* [E+1, B] */
  int64_t* exit_hist;       /* [E+1]      documents per exit */
} mmee_outputs;

int  mmee_create(const mmee_model_desc* desc, int device, int max_batch, mmee_engine** out);
void mmee_destroy(mmee_engine* e);

/* Copy one parameter (fp32, host memory) under its reference state-dict name
 * (e.g. "layoutlmv3.encoder.layer.3.attention.self.query.weight"; SURVEY.md Appendix A.6). */
int  mmee_set_weight(mmee_engine* e, const char* hf_name, const float* host_data, const int64_t* shape, int rank);
/* Optional: |rel| -> bucket tables of HF relative_position_bucket (modeling_layoutlmv3.py:393-414) computed
 * by the caller; which = 0 (1-D, rel_pos_bins/max_rel_pos) or 1 (2-D).  Defaults are computed in C. */
int  mmee_set_bucket_lut(mmee_engine* e, int which, const uint8_t* lut, int n);
/* Read back the table in use (for tests). Returns the table length or < 0. */
int  mmee_get_bucket_lut(mmee_engine* e, int which, uint8_t* lut_out, int capacity);
/* Pack weights (bf16 conversion, fused QKV, 1/sqrt(d) folded into W_q) and verify none is missing. */
int  mmee_finalize_weights(mmee_engine* e);

/* One forward over B <= max_batch documents; inputs and outputs in HOST memory (the reference-facing call:
 * host->device and device->host copies are part of it).
 *   input_ids i64[B,n_text], bbox i64[B,n_text,4], attention_mask i64[B,n_text], pixel_values f32[B,C,img,img] */
int  mmee_forward(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                  const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out);
/* Same, inputs and outputs already in DEVICE memory of the engine's GPU; asynchronous on `cuda_stream`
 * (a cudaStream_t; NULL = the engine's own stream, synchronised before returning). */
int  mmee_forward_device(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                         const int64_t* attention_mask, const float* pixel_values, const mmee_policy* policy,
                         const mmee_outputs* out, void* cuda_stream);

/* Document images as uint8 pages, for callers that would otherwise run the LayoutLMv3 image processor on the host:
 * the engine resizes, rescales and normalises them on the device, bit for bit as that processor does (Pillow's
 * Image.resize((image, image), BILINEAR) of Image.fromarray(page).convert("RGB"), then (r / 255 - 0.5) / 0.5 in fp32;
 * oracle/image_port.py).  Decoding stays with the caller. */
typedef struct {
  const uint8_t* data;     /* all B images back to back, row-major HWC */
  const int64_t* offsets;  /* [B] byte offset of image b in data        (HOST memory) */
  const int32_t* sizes;    /* [B, 2] (height, width), each in [1, 16384] (HOST memory) */
  int channels;            /* 1 (grayscale) or 3 (RGB), the whole batch */
  int64_t total_bytes;     /* size of data: what the host path uploads, and the bound every image is checked against */
} mmee_images;
/* data and pixel_values in DEVICE memory; pixel_values f32 [B, 3, image, image]; async on cuda_stream
   (NULL = engine stream, synchronised).  Composes with mmee_forward_device and mmee_plan_forward_device.
   Rejected before any launch: channels other than 1 or 3, a size outside [1, 16384], an image whose bytes run past
   total_bytes, B outside [1, max_batch], an engine whose channels are not 3. */
int  mmee_preprocess_images(mmee_engine* e, int B, const mmee_images* images, float* pixel_values, void* cuda_stream);
/* mmee_forward with images (and everything else) in HOST memory instead of pixel_values.  The image bytes go up and
   are preprocessed on the engine's copy stream, overlapping the text embedding and the bias build as the pixel upload
   of mmee_forward does. */
int  mmee_forward_images(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                         const int64_t* attention_mask, const mmee_images* images, const mmee_policy* policy,
                         const mmee_outputs* out);

/* Pipelined form of mmee_forward for throughput callers (a dataset loop such as EE/utils.py:169-193): up to TWO
 * forwards in flight, so the upload of batch n+1 (160 MB of pixels at 256 documents) overlaps the computation of
 * batch n.  submit enqueues the host->device copies, the forward and the result staging and returns a ticket (0 or 1)
 * without waiting; the host input buffers must stay valid (and should be pinned) until the ticket is collected.
 * collect blocks until that forward has finished and copies logits / exit_index / criterion / exit_hist to the host
 * buffers of `out` (the all_* outputs are not available on this path). */
int  mmee_forward_submit(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                         const int64_t* attention_mask, const float* pixel_values, const mmee_policy* policy);
int  mmee_forward_collect(mmee_engine* e, int ticket, const mmee_outputs* out);

/* Forward plans: one forward captured into a CUDA graph and instantiated, for a fixed batch size, criterion, mode and
 * set of outputs.  A run launches the graph once instead of ~100 kernels, which is what a caller with few documents
 * per call (the reference's eval loop runs one, EE/utils.py:169-193) pays for.  In early-exit mode every exit opens an
 * IF node around the rest of the forward: once every document has left, the deeper layers are not launched at all.
 * Thresholds and temperatures are inputs of every run (uploaded to the device before the graph starts), so one plan
 * serves every policy.  A plan uses the engine's scratch buffers and staged-input buffers: its runs are ordered with
 * the engine's other forwards, on any stream, as those are with each other.  Stage profiling (mmee_set_profiling)
 * does not apply to plan runs. */
typedef struct mmee_plan mmee_plan;
/* Capture one forward for a fixed batch B <= max_batch.  criterion and mode come from `shape` (thresholds and
 * temperatures are ignored here: they are inputs of every run); want_all = 1 also produces the all_* outputs.
 * Creation runs one eager forward of neutral inputs first (kernel attributes, module loading) and synchronises. */
int  mmee_plan_create(mmee_engine* e, int B, const mmee_policy* shape, int want_all, mmee_plan** out);
/* Same inputs / outputs / errors as mmee_forward and mmee_forward_device, for exactly B documents; policy->criterion and
 * policy->mode must equal the plan's.  Bit-identical results to the eager entry points. */
int  mmee_plan_forward(mmee_plan* p, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                       const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out);
int  mmee_plan_forward_device(mmee_plan* p, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                              const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out,
                              void* cuda_stream);
void mmee_plan_destroy(mmee_plan* p);   /* before mmee_destroy; mmee_destroy frees plans still alive */

/* Number of kernels launched by the engine in the last eager forward (for the bench's gpu_launches). */
int64_t mmee_last_launch_count(mmee_engine* e);
/* Device time per stage ("total", "embed", "gemm", "attention", "norm", "exit"), SUMMED in ms over the forwards run
 * since profiling was switched on or last collected, and the number of those forwards ("forwards"): only recorded when
 * mmee_set_profiling(e, 1) is on (adds event records between stages; calling it again restarts the accumulation). */
int  mmee_set_profiling(mmee_engine* e, int on);
/* Wait for the forwards enqueued on `cuda_stream` (NULL: the engine's own stream), fold the stage events and turn a
 * tripped attention guard into an error: what the synchronous entry points do before they return, for callers of the
 * asynchronous mmee_forward_device. */
int  mmee_sync(mmee_engine* e, void* cuda_stream);
/* Synchronise the device and fold the recorded stage events of the last forward into per-stage times. */
int  mmee_collect_profile(mmee_engine* e);
double mmee_last_stage_ms(mmee_engine* e, const char* stage);
/* Test hook: copy an internal activation buffer ("X0","X1","QK","VT","CTX","A1","MID","Y","VIS","POOL","BIAS")
 * to host memory (synchronises the device). Returns bytes copied or < 0.  "NDEV": the active documents per exit stage
 * (int32 [n_exits + 3]; a plan run first sets entries 1.. to -1, so a stage whose exit kernel was skipped reads -1). */
int64_t mmee_debug_read(mmee_engine* e, const char* name, void* host_dst, int64_t capacity_bytes);

/* Post-hoc exit policy over stored per-exit logits: the device replacement of the per-sample double loop of
 * Policy.max_confidence_global_thresholding_policy / accuracy_calibration_heuristic (EE/policy.py:12-53, 55-111),
 * of the threshold sweeps that re-run it once per threshold (EE/eval.py:227-274 full_test_iteration,
 * EE/thresh.py:106-132) and of the per-exit threshold-vector ("mixture") sweeps opt0_2D / check_2D_threshold
 * (EE/thresh.py:184-215, EE/large_scale.py:42-84: 1.5 M mixtures over the whole test set).
 *
 * A policy store holds the criteria of one logits store on the device (fp64 like the reference: scipy softmax on the
 * f64 store, EE/utils.py:160-164); every scan after that moves only thresholds in and counts out.
 *   logits       f64 [E1, N, K]   per-exit logits incl. the final classifier (EE/utils.py:160-193 `logits_store`)
 *   temperatures f64 [E1] or NULL logits[e] / T_e before the criterion (EE/generic_scaling.py:54-61)
 *   criterion    0 max softmax ; 1 entropy (EE/models/EE_modules.py:149-160) ; 2 the "margin" CSF of
 *                EE/thresh.py:48-62 as the reference computes it (smallest minus second-smallest logit; larger fires)
 *   labels       i64 [N] or NULL  enables correct_out
 * All buffers in HOST memory. */
typedef struct mmee_policy_store mmee_policy_store;
int  mmee_policy_store_create(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                              const double* temperatures, int criterion, const int64_t* labels,
                              mmee_policy_store** out);
void mmee_policy_store_destroy(mmee_policy_store* store);
/* crit_out f64 [E1, N]: the criterion of every (exit, sample) as held on the device. */
int  mmee_policy_store_criteria(mmee_policy_store* store, double* crit_out);
/* One scan = n_thr sweep points (any number: 1 for Policy, ~50 for full_test_iteration, 1.5 M for large_scale.py).
 *   thresholds   f64 [n_thr, E1]  one row per sweep point (a global threshold = a constant row)
 *   mode 0       EE/policy.py:28-45: exit iff crit > thr (entropy: crit < thr), strict; the last column is ignored:
 *                the final classifier always fires (:40-45)
 *   mode 1       check_2D_threshold (EE/thresh.py:184-185): (CSF >= thr[:, None]).argmax(0) with CSF = max softmax, or
 *                the NEGATED entropy (EE/large_scale.py:15); every column is tested, a sample that fires nowhere gets
 *                exit 0
 * Outputs, each nullable: exits_out i32 [n_thr, N] (`exits_store`; leave NULL for large sweeps: nothing of that size
 * is then allocated anywhere), hist_out i64 [n_thr, E1] (exit_distribution * N), correct_out i64 [n_thr] (samples
 * whose arg-max class at the exit taken equals the label; needs labels). */
int  mmee_policy_store_scan(mmee_policy_store* store, const double* thresholds, int64_t n_thr, int mode,
                            int32_t* exits_out, int64_t* hist_out, int64_t* correct_out);
/* One-shot form (store created, scanned in mode 0 and dropped): crit_out f64 [E1, N] nullable. */
int  mmee_policy_scan(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                      const double* temperatures, int criterion, const double* thresholds, int n_thr,
                      const int64_t* labels, int32_t* exits_out, double* crit_out, int64_t* hist_out,
                      int64_t* correct_out);

/* Temperature calibration of the per-exit logits: the device replacement of TemperatureScaler.set_temperature
 * (EE/generic_scaling.py:64-111, scipy L-BFGS-B on log_loss(labels, softmax(logits / T))) as EE/eval.py:311-335 runs
 * it once per exit.  Minimises nll(T_e) = mean_i -log softmax(logits[e][i] / T_e)[labels[i]] for every exit at once
 * (safeguarded Newton on 1 / T, fp64; the problem is convex in 1 / T).  All buffers in HOST memory.
 *   logits   f64 [E1, N, K] ; labels i64 [N] in [0, K) ; t_init f64 [E1] or NULL (= 1.0, the reference's start)
 *   max_iter <= 0 : 40
 * Outputs ([E1] each, all but t_out nullable): t_out fitted temperatures, nll_before (at t_init), nll_after,
 * mean_conf_out = mean max softmax(logits / T) and accuracy_out = mean(argmax == label) at the fitted T.
 * An exit whose data are separable has no finite minimiser (nll -> 0 as T -> 0); the iteration then stops where the
 * fp64 gradient vanishes, as the reference's does. */
int  mmee_temperature_fit(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                          const int64_t* labels, const double* t_init, int max_iter, double* t_out, double* nll_before,
                          double* nll_after, double* mean_conf_out, double* accuracy_out);
/* The same statistics for given temperatures (NULL = 1.0): what EE/eval.py:325-335 collects from the calibrated
 * test logits.  Outputs f64 [E1], each nullable. */
int  mmee_calibration_stats(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                            const int64_t* labels, const double* temperatures, double* nll_out, double* mean_conf_out,
                            double* accuracy_out);

const char* mmee_last_error(void);
const char* mmee_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MMEE_H_ */
