/*
 * include/llm_b200.h -- native host runtime of libllm_b200.so: the reference's model/session interface for the
 * LLaMA graph, as a C ABI (the reference's own host layer is Rust; no Rust toolchain exists here, so the same interface
 * is offered to C / ctypes callers -- see INTEGRATION.md for the Rust `extern "C"` block that binds it).
 *
 * Names, argument meaning and error behaviour mirror:
 *   Hyperparameters                 crates/models/llama/src/lib.rs:403-447
 *   ModelParameters                 crates/llm-base/src/model/mod.rs:197-229   (context_size, rope overrides)
 *   KnownModel::new / TensorLoader  crates/models/llama/src/lib.rs:43-140      (tensor names "layers.N.attention.wq.weight", ...)
 *   KnownModel::start_session       crates/models/llama/src/lib.rs:130-141  -> InferenceSession::new (inference_session.rs:114-217)
 *   InferenceSessionConfig          crates/llm-base/src/inference_session.rs:799-841 (n_batch; KV cache is f16)
 *   Model::evaluate + OutputRequest crates/models/llama/src/lib.rs:144-368, crates/llm-base/src/model/common.rs:6-39
 *   InferenceSession::feed_prompt   crates/llm-base/src/inference_session.rs:299-350 (chunks of n_batch, ContextFull)
 *
 * Where the per-node seam (ggml_b200.h) replays the reference's graph one node per call, this front end owns the whole
 * forward pass: a static schedule of fused sm_100a kernels (captured as a CUDA graph for decode), weights and KV cache
 * resident in HBM.  Both front ends run the same kernels and are held to the same parity bar.
 *
 * Threading / device contract: one process drives ONE device (b200_init picks it; multi-GPU = one process per GPU, see b200_llama_new_tp), and
 * the entry points of this header are to be called from one host thread at a time -- the launch code keeps per-process caches (kernel attributes,
 * occupancy tables, the RoPE / LUT tables) that are not synchronised.  Everything is ordered on the backend's single non-blocking stream.
 * b200_session_evaluate validates token ids; b200_session_evaluate_device takes them from HBM unchecked: ids in [0, n_vocab) are its precondition.
 */
#ifndef LLM_B200_H
#define LLM_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_model b200_model;
typedef struct b200_session b200_session;

typedef struct {
    int32_t n_vocab, n_embd, n_head, n_head_kv, n_layer, n_rot, n_ff;
    int32_t wtype;            /* enum ggml_type of the 2-D weights: 2 Q4_0, 3 Q4_1, 6 Q5_0, 7 Q5_1, 8 Q8_0 */
    int32_t context_size;     /* ModelParameters::context_size (default 2048) */
    float   rope_freq_base;   /* RoPEOverrides::frequency_base (10000) */
    float   rope_freq_scale;  /* RoPEOverrides::frequency_scale (1) */
} b200_llama_hparams;

typedef struct {
    int32_t n_batch;          /* InferenceSessionConfig::n_batch: largest evaluate() batch; reference default 8, prefill@512 uses 512 */
    int32_t flags;            /* B200_SESSION_* */
} b200_session_config;

enum {
    B200_SESSION_NO_GRAPH = 1,     /* launch the decode kernels one by one instead of replaying the captured CUDA graph (debug) */
    B200_SESSION_UNFUSED  = 2,     /* decode with the prefill schedule (one kernel per reference graph node, the seam's kernels) */
    B200_SESSION_MEGA     = 8,     /* experimental: one persistent cooperative kernel per decoded token (decode.cu) instead of the graph */
    B200_SESSION_FAST     = 4,     /* order-free kernels: integer-exact block dots but a different f32 summation order than the
                                      reference's AVX2 build.  NOT conformant: the reference graph amplifies 1e-7 differences to ~1e-2
                                      in the logits (DESIGN.md "chaos").  Default (flag clear) = bit-exact kernels. */
};

enum {                            /* return codes (0 = ok).  CUDA failures print and exit(1) like the reference backend. */
    B200_OK = 0,
    B200_ERR_CONTEXT_FULL = -1,   /* InferenceError::ContextFull (inference_session.rs:311-313, 388-390) */
    B200_ERR_BAD_ARG = -2,
    B200_ERR_UNKNOWN_TENSOR = -3, /* LoadError::UnknownTensor */
    B200_ERR_TENSOR_SHAPE = -4,   /* LoadError::TensorWrongSize */
    B200_ERR_NOT_LOADED = -5,
    /* file loading (ggml::format::LoadError, crates/ggml/src/format/loader.rs:38-70; llm_base::LoadError) */
    B200_ERR_IO = -10,
    B200_ERR_INVALID_MAGIC = -11,
    B200_ERR_INVALID_FORMAT_VERSION = -12,
    B200_ERR_INVARIANT_BROKEN = -13,        /* n_dims > 2, negative sizes, Q4_0/Q4_1 rows with ne0 % 64 != 0 */
    B200_ERR_UNSUPPORTED_ELEMENT_TYPE = -14,
    B200_ERR_QUANTIZATION_VERSION = -15,    /* quantized tensors need quantization version 2 (llm-base loader.rs:481-484) */
};

int  b200_init(int device);                                   /* accelerator::initialize(device), accelerator/mod.rs:68-77 */
int  b200_device_info(int32_t *sm_count, size_t *free_bytes, size_t *total_bytes);

b200_model *b200_llama_new(const b200_llama_hparams *hp);
/* Tensor-parallel shard tp_rank of tp_world (one process per GPU, <= 8; the north star's "weight rows shard across the 8 GPUs"): every 2-D weight but
 * tok_embeddings holds only this rank's OUTPUT ROWS -- wq/wk/wv: its heads, w1/w3: rows [rank*n_ff/G, +n_ff/G), wo/w2: rows [rank*n_embd/G, +n_embd/G),
 * output: rows [rank*n_vocab/G, +n_vocab/G) -- and b200_model_load_tensor takes exactly those rows.  Contrast: LC/ggml-cuda.cu:3355-3583 (row split by
 * g_tensor_split + a gather per mat-mul).  Sessions of such a model decode one token per step (b200_session_evaluate loops over a batch). */
b200_model *b200_llama_new_tp(const b200_llama_hparams *hp, int32_t tp_rank, int32_t tp_world);
/* TensorLoader::load(name) + Tensor::transfer_to(Backend::Gpu): host bytes in GGML layout (block arrays for quantized types) */
int  b200_model_load_tensor(b200_model *m, const char *name, int32_t type, const void *host_data, size_t nbytes);
/* fill every tensor with seeded synthetic weights generated ON the device (N(0,1/K) -> the reference's quantizer rule);
 * used by bench.py / smoke: there are no model files in this environment */
int  b200_model_synthesize(b200_model *m, uint64_t seed);
/* copy a tensor back in GGML layout (tests; lets the CPU oracle run on device-generated weights) */
int  b200_model_read_tensor(b200_model *m, const char *name, void *host_out, size_t nbytes);
size_t b200_model_tensor_nbytes(b200_model *m, const char *name);
size_t b200_model_weight_bytes(b200_model *m);                /* bytes of all 2-D weights resident in HBM */
int  b200_model_is_loaded(b200_model *m);                     /* every tensor of the architecture has been loaded */
void b200_model_free(b200_model *m);

/* ---- GGML / GGMF / GGJT model files (SURVEY.md §8f-2): ggml::format::load / save, llm::load::<Llama> -------------------------
 * The parser is host-only (mmap; usable without a GPU).  Offsets are from the start of the file; GGJT tensor data is 32-byte aligned. */
typedef struct b200_ggml_file b200_ggml_file;
typedef struct {
    char     name[96];
    int32_t  type, n_dims;        /* enum ggml_type; n_dims <= 2 */
    int64_t  ne[2];               /* ne[0] = row length */
    uint64_t offset, nbytes;      /* TensorLoadInfo::start_offset, calc_size() */
} b200_ggml_tensor_info;

enum { B200_ARCH_LLAMA = 0, B200_ARCH_GPT2 = 1, B200_ARCH_GPTNEOX = 2 };         /* whose Hyperparameters::read_ggml lays out the header */
b200_ggml_file *b200_ggml_open(const char *path, int *err);                     /* LLaMA header; NULL + *err on LoadError */
b200_ggml_file *b200_ggml_open_arch(const char *path, int32_t arch, int *err);
/* the header words in file order: llama n_vocab n_embd n_mult n_head n_layer n_rot file_type | gpt2 n_vocab n_ctx n_embd n_head n_layer file_type n_vocab |
 * gptneox n_vocab n_ctx n_embd n_head n_layer n_rot use_parallel_residual file_type */
int     b200_ggml_hparams(const b200_ggml_file *f, int32_t *arch, int32_t *words8, int32_t *n_words);
void    b200_ggml_close(b200_ggml_file *f);
int     b200_ggml_container(const b200_ggml_file *f, uint32_t *magic, uint32_t *version);      /* ContainerType */
int64_t b200_ggml_n_tensors(const b200_ggml_file *f);
int     b200_ggml_tensor(const b200_ggml_file *f, int64_t i, b200_ggml_tensor_info *out);
const void *b200_ggml_tensor_data(const b200_ggml_file *f, int64_t i);          /* into the mapping */
int64_t b200_ggml_n_vocab(const b200_ggml_file *f);
int     b200_ggml_token(const b200_ggml_file *f, int64_t i, const uint8_t **bytes, uint32_t *len, float *score);
/* llama Hyperparameters::read_ggml + FileType + the quantization-version rule; n_ff / wtype are taken from the tensor table */
int     b200_ggml_llama_hparams(const b200_ggml_file *f, b200_llama_hparams *out, int32_t *n_mult, int32_t *llama_ftype, int32_t *quantization_version);
/* ggml::format::save (GGJT v3): header words verbatim (any architecture), or the LLaMA convenience form */
int     b200_ggml_write(const char *path, const int32_t *hparam_words, int32_t n_words, int32_t n_vocab, const uint8_t *const *token_bytes, const uint32_t *token_len,
                        const float *token_score, const b200_ggml_tensor_info *tensors, const void *const *data, int64_t n_tensors);
int     b200_ggml_write_llama(const char *path, const b200_llama_hparams *hp, int32_t n_mult, int32_t file_type, const uint8_t *const *token_bytes, const uint32_t *token_len,
                              const float *token_score, const b200_ggml_tensor_info *tensors, const void *const *data, int64_t n_tensors);
/* llm::load::<Llama>(path, ModelParameters): parse + b200_llama_new + one b200_model_load_tensor per tensor, straight from the mapping;
 * context_size / rope_* <= 0 keep the defaults (2048, 10000, 1) */
b200_model *b200_llama_load_file(const char *path, int32_t context_size, float rope_freq_base, float rope_freq_scale, int *err);
/* same with ModelParameters::n_gqa (grouped-query attention: n_head_kv = n_head / n_gqa, e.g. 8 for 70B files) */
b200_model *b200_llama_load_file_gqa(const char *path, int32_t context_size, float rope_freq_base, float rope_freq_scale, int32_t n_gqa, int *err);
/* b200_model_load_tensor + the loader's dims check (LoadError::TensorWrongSize on a dims mismatch even when the byte count matches) */
int  b200_model_load_tensor_shaped(b200_model *m, const char *name, int32_t type, int32_t n_dims, int64_t ne0, int64_t ne1, const void *host_data, size_t nbytes);

b200_session *b200_model_start_session(b200_model *m, const b200_session_config *cfg);
/* One forward pass over `n` tokens appended at n_past (InferenceSession::compute + Llama::evaluate).  tokens: HOST int32.
 * logits_out: HOST f32, n rows of n_vocab when all_logits (OutputRequest::all_logits), else the last row (read_last_token).
 * May be NULL (feed only).  n must be <= n_batch. */
int  b200_session_evaluate(b200_session *s, const int32_t *tokens, int32_t n, float *logits_out, int32_t all_logits);
/* feed_prompt: evaluate in chunks of n_batch; last row of logits returned */
/* sampler hand-off (SURVEY.md 8f-3): the k (<= 1024) largest logits of the last evaluated row, selected on the device -- descending logit,
 * ties by ascending token id -- so that 8 k bytes cross PCIe instead of n_vocab floats */
int  b200_session_top_k(b200_session *s, int32_t k, int32_t *ids_out, float *logits_out);
int  b200_session_feed_prompt(b200_session *s, const int32_t *tokens, int32_t n, float *last_logits_out);
/* Device-resident variant for measurements: tokens already in HBM, logits stay in HBM (no host copies, no sync) */
int  b200_session_evaluate_device(b200_session *s, const int32_t *d_tokens, int32_t n);
const float *b200_session_device_logits(b200_session *s);    /* [n][n_vocab] of the last evaluate */
int32_t b200_session_n_past(const b200_session *s);
int  b200_session_set_n_past(b200_session *s, int32_t n_past);   /* rewind (supports_rewind, llama lib.rs:396-398) */
/* raw f16 KV cache bytes (get_snapshot, inference_session.rs:599-646): which = 0 memory_k, 1 memory_v */
int  b200_session_read_kv(b200_session *s, int32_t which, void *host_out, size_t nbytes);
int  b200_session_sync(b200_session *s);
/* with B200_DECODE_PROF=1 in the environment the decode kernel stamps %globaltimer (ns) at its phase boundaries (CTA 0);
 * slot 0 = start, then pairs (before / after grid barrier) per phase in graph order, slot 127 = end of token */
int  b200_session_decode_profile(b200_session *s, unsigned long long *out128);
/* tuning aid (B200_DECODE_PROF=1): per-launch %globaltimer stamps of the graph decode schedule; out = 9*n values, see session.cu */
int  b200_session_decode_timeline(b200_session *s, unsigned long long *out, int n, int reset);
/* debug taps for parity work: keep a copy of one intermediate buffer of (layer, stage) during the next evaluate.
 * stages: 1 attn-norm out [n][e], 2 qkv before rope [n][e+2gqa], 3 qkv after rope, 4 KQ raw [h][n][n_kv], 5 KQ softmax, 6 merged
 * KQV [n][e], 7 inpFF, 8 ffn-norm out, 9 [w1x | w3x] [n][2f], 10 silu*mul [n][f], 11 layer output [n][e] */
int  b200_session_set_tap(b200_session *s, int32_t layer, int32_t stage);
int64_t b200_session_read_tap(b200_session *s, float *host_out, int64_t max_count);
/* kernels launched by the last evaluate (for bench.py's gpu_launches) and whether it replayed a CUDA graph */
int32_t b200_session_last_launches(const b200_session *s);
void b200_session_free(b200_session *s);
/* Tensor-parallel sessions: each rank exports the CUDA IPC handle (64 bytes) of its exchange slab, the host layer gathers the handles of all ranks
 * (any channel: torch.distributed, MPI, a pipe) and hands the table [tp_world][64] back; after that the decode kernels store their output slices
 * straight into every peer's slab over NVLink (llm_b200/csrc/tp.cuh).  Every rank must call evaluate with the same tokens in the same order.
 * ONE tensor-parallel session per process: the exchange context (peer pointers, epoch) lives in constant memory of the decode kernels' module
 * (one process per GPU, like the reference's one-session-per-process global state, LC/ggml-cuda.cu:2598-2686). */
int  b200_session_tp_handle(b200_session *s, void *handle_out64);
int  b200_session_tp_connect(b200_session *s, const void *handles_by_rank);
int32_t b200_session_tp_timeouts(b200_session *s);
/* measurement aid: nowait 1 skips the tag waits (garbage results; time = compute + peer stores), 2 also keeps every store local (time = compute alone):
 * sizes the exchange's share of a token */
int  b200_session_tp_set_nowait(b200_session *s, int32_t nowait);

/* stream handle (cudaStream_t) on which everything above is ordered -- for CUDA-event timing from the host side */
void *b200_stream(void);
/* CUDA-event stopwatch on that stream: begin records an event; end records a second one, waits for it and returns ms */
int   b200_timing_begin(void);
float b200_timing_end_ms(void);
/* Roofline probe for the dominant decode kernel: `reps` passes over EVERY weight mat-vec of the model (wqkv, wo, w13, w2 per
 * layer + output; 3.7 GB for 7B Q4_0, far larger than L2) on the session's current quantized activations, timed with CUDA
 * events.  Returns total ms; *launches = kernels launched, *bytes = algorithmic weight bytes streamed (all reps). */
float b200_session_probe_matvec(b200_session *s, int32_t reps, int64_t *launches, double *bytes);

/* ---- GPT-NeoX (crates/models/gptneox): KnownModel + InferenceSession, same conventions as the LLaMA entry points above --------------------------
 * Hyperparameters (gptneox lib.rs:403-447 region): tensor names are the loader's ("gpt_neox.embed_in.weight", "gpt_neox.layers.N.attention.
 * query_key_value.weight" [3e x e, rows per head: q | k | v], ..., "embed_out.weight"); every 2-D ".weight" is quantized to wtype, biases / LayerNorm f32. */
typedef struct b200_neox_hparams {
    int32_t n_vocab, n_embd, n_head, n_layer, n_rot, use_parallel_residual, wtype, context_size;
    int32_t arch;          /* 0 = GPT-NeoX; 1 = GPT-2 (crates/models/gpt2): tensor names "model/wte", "model/wpe" (f32 [n_ctx][n_embd]), "model/hN/attn/c_attn/w" ...,
                              c_attn rows in thirds, no RoPE (n_rot ignored), sequential residual; context_size = the model's n_ctx (rows of wpe) */
    int32_t has_lm_head;   /* GPT-2: "model/lm_head" present; 0 = output projection tied to model/wte (gpt2 lib.rs:319-320) */
} b200_neox_hparams;
typedef struct b200_neox_model b200_neox_model;
typedef struct b200_neox_session b200_neox_session;
b200_neox_model *b200_neox_new(const b200_neox_hparams *hp);
int  b200_neox_load_tensor(b200_neox_model *m, const char *name, int32_t type, const void *host_data, size_t nbytes);
int  b200_neox_synthesize(b200_neox_model *m, uint64_t seed);          /* seeded weights generated in HBM (bench) */
size_t b200_neox_weight_bytes(b200_neox_model *m);                     /* bytes streamed per decoded token */
void b200_neox_free(b200_neox_model *m);
b200_neox_session *b200_neox_start_session(b200_neox_model *m, int32_t n_batch);
int  b200_neox_evaluate(b200_neox_session *s, const int32_t *tokens, int32_t n, float *logits_out, int32_t all_logits);
int  b200_neox_evaluate_device(b200_neox_session *s, int32_t n);       /* tokens of the last evaluate stay in HBM, logits stay in HBM */
int32_t b200_neox_n_past(const b200_neox_session *s);
int  b200_neox_set_n_past(b200_neox_session *s, int32_t n_past);
int32_t b200_neox_last_launches(const b200_neox_session *s);
int  b200_neox_sync(b200_neox_session *s);
void b200_neox_session_free(b200_neox_session *s);

/* ---- single-op entry points on HOST buffers (unit tests, INTEGRATION examples).  Each uploads, runs the kernel, downloads. */
int  b200_op_quantize_act(int32_t vec_dot_type, const float *x, int64_t K, int64_t B, int8_t *qs_out, float *d_out, float *aux_out);
/* ggml_quantize_q{4_0,4_1,5_0,5_1,8_0} (LC/ggml.c:18083-18230) on the GPU: w_host f32 [N][K] -> N rows of GGML blocks, bit-exact with the reference */
int  b200_op_quantize_weights(int32_t wtype, const float *w_host, int64_t K, int64_t N, void *ggml_blocks_out);
/* wtype: GGML_TYPE_Q4_0/Q4_1/Q5_0/Q5_1/Q8_0 (2,3,6,7,8; K % 64 == 0), or the K-quants Q2_K..Q6_K (10..14; K % 256 == 0, impl AUTO or EXACT:
 * ggml_vec_dot_q{2,3,4,5,6}_K_q8_K of LC/k_quants.c:1240,1763,2492,3023,3592 on quantize_row_q8_K activations, bit-exact with the reference's AVX2 build) */
int  b200_op_mul_mat(int32_t wtype, const void *w_ggml, int64_t K, int64_t N, const float *x, int64_t B, float *dst, int32_t impl);
/* quantize_row_q8_K (LC/k_quants.c:1133-1183) of B rows of K floats -> B * K/256 block_q8_K {f32 d; i8 qs[256]; i16 bsums[16]} (292 bytes each), bit-exact */
int  b200_op_quantize_q8_K(const float *x, int64_t K, int64_t B, void *blocks_out);
enum { B200_MM_AUTO = 0, B200_MM_VEC = 1, B200_MM_SIMPLE = 2, B200_MM_TENSOR = 3, B200_MM_EXACT = 4, B200_MM_EXACT_STREAM = 5, B200_MM_EXACT_MMA = 6, B200_MM_EXACT_TC5 = 7, B200_MM_FAST_TC5 = 8 };   /* AUTO = EXACT; TC5 = tcgen05/TMEM/TMA kernel (exact_tc5.cu); FAST_TC5 = order-free dequant->tcgen05 GEMM (mmq_tc5.cu, non-conformant) */

#ifdef __cplusplus
}
#endif
#endif
