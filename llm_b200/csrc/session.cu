// llm_b200/csrc/session.cu -- native host runtime (include/llm_b200.h): Llama model + InferenceSession on the B200.
//
// Mirrors, in C++ over the kernels of this directory, what the reference does in Rust over ggml:
//   Llama::new / TensorLoader          crates/models/llama/src/lib.rs:43-140
//   InferenceSession::new / compute    crates/llm-base/src/inference_session.rs:114-295
//   Llama::evaluate (the graph)        crates/models/llama/src/lib.rs:144-368
// The forward pass below is that graph, node for node in arithmetic, but scheduled statically: no per-eval graph
// construction, no arena reset, weights resident in HBM in the planes layout, wq|wk|wv and w1|w3 stored as single matrices
// so one activation quantization and one mat-mul launch serve them.
#include <string.h>

#include <string>
#include <vector>

#include "../../include/llm_b200.h"
#include "decode.h"
#include "kernels.cuh"
#include "runtime.h"

namespace b200 {
void synth_qweight(const QWeight &w, uint64_t seed, cudaStream_t st);
void synth_gain(float *g, int64_t n, uint64_t seed, cudaStream_t st);
}  // namespace b200
using namespace b200;

namespace {

QWeight row_view(const QWeight &w, int64_t row0, int64_t nrows) {   // rows [row0, row0+nrows) of a planes matrix
    QWeight v = w;
    v.N = nrows;
    v.qs = w.qs + (size_t)row0 * w.nb * qs_bytes(w.type);
    if (w.qh) v.qh = w.qh + (size_t)row0 * w.nb;
    v.dm = (const uint8_t *)w.dm + (size_t)row0 * w.nb * (has_min(w.type) ? 4 : 2);
    v.base = nullptr;
    return v;
}

struct Layer {
    float *attention_norm = nullptr, *ffn_norm = nullptr;
    QWeight wqkv, wo, w13, w2;          // wqkv rows: [wq | wk | wv]; w13 rows: [w1 | w3]
};

}  // namespace

struct b200_model {
    b200_llama_hparams hp;
    int gqa = 0, hd = 0;
    // tensor parallelism (b200_llama_new_tp): this rank holds 1/tp_world of the ROWS of every weight matrix (tp.cuh); *_loc = local row counts
    int tp_rank = 0, tp_world = 1;
    int e_loc = 0, gqa_loc = 0, f_loc = 0, v_loc = 0;
    char *slab = nullptr;               // one HBM allocation for every weight
    size_t slab_bytes = 0, weight_bytes = 0;
    QWeight wte, output;
    float *norm = nullptr;
    std::vector<Layer> layers;
    std::vector<uint8_t> loaded;        // per tensor slot
    int n_loaded = 0;

    // chunk > 0: the tensor's rows live in `chunk`-row pieces, piece c at rows [c * stride + q_row0, + chunk) of the matrix `q`
    // (w1 / w3 are interleaved in 32-row pieces inside w13 so that 64 consecutive rows hold both factors of 32 silu*mul outputs)
    struct Slot { QWeight q; float *f = nullptr; int64_t n = 0; bool is_q = false; int chunk = 0; int64_t row0 = 0, stride = 0, rows = 0; };
    bool lookup(const char *name, Slot &s, int &slot_id);
    int n_slots() const { return 3 + 9 * hp.n_layer; }
};

struct b200_session {
    b200_model *m = nullptr;
    b200_session_config cfg;
    int n_past = 0;
    __half *memory_k = nullptr, *memory_v = nullptr;     // [n_layer][n_ctx][gqa] and [n_layer][gqa][n_ctx] (V transposed)
    // activations (sized for n_batch rows)
    int32_t *d_tokens = nullptr;
    float *x = nullptr, *cur = nullptr, *ff = nullptr, *qkv = nullptr, *kq = nullptr, *h13 = nullptr, *hmul = nullptr, *logits = nullptr;
    int32_t *topk = nullptr;            // 1024 ids + 1024 logits (b200_session_top_k)
    int8_t *xq = nullptr; float2 *xds = nullptr; int4 *xpack = nullptr; __half *xh = nullptr;
    // pinned host staging
    int32_t *h_tokens = nullptr; float *h_logits = nullptr; int32_t *h_topk = nullptr;
    cudaEvent_t tokens_uploaded = nullptr;   // guards reuse of h_tokens by the next evaluate()
    int last_launches = 0;
    int last_n = 0;
    // debug taps (tests): copy one intermediate buffer of (layer, stage) aside during forward()
    // one-launch-per-token decode kernel (decode.cu)
    unsigned long long *d_prof = nullptr;
    DecodeLayer *d_layers = nullptr; unsigned int *d_bar = nullptr; int *d_n_past = nullptr; int *h_n_past = nullptr;
    float *qbuf = nullptr, *attn = nullptr; int4 *xpack_d = nullptr, *xpack_f = nullptr;
    int dev_n_past = -1;             // value currently held by *d_n_past (-1: unknown)
    bool mega_ok = false; int mega_grid = 0;
    std::vector<DecodeLayer> h_layers;                 // host copy of the layer table (kernel arguments of the decode graph)
    int4 *xpack_a = nullptr;
    bool decode_warm = false;                          // first decode step runs eagerly (sets kernel attributes), later ones replay a graph
    // instantiated decode graph per n_kv bucket, with its kernel count: buckets past 3072 positions run the two-kernel attention (one more per layer)
    struct DecodeGraph { int bucket; cudaGraphExec_t exec; int nodes; };
    std::vector<DecodeGraph> graphs;
    DecodeParams dp;
    int tap_layer = -2, tap_stage = 0;
    float *tap = nullptr; size_t tap_cap = 0, tap_count = 0;
    // tensor parallelism: the exchange slab (x | ff | records | logits | flags), [epoch, timeouts, CTA-arrival counters], peers' slabs mapped through CUDA IPC
    char *tp_slab = nullptr; size_t tp_slab_bytes = 0; unsigned *tp_state = nullptr;
    void *tp_peer_map[TP_MAX] = {};
    bool tp_connected = false;
};

bool b200_model::lookup(const char *name, Slot &s, int &slot_id) {
    const int e = hp.n_embd;
    const int eq = e_loc, f = f_loc;          // local row counts (== n_embd, n_ff on a single GPU)
    const int gqa = gqa_loc;
    s = Slot();
    if (!strcmp(name, "tok_embeddings.weight")) { s.q = wte; s.is_q = true; slot_id = 0; return true; }
    if (!strcmp(name, "norm.weight")) { s.f = norm; s.n = e; slot_id = 1; return true; }
    if (!strcmp(name, "output.weight")) { s.q = output; s.is_q = true; slot_id = 2; return true; }
    int il = -1; char sub[64];
    if (sscanf(name, "layers.%d.%63s", &il, sub) != 2 || il < 0 || il >= hp.n_layer) return false;
    Layer &L = layers[il];
    const int base = 3 + 9 * il;
    if (!strcmp(sub, "attention_norm.weight")) { s.f = L.attention_norm; s.n = e; slot_id = base + 0; return true; }
    if (!strcmp(sub, "ffn_norm.weight"))       { s.f = L.ffn_norm; s.n = e; slot_id = base + 1; return true; }
    s.is_q = true;
    if (!strcmp(sub, "attention.wq.weight")) { s.q = row_view(L.wqkv, 0, eq); slot_id = base + 2; return true; }
    if (!strcmp(sub, "attention.wk.weight")) { s.q = row_view(L.wqkv, eq, gqa); slot_id = base + 3; return true; }
    if (!strcmp(sub, "attention.wv.weight")) { s.q = row_view(L.wqkv, eq + gqa, gqa); slot_id = base + 4; return true; }
    if (!strcmp(sub, "attention.wo.weight")) { s.q = L.wo; slot_id = base + 5; return true; }
    if (!strcmp(sub, "feed_forward.w1.weight")) { s.q = L.w13; s.chunk = 32; s.row0 = 0;  s.stride = 64; s.rows = f; slot_id = base + 6; return true; }
    if (!strcmp(sub, "feed_forward.w3.weight")) { s.q = L.w13; s.chunk = 32; s.row0 = 32; s.stride = 64; s.rows = f; slot_id = base + 7; return true; }
    if (!strcmp(sub, "feed_forward.w2.weight")) { s.q = L.w2; slot_id = base + 8; return true; }
    return false;
}

namespace {

// ---- the forward pass (crates/models/llama/src/lib.rs:166-362) ---------------------------------------------------------------
struct Launches { int n = 0; };
}  // namespace
void silu_mul_rows(const float *h13, float *out, int64_t f, int64_t n, cudaStream_t st);
// B200_PREFILL_GEMM=mma selects the round-1 mma.sync kernel for every batch size (default: tcgen05 for batches >= 96 tokens)
namespace b200 {
bool prefill_gemm_tc5() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("B200_PREFILL_GEMM"); v = (e && !strcmp(e, "mma")) ? 0 : 1; }
    return v != 0;
}
}  // namespace b200

namespace {

// ggml_mul_mat(w, x): quantize the f32 activation rows (the INIT phase of ggml_compute_forward_mul_mat) and multiply
void matmul(b200_session *s, const QWeight &w, const float *x, float *dst, int64_t ldd, int64_t B, const float *addend, int64_t lda,
            cudaStream_t st, Launches &L, bool fast) {
    if (B == 1 && !fast && mmv_exact_stream_supported(w)) {
        quantize_act_pack(w.type, x, s->xpack, w.K, st);
        mul_mat_vec_q_exact_stream(w, s->xpack, dst, addend, st);
        L.n += 2;
        return;
    }
    if (!fast && B >= 16) {                          // prefill: bit-exact, block dots on tensor cores
        if (prefill_gemm_tc5() && B >= 96) {         // tcgen05 / TMEM / TMA kernel: 128-token tiles (exact_tc5.cu)
            quantize_act_f16_rm(vec_dot_type(w.type), x, w.K, s->xh, s->xds, w.K, B, st);
            mul_mat_q_exact_tc5(w, s->xh, s->xds, dst, ldd, B, addend, lda, st);
        } else {                                     // mma.sync kernel: 64-token tiles, better for short batches (exact_mma.cu)
            quantize_act_f16(vec_dot_type(w.type), x, w.K, s->xh, s->xds, w.K, B, st);
            mul_mat_q_exact_mma(w, s->xh, s->xds, dst, ldd, B, addend, lda, st);
        }
        L.n += 2;
        return;
    }
    quantize_act(vec_dot_type(w.type), x, w.K, s->xq, s->xds, w.K, B, st);
    if (!fast)       mul_mat_q_exact(w, s->xq, s->xds, dst, ldd, B, addend, lda, st);
    else if (B == 1) mul_mat_vec_q(w, s->xq, s->xds, dst, addend, st);
    else if (B < 16) mul_mat_q_simple(w, s->xq, s->xds, dst, ldd, B, addend, lda, st);
    else if (prefill_gemm_tc5() && B >= 64) { cvt_act_f16(x, w.K, s->xh, w.K, B, st); mul_mat_q_fast_tc5(w, s->xh, dst, ldd, B, addend, lda, st); }   // fused dequant -> tcgen05 GEMM
    else             mul_mat_q(w, s->xq, s->xds, dst, ldd, B, addend, lda, st);
    L.n += 2;
}

// all_rows == false: only the last row goes through the final norm and the lm_head (OutputRequest without all_logits reads nothing else:
// model/common.rs:6-39); rows are independent, so that row is bit-identical to the all-rows pass.
void forward(b200_session *s, int n, bool all_rows = true) {
    b200_model *m = s->m;
    const b200_llama_hparams &hp = m->hp;
    cudaStream_t st = rt().stream;
    const int e = hp.n_embd, f = hp.n_ff, hd = m->hd, gqa = m->gqa, n_head = hp.n_head, n_head_kv = hp.n_head_kv;
    const int n_ctx = hp.context_size, n_past = s->n_past, n_kv = n_past + n;
    const int qkv_ld = e + 2 * gqa;
    const float kq_scale = 1.0f / sqrtf((float)e / (float)n_head);                           // llama lib.rs:268-270
    const RopeTable &rope = rope_table(hp.n_rot, 0, hp.rope_freq_base, hp.rope_freq_scale, hd, n_ctx);
    Launches L;
    const bool tp = m->tp_world > 1;
    const bool fast = !tp && (s->cfg.flags & B200_SESSION_FAST) != 0;
    if (tp && (n != 1 || !s->tp_connected)) { fprintf(stderr, "llm_b200: tensor-parallel sessions decode one token per step, after b200_session_tp_connect\n"); exit(1); }
    if (n == 1 && s->mega_ok && !fast && (tp || (!(s->cfg.flags & B200_SESSION_UNFUSED) && s->tap_layer == -2))) {
        if (s->dev_n_past != n_past) {                 // after a prefill / rewind the device copy of n_past is stale
            B200_CHECK(cudaStreamSynchronize(st));      // (the pinned staging word may still be in flight)
            *s->h_n_past = n_past;
            B200_CHECK(cudaMemcpyAsync(s->d_n_past, s->h_n_past, sizeof(int), cudaMemcpyHostToDevice, st));
        }
        if (!tp && (s->cfg.flags & B200_SESSION_MEGA)) {
            // experimental: the whole token in one persistent cooperative kernel (decode.cu)
            if (launch_decode(s->dp, hp.wtype, st, &s->mega_grid)) {
                s->dev_n_past = n_past + 1;
                s->last_launches = 1; s->last_n = 1; s->n_past += 1;
                return;
            }
            s->mega_ok = false;
        } else {
            // default: 7 fused kernels per layer, replayed from one CUDA graph per token (decode_ops.cu)
            int bucket = ((n_kv + 255) / 256) * 256; if (bucket > n_ctx) bucket = n_ctx;
            int nodes = 0;
            if (!s->decode_warm || (s->cfg.flags & B200_SESSION_NO_GRAPH)) {
                decode_ops_enqueue(s->dp, s->h_layers, hp.wtype, bucket, s->xpack_a, st, &nodes);
                s->decode_warm = true;
            } else {
                const b200_session::DecodeGraph *g = nullptr;
                for (auto &c : s->graphs) if (c.bucket == bucket) g = &c;
                if (!g) {
                    cudaGraph_t graph;
                    cudaGraphExec_t exec;
                    B200_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                    decode_ops_enqueue(s->dp, s->h_layers, hp.wtype, bucket, s->xpack_a, st, &nodes);
                    B200_CHECK(cudaStreamEndCapture(st, &graph));
                    B200_CHECK(cudaGraphInstantiate(&exec, graph, 0));
                    B200_CHECK(cudaGraphDestroy(graph));
                    s->graphs.push_back({bucket, exec, nodes});
                    g = &s->graphs.back();
                }
                nodes = g->nodes;
                B200_CHECK(cudaGraphLaunch(g->exec, st));
            }
            s->dev_n_past = n_past + 1;
            s->last_launches = nodes; s->last_n = 1; s->n_past += 1;
            return;
        }
    }
    int il = -1;
    auto TAP = [&](int stage, const float *buf, size_t count) {
        if (s->tap_layer != il || s->tap_stage != stage) return;
        if (count > s->tap_cap) { if (s->tap) B200_CHECK(cudaFree(s->tap)); B200_CHECK(cudaMalloc(&s->tap, count * 4)); s->tap_cap = count; }
        B200_CHECK(cudaMemcpyAsync(s->tap, buf, count * 4, cudaMemcpyDeviceToDevice, st));
        s->tap_count = count;
    };

    get_rows_q(m->wte, s->d_tokens, s->x, n, st); L.n++;                                      // :170
    for (il = 0; il < hp.n_layer; il++) {
        const Layer &ly = m->layers[il];
        __half *Kl = s->memory_k + (size_t)il * n_ctx * gqa;                                  // :227-231
        __half *Vl = s->memory_v + (size_t)il * n_ctx * gqa;                                  // :233-239
        rms_norm(s->x, s->cur, ly.attention_norm, e, n, 5e-6f, st); L.n++;                    // :183,186
        TAP(1, s->cur, (size_t)n * e);
        matmul(s, ly.wqkv, s->cur, s->qkv, qkv_ld, n, nullptr, 0, st, L, fast);                // :194,208,223
        TAP(2, s->qkv, (size_t)n * qkv_ld);
        // RoPE on Q and K heads in place: [hd, n_head + n_head_kv, n] with row stride qkv_ld    :190-217
        rope_f32(s->qkv, s->qkv, hd, n_head + n_head_kv, n, hd, qkv_ld, hd, qkv_ld, n_past, rope, st); L.n++;
        TAP(3, s->qkv, (size_t)n * qkv_ld);
        {   // store K (row per position) and V (transposed) into the f16 cache                   :243-244
            StridedDesc sk{{gqa, n, 1, 1}, {4, (int64_t)qkv_ld * 4, 0, 0}}, dk{{gqa, n, 1, 1}, {2, (int64_t)gqa * 2, 0, 0}};
            cpy_strided(s->qkv + e, T_F32, sk, Kl + (size_t)n_past * gqa, T_F16, dk, st); L.n++;
            StridedDesc sv{{n, gqa, 1, 1}, {(int64_t)qkv_ld * 4, 4, 0, 0}}, dv{{n, gqa, 1, 1}, {2, (int64_t)n_ctx * 2, 0, 0}};
            cpy_strided(s->qkv + e + gqa, T_F32, sv, Vl + n_past, T_F16, dv, st); L.n++;
        }
        // KQ[h][i][j] = K[j][h] . f16(Q[i][h])                                                    :246-265
        if (fast) mul_mat_f16(Kl, hd, n_kv, n_head_kv, (int64_t)gqa * 2, (int64_t)hd * 2,
                              s->qkv, n, n_head, (int64_t)qkv_ld * 4, (int64_t)hd * 4,
                              s->kq, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4, st);
        else mul_mat_f16_exact(Kl, hd, n_kv, n_head_kv, (int64_t)gqa * 2, (int64_t)hd * 2,
                               s->qkv, n, n_head, (int64_t)qkv_ld * 4, (int64_t)hd * 4,
                               s->kq, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4, n_past, st);
        L.n++;
        TAP(4, s->kq, (size_t)n_head * n * n_kv);
        soft_max(s->kq, s->kq, n_kv, (int64_t)n_head * n, n, kq_scale, true, n_past, true, true, st); L.n++;   // :268-281
        TAP(5, s->kq, (size_t)n_head * n * n_kv);
        // KQV[h][i][c] = V[h][c][:] . f16(P[h][i][:]) written straight into the merged [n][e] layout     :284-307
        if (fast) mul_mat_f16(Vl, n_kv, hd, n_head_kv, (int64_t)n_ctx * 2, (int64_t)n_ctx * hd * 2,
                              s->kq, n, n_head, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4,
                              s->cur, (int64_t)e * 4, (int64_t)hd * 4, st);
        else mul_mat_f16_exact(Vl, n_kv, hd, n_head_kv, (int64_t)n_ctx * 2, (int64_t)n_ctx * hd * 2,
                               s->kq, n, n_head, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4,
                               s->cur, (int64_t)e * 4, (int64_t)hd * 4, -1, st);
        L.n++;
        TAP(6, s->cur, (size_t)n * e);
        matmul(s, ly.wo, s->cur, s->ff, e, n, s->x, e, st, L, fast);                           // :310,314  (inpFF = wo.cur + inpSA)
        TAP(7, s->ff, (size_t)n * e);
        rms_norm(s->ff, s->cur, ly.ffn_norm, e, n, 5e-6f, st); L.n++;                         // :318,321
        TAP(8, s->cur, (size_t)n * e);
        matmul(s, ly.w13, s->cur, s->h13, 2 * f, n, nullptr, 0, st, L, fast);                  // :323,325
        TAP(9, s->h13, (size_t)n * 2 * f);
        silu_mul_rows(s->h13, s->hmul, f, n, st); L.n++;                                      // :328,330  silu(w1 x) * (w3 x)
        TAP(10, s->hmul, (size_t)n * f);
        matmul(s, ly.w2, s->hmul, s->x, e, n, s->ff, e, st, L, fast);                          // :332,334
        TAP(11, s->x, (size_t)n * e);
    }
    il = -1;
    if (all_rows || n == 1 || s->tap_layer != -2) {
        rms_norm(s->x, s->cur, m->norm, e, n, 5e-6f, st); L.n++;                              // :343,346
        matmul(s, m->output, s->cur, s->logits, hp.n_vocab, n, nullptr, 0, st, L, fast);       // :352
    } else {
        const size_t last = (size_t)(n - 1);
        rms_norm(s->x + last * e, s->cur + last * e, m->norm, e, 1, 5e-6f, st); L.n++;
        matmul(s, m->output, s->cur + last * e, s->logits + last * hp.n_vocab, hp.n_vocab, 1, nullptr, 0, st, L, fast);
    }
    s->last_launches = L.n;
    s->last_n = n;
    s->n_past += n;                                                                           // inference_session.rs:288
}

}  // namespace

// silu(a)*b over rows of [w1 x | w3 x] interleaved in 32-column pieces: h1[c] at (c/32)*64 + c%32, h3[c] 32 further
__global__ void silu_mul_rows_kernel(const uint16_t *__restrict__ t, const float *__restrict__ h13, float *__restrict__ out, int64_t f, int64_t total) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int64_t r = i / f, c = i - r * f;
    const int64_t o = r * 2 * f + (c >> 5) * 64 + (c & 31);
    const float a = h13[o], b = h13[o + 32];
    out[i] = __fmul_rn(f16_bits_to_f32(__ldg(t + f32_to_f16_bits(a))), b);
}
void silu_mul_rows(const float *h13, float *out, int64_t f, int64_t n, cudaStream_t st) {
    const int64_t total = f * n;
    if (total == 0) return;
    silu_mul_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(luts().silu, h13, out, f, total);
    B200_CHECK(cudaGetLastError());
}

// ==== exported C ABI ==========================================================================================================
extern "C" {

int b200_init(int device) {
    Runtime &R = rt();
    if (!R.inited) R.device = device;
    R.ensure_init();
    return R.device == device ? B200_OK : B200_ERR_BAD_ARG;
}

int b200_device_info(int32_t *sm_count, size_t *free_bytes, size_t *total_bytes) {
    rt().ensure_init();
    if (sm_count) *sm_count = rt().sm_count;
    size_t fr = 0, tot = 0;
    B200_CHECK(cudaMemGetInfo(&fr, &tot));
    if (free_bytes) *free_bytes = fr;
    if (total_bytes) *total_bytes = tot;
    return B200_OK;
}

void *b200_stream(void) { rt().ensure_init(); return (void *)rt().stream; }

static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
int b200_timing_begin(void) {
    rt().ensure_init();
    if (!g_ev0) { B200_CHECK(cudaEventCreate(&g_ev0)); B200_CHECK(cudaEventCreate(&g_ev1)); }
    B200_CHECK(cudaEventRecord(g_ev0, rt().stream));
    return B200_OK;
}
float b200_timing_end_ms(void) {
    B200_CHECK(cudaEventRecord(g_ev1, rt().stream));
    B200_CHECK(cudaEventSynchronize(g_ev1));
    float ms = 0.f;
    B200_CHECK(cudaEventElapsedTime(&ms, g_ev0, g_ev1));
    return ms;
}

float b200_session_probe_matvec(b200_session *s, int32_t reps, int64_t *launches, double *bytes) {
    if (!s || reps < 1 || s->m->tp_world > 1) return -1.f;
    b200_model *m = s->m;
    cudaStream_t st = rt().stream;
    const int e = m->hp.n_embd, f = m->hp.n_ff;
    // a valid quantized activation row for both K = n_embd and K = n_ff
    const bool fast = (s->cfg.flags & B200_SESSION_FAST) != 0;
    B200_CHECK(cudaMemsetAsync(s->hmul, 0, (size_t)f * 4, st));
    quantize_act(vec_dot_type(m->hp.wtype), s->hmul, f, s->xq, s->xds, f, 1, st);
    quantize_act_pack(m->hp.wtype, s->hmul, s->xpack, f, st);
    (void)e;
    int64_t n = 0;
    auto mv = [&](const QWeight &w, float *out) {
        if (fast) mul_mat_vec_q(w, s->xq, s->xds, out, nullptr, st);
        else if (mmv_exact_stream_supported(w)) mul_mat_vec_q_exact_stream(w, s->xpack, out, nullptr, st);
        else mul_mat_q_exact(w, s->xq, s->xds, out, w.N, 1, nullptr, 0, st);
        n++;
    };
    auto pass = [&]() {
        for (auto &L : m->layers) { mv(L.wqkv, s->qkv); mv(L.wo, s->ff); mv(L.w13, s->h13); mv(L.w2, s->cur); }
        mv(m->output, s->logits);
    };
    pass();                      // warm-up (also first-touch of every page)
    n = 0;
    b200_timing_begin();
    for (int r = 0; r < reps; r++) pass();
    const float ms = b200_timing_end_ms();
    if (launches) *launches = n;
    if (bytes) *bytes = (double)m->weight_bytes * reps;
    return ms;
}

static b200_model *llama_new_impl(const b200_llama_hparams *hp, int tp_rank, int tp_world) {
    if (!hp || !is_quant(hp->wtype) || hp->n_embd % 64 || hp->n_ff % 64 || hp->n_head <= 0 || hp->n_head_kv <= 0 ||
        hp->n_head % hp->n_head_kv || hp->n_embd % hp->n_head || hp->n_layer <= 0 || hp->context_size <= 0) return nullptr;
    const int G = tp_world;
    if (G < 1 || G > TP_MAX || tp_rank < 0 || tp_rank >= G) return nullptr;
    const int gqa_full = hp->n_embd / (hp->n_head / hp->n_head_kv);
    // row split: whole heads per rank, 32-row pieces of w1|w3 and of the lm_head, 32-element blocks of wo / w2's output slices
    if (G > 1 && (hp->n_head % G || hp->n_head_kv % G || (hp->n_ff / G) % 32 || hp->n_ff % G || (hp->n_embd / G) % 32 || hp->n_vocab % G || (hp->n_vocab / G) % 32)) return nullptr;
    rt().ensure_init();
    b200_model *m = new b200_model();
    m->hp = *hp;
    if (m->hp.rope_freq_base == 0.f) m->hp.rope_freq_base = 10000.0f;
    if (m->hp.rope_freq_scale == 0.f) m->hp.rope_freq_scale = 1.0f;
    const int e = hp->n_embd, v = hp->n_vocab, t = hp->wtype;
    m->hd = e / hp->n_head;
    m->gqa = gqa_full;
    m->tp_rank = tp_rank; m->tp_world = G;
    m->e_loc = e / G; m->gqa_loc = gqa_full / G; m->f_loc = hp->n_ff / G; m->v_loc = v / G;
    m->layers.resize(hp->n_layer);
    // pass 1: sizes, pass 2: carve
    for (int pass = 0; pass < 2; pass++) {
        size_t off = 0;
        auto carve_q = [&](QWeight &w, int64_t K, int64_t N) {
            const size_t b = qweight_layout(w, t, K, N, pass ? m->slab + off : nullptr);
            off += b;
            if (pass) m->weight_bytes += (size_t)N * (K / QK) * ggml_block_bytes(t);
        };
        auto carve_f = [&](float *&p, int64_t n) { if (pass) p = (float *)(m->slab + off); off += ((size_t)n * 4 + 255) & ~(size_t)255; };
        carve_q(m->wte, e, v); carve_q(m->output, e, m->v_loc); carve_f(m->norm, e);
        for (auto &L : m->layers) {
            carve_f(L.attention_norm, e); carve_f(L.ffn_norm, e);
            carve_q(L.wqkv, e, m->e_loc + 2 * m->gqa_loc); carve_q(L.wo, e, m->e_loc); carve_q(L.w13, e, 2 * m->f_loc); carve_q(L.w2, hp->n_ff, m->e_loc);
        }
        if (!pass) { m->slab_bytes = off; B200_CHECK(cudaMalloc(&m->slab, off)); }
    }
    m->weight_bytes -= (size_t)v * (e / QK) * ggml_block_bytes(t);   // tok_embeddings is only gathered from, never streamed
    m->loaded.assign(m->n_slots(), 0);
    return m;
}

b200_model *b200_llama_new(const b200_llama_hparams *hp) { return llama_new_impl(hp, 0, 1); }

// Tensor-parallel shard `tp_rank` of `tp_world` (one process per GPU): the model's tensors keep their names, but every 2-D weight except
// tok_embeddings holds only this rank's rows -- wq / wk / wv: its heads; w1 / w3: rows [rank * n_ff/G, +n_ff/G); wo / w2: rows
// [rank * n_embd/G, +n_embd/G); output: rows [rank * n_vocab/G, +n_vocab/G) -- and b200_model_load_tensor expects exactly those rows.
b200_model *b200_llama_new_tp(const b200_llama_hparams *hp, int32_t tp_rank, int32_t tp_world) { return llama_new_impl(hp, tp_rank, tp_world); }

size_t b200_model_weight_bytes(b200_model *m) { return m ? m->weight_bytes : 0; }

static size_t slot_bytes(const b200_model::Slot &s) {
    if (!s.is_q) return (size_t)s.n * 4;
    return (size_t)(s.chunk ? s.rows : s.q.N) * s.q.nb * ggml_block_bytes(s.q.type);
}

size_t b200_model_tensor_nbytes(b200_model *m, const char *name) {
    b200_model::Slot s; int id;
    if (!m || !m->lookup(name, s, id)) return 0;
    return slot_bytes(s);
}

int b200_model_load_tensor(b200_model *m, const char *name, int32_t type, const void *host_data, size_t nbytes) {
    if (!m || !name || !host_data) return B200_ERR_BAD_ARG;
    b200_model::Slot s; int id;
    if (!m->lookup(name, s, id)) return B200_ERR_UNKNOWN_TENSOR;
    Runtime &R = rt();
    if (s.is_q) {
        if (type != s.q.type || nbytes != slot_bytes(s)) return B200_ERR_TENSOR_SHAPE;
        R.op_arena.reset();
        void *raw = R.op_arena.get(nbytes, R.stream);
        B200_CHECK(cudaMemcpyAsync(raw, host_data, nbytes, cudaMemcpyHostToDevice, R.stream));
        if (!s.chunk) repack_weights(s.q, raw, R.stream);
        else {
            const size_t piece = (size_t)s.chunk * s.q.nb * ggml_block_bytes(type);
            for (int64_t c = 0; c * s.chunk < s.rows; c++)
                repack_weights(row_view(s.q, c * s.stride + s.row0, s.chunk), (const char *)raw + c * piece, R.stream);
        }
        B200_CHECK(cudaStreamSynchronize(R.stream));
    } else {
        if (type != T_F32 || nbytes != (size_t)s.n * 4) return B200_ERR_TENSOR_SHAPE;
        B200_CHECK(cudaMemcpy(s.f, host_data, nbytes, cudaMemcpyHostToDevice));
        B200_CHECK(cudaDeviceSynchronize());   // legacy-stream copy/memset: not ordered with our non-blocking stream, and a pageable H2D cudaMemcpy may return before its DMA lands
    }
    if (!m->loaded[id]) { m->loaded[id] = 1; m->n_loaded++; }
    return B200_OK;
}

// TensorLoader::load checks the dims too (TensorWrongSize): a file whose tensor has the right byte count but swapped / wrong dims must not load
int b200_model_load_tensor_shaped(b200_model *m, const char *name, int32_t type, int32_t n_dims, int64_t ne0, int64_t ne1, const void *host_data, size_t nbytes) {
    if (!m || !name) return B200_ERR_BAD_ARG;
    b200_model::Slot s; int id;
    if (!m->lookup(name, s, id)) return B200_ERR_UNKNOWN_TENSOR;
    if (s.is_q) { if (n_dims != 2 || ne0 != s.q.K || ne1 != (s.chunk ? s.rows : s.q.N)) return B200_ERR_TENSOR_SHAPE; }
    else if (n_dims != 1 || ne0 != s.n) return B200_ERR_TENSOR_SHAPE;
    return b200_model_load_tensor(m, name, type, host_data, nbytes);
}

int b200_model_read_tensor(b200_model *m, const char *name, void *host_out, size_t nbytes) {
    if (!m || !name || !host_out) return B200_ERR_BAD_ARG;
    b200_model::Slot s; int id;
    if (!m->lookup(name, s, id)) return B200_ERR_UNKNOWN_TENSOR;
    Runtime &R = rt();
    if (s.is_q) {
        if (nbytes != slot_bytes(s)) return B200_ERR_TENSOR_SHAPE;
        R.op_arena.reset();
        void *raw = R.op_arena.get(nbytes, R.stream);
        if (!s.chunk) unpack_weights(s.q, raw, R.stream);
        else {
            const size_t piece = (size_t)s.chunk * s.q.nb * ggml_block_bytes(s.q.type);
            for (int64_t c = 0; c * s.chunk < s.rows; c++)
                unpack_weights(row_view(s.q, c * s.stride + s.row0, s.chunk), (char *)raw + c * piece, R.stream);
        }
        B200_CHECK(cudaMemcpyAsync(host_out, raw, nbytes, cudaMemcpyDeviceToHost, R.stream));
        B200_CHECK(cudaStreamSynchronize(R.stream));
    } else {
        if (nbytes != (size_t)s.n * 4) return B200_ERR_TENSOR_SHAPE;
        B200_CHECK(cudaStreamSynchronize(R.stream));
        B200_CHECK(cudaMemcpy(host_out, s.f, nbytes, cudaMemcpyDeviceToHost));
    }
    return B200_OK;
}

int b200_model_synthesize(b200_model *m, uint64_t seed) {
    if (!m || m->tp_world > 1) return B200_ERR_BAD_ARG;       // shards are cut from a full model's tensors by the host (llm_b200/tp.py)
    cudaStream_t st = rt().stream;
    uint64_t id = 0;
    auto q = [&](const QWeight &w) { synth_qweight(w, seed + 0x1000003ull * (++id), st); };
    auto g = [&](float *p, int64_t n) { synth_gain(p, n, seed + 0x1000003ull * (++id), st); };
    q(m->wte); g(m->norm, m->hp.n_embd); q(m->output);
    for (auto &L : m->layers) { g(L.attention_norm, m->hp.n_embd); g(L.ffn_norm, m->hp.n_embd); q(L.wqkv); q(L.wo); q(L.w13); q(L.w2); }
    B200_CHECK(cudaStreamSynchronize(st));
    m->loaded.assign(m->n_slots(), 1);
    m->n_loaded = m->n_slots();
    return B200_OK;
}

int b200_model_is_loaded(b200_model *m) { return m && m->n_loaded == m->n_slots(); }

void b200_model_free(b200_model *m) {
    if (!m) return;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    if (m->slab) B200_CHECK(cudaFree(m->slab));
    delete m;
}

// ---- tensor-parallel session: decode only (prompts are fed token by token), activations that cross GPUs live in ONE exchange slab -------------
static b200_session *start_session_tp(b200_session *s) {
    b200_model *m = s->m;
    const b200_llama_hparams &hp = m->hp;
    const int G = m->tp_world, r = m->tp_rank;
    const size_t e = hp.n_embd, f = hp.n_ff, n_ctx = hp.context_size, gqa = m->gqa_loc, V = hp.n_vocab;
    s->cfg.n_batch = s->cfg.n_batch < 1 ? 1 : s->cfg.n_batch;
    const size_t kv_elems = (size_t)hp.n_layer * n_ctx * gqa;
    B200_CHECK(cudaMalloc(&s->memory_k, kv_elems * 2));
    B200_CHECK(cudaMalloc(&s->memory_v, kv_elems * 2));
    B200_CHECK(cudaMemset(s->memory_k, 0, kv_elems * 2));
    B200_CHECK(cudaMemset(s->memory_v, 0, kv_elems * 2));
    B200_CHECK(cudaMalloc(&s->d_tokens, (size_t)s->cfg.n_batch * 4));
    B200_CHECK(cudaMallocHost(&s->h_tokens, (size_t)s->cfg.n_batch * 4));
    B200_CHECK(cudaMallocHost(&s->h_logits, (size_t)s->cfg.n_batch * V * 4));
    B200_CHECK(cudaMallocHost(&s->h_topk, 2048 * 4));
    B200_CHECK(cudaMalloc(&s->topk, 2048 * 4));
    B200_CHECK(cudaEventCreateWithFlags(&s->tokens_uploaded, cudaEventDisableTiming));
    B200_CHECK(cudaMalloc(&s->qbuf, (size_t)m->e_loc * 4));
    B200_CHECK(cudaMalloc(&s->xpack_a, (e / QK) * 64));
    B200_CHECK(cudaMalloc(&s->d_n_past, sizeof(int)));
    B200_CHECK(cudaMallocHost(&s->h_n_past, sizeof(int)));
    B200_CHECK(cudaMalloc(&s->d_prof, B200_PROF_SLOTS * 9 * sizeof(unsigned long long)));
    B200_CHECK(cudaMemset(s->d_prof, 0, B200_PROF_SLOTS * 9 * sizeof(unsigned long long)));
    // the exchange slab: arrays of 8-byte {word, tag} units (tp.cuh) -- x | ff | attention records | ffn records | logits, 256-byte aligned pieces
    TpCtx &T = s->dp.tp;
    T = TpCtx();
    T.world = G; T.rank = r; T.vmul = (unsigned)hp.n_layer + 1;
    { const char *e = getenv("B200_TP_RELAX"); T.relax = e ? atoi(e) : 0; }
    size_t off = 0;
    auto piece = [&](size_t units) { const size_t o = off; off += (units * 8 + 255) & ~(size_t)255; return (uint32_t)o; };
    T.off[TPB_X] = piece(e); T.off[TPB_FF] = piece(e); T.off[TPB_XD] = piece((e / QK) * 16); T.off[TPB_XF] = piece((f / QK) * 16); T.off[TPB_LOGITS] = piece(V);
    s->tp_slab_bytes = off;
    B200_CHECK(cudaMalloc(&s->tp_slab, off));
    B200_CHECK(cudaMemset(s->tp_slab, 0, off));                           // tag 0 never matches
    B200_CHECK(cudaMalloc(&s->tp_state, 2 * sizeof(unsigned)));
    B200_CHECK(cudaMemset(s->tp_state, 0, 2 * sizeof(unsigned)));
    T.epoch = s->tp_state;
    for (int p = 0; p < TP_MAX; p++) T.peer[p] = nullptr;
    T.peer[r] = s->tp_slab;                                              // peers are mapped by b200_session_tp_connect
    B200_CHECK(cudaMalloc(&s->x, e * 4));                                 // the embedding row (plain f32) before it is spread into the X units
    B200_CHECK(cudaMalloc(&s->logits, V * 4));                            // the gathered logits, plain f32 for the host
    s->ff = nullptr; s->xpack_d = nullptr; s->xpack_f = nullptr;
    const RopeTable &rt_ = rope_table(hp.n_rot, 0, hp.rope_freq_base, hp.rope_freq_scale, m->hd, (int)n_ctx);
    {
        std::vector<DecodeLayer> hl(hp.n_layer);
        for (int il = 0; il < hp.n_layer; il++) {
            const Layer &L = m->layers[il];
            hl[il] = DecodeLayer{L.wqkv, L.wo, L.w13, L.w2, L.attention_norm, L.ffn_norm,
                                 s->memory_k + (size_t)il * n_ctx * gqa, s->memory_v + (size_t)il * n_ctx * gqa};
        }
        s->h_layers = hl;
    }
    DecodeParams &P = s->dp;
    P.layers = nullptr; P.n_layer = hp.n_layer; P.wte = m->wte; P.output = m->output; P.norm = m->norm;
    P.e = (int)e; P.f = m->f_loc; P.hd = m->hd; P.gqa = m->gqa_loc; P.n_head = hp.n_head / G; P.n_head_kv = hp.n_head_kv / G; P.n_ctx = (int)n_ctx; P.n_vocab = m->v_loc;
    P.kq_scale = 1.0f / sqrtf((float)hp.n_embd / (float)hp.n_head); P.eps = 5e-6f;
    P.rope_cs = rt_.cs; P.rope_half = rt_.half;
    P.lut_silu = luts().silu; P.lut_exp = luts().exp;
    P.token = s->d_tokens; P.n_past = s->d_n_past;
    P.x = s->x; P.q = s->qbuf; P.kq = nullptr; P.attn = nullptr; P.ff = s->ff; P.h13 = nullptr; P.logits = s->logits;
    P.xpack_d = s->xpack_d; P.xpack_f = s->xpack_f; P.bar = nullptr; P.scratch_bytes = 0;
    P.e_loc = m->e_loc; P.head0 = r * (hp.n_head / G); P.n_vocab_full = hp.n_vocab;
    P.row0_e = (int64_t)r * m->e_loc; P.row0_w13 = (int64_t)r * 2 * m->f_loc; P.row0_v = (int64_t)r * m->v_loc;
    P.prof = nullptr;
    QWeight probe; probe.nb = (int64_t)e / QK;
    QWeight probe2; probe2.nb = (int64_t)f / QK;
    s->mega_ok = hp.n_rot == m->hd && (m->hd == 64 || m->hd == 128) && mmv_exact_stream_supported(probe) && mmv_exact_stream_supported(probe2) &&
                 m->gqa_loc % 32 == 0 && m->e_loc % 32 == 0 && hp.context_size % 8 == 0;
    B200_CHECK(cudaDeviceSynchronize());
    if (!s->mega_ok) { fprintf(stderr, "llm_b200: tensor-parallel session: geometry not supported by the fused decode schedule\n"); b200_session_free(s); return nullptr; }
    // the ranks exchange attention rows in the cluster attention's epilogue, so every context bucket must fit it; the largest one is n_ctx itself
    if (!attn_fused_fits((int)n_ctx, m->hd)) {
        fprintf(stderr, "llm_b200: tensor-parallel session: context_size %d not supported by the fused decode attention (shared memory)\n", (int)n_ctx);
        b200_session_free(s); return nullptr;
    }
    return s;
}

b200_session *b200_model_start_session(b200_model *m, const b200_session_config *cfg) {
    if (!m || !cfg || cfg->n_batch < 1) return nullptr;
    if (m->n_loaded != m->n_slots()) { fprintf(stderr, "llm_b200: start_session: %d of %d tensors loaded\n", m->n_loaded, m->n_slots()); return nullptr; }
    b200_session *s = new b200_session();
    s->m = m; s->cfg = *cfg;
    if (m->tp_world > 1) return start_session_tp(s);
    const b200_llama_hparams &hp = m->hp;
    const size_t e = hp.n_embd, f = hp.n_ff, B = cfg->n_batch, n_ctx = hp.context_size, gqa = m->gqa;
    const size_t kv_elems = (size_t)hp.n_layer * n_ctx * gqa;
    B200_CHECK(cudaMalloc(&s->memory_k, kv_elems * 2));
    B200_CHECK(cudaMalloc(&s->memory_v, kv_elems * 2));
    B200_CHECK(cudaMemset(s->memory_k, 0, kv_elems * 2));           // offload_no_scratch zero-fills (LC/ggml-cuda.cu:3967-3973)
    B200_CHECK(cudaMemset(s->memory_v, 0, kv_elems * 2));
    const size_t kmax = e > f ? e : f;
    B200_CHECK(cudaMalloc(&s->d_tokens, B * 4));
    B200_CHECK(cudaMalloc(&s->x, B * e * 4));
    B200_CHECK(cudaMalloc(&s->cur, B * e * 4));
    B200_CHECK(cudaMalloc(&s->ff, B * e * 4));
    B200_CHECK(cudaMalloc(&s->qkv, B * (e + 2 * gqa) * 4));
    B200_CHECK(cudaMalloc(&s->kq, (size_t)hp.n_head * B * n_ctx * 4));
    B200_CHECK(cudaMalloc(&s->h13, B * 2 * f * 4));
    B200_CHECK(cudaMalloc(&s->hmul, B * f * 4));
    B200_CHECK(cudaMalloc(&s->logits, B * (size_t)hp.n_vocab * 4));
    B200_CHECK(cudaMalloc(&s->xq, B * kmax));
    B200_CHECK(cudaMalloc(&s->topk, 2048 * 4));
    B200_CHECK(cudaMalloc(&s->xds, B * (kmax / QK) * sizeof(float2)));
    B200_CHECK(cudaMalloc(&s->xpack, (kmax / QK) * 64));
    B200_CHECK(cudaMalloc(&s->xh, xh_bytes(kmax, B)));
    B200_CHECK(cudaMallocHost(&s->h_tokens, B * 4));
    B200_CHECK(cudaMallocHost(&s->h_logits, B * (size_t)hp.n_vocab * 4));
    B200_CHECK(cudaMallocHost(&s->h_topk, 2048 * 4));
    B200_CHECK(cudaEventCreateWithFlags(&s->tokens_uploaded, cudaEventDisableTiming));
    const RopeTable &rt_ = rope_table(hp.n_rot, 0, hp.rope_freq_base, hp.rope_freq_scale, m->hd, (int)n_ctx);
    // decode kernel parameters
    B200_CHECK(cudaMalloc(&s->qbuf, e * 4));
    B200_CHECK(cudaMalloc(&s->attn, e * 4));
    B200_CHECK(cudaMalloc(&s->d_bar, 2 * sizeof(unsigned int)));
    B200_CHECK(cudaMemset(s->d_bar, 0, 2 * sizeof(unsigned int)));
    B200_CHECK(cudaMalloc(&s->d_n_past, sizeof(int)));
    B200_CHECK(cudaMallocHost(&s->h_n_past, sizeof(int)));
    {
        std::vector<DecodeLayer> hl(hp.n_layer);
        for (int il = 0; il < hp.n_layer; il++) {
            const Layer &L = m->layers[il];
            hl[il] = DecodeLayer{L.wqkv, L.wo, L.w13, L.w2, L.attention_norm, L.ffn_norm,
                                 s->memory_k + (size_t)il * n_ctx * gqa, s->memory_v + (size_t)il * n_ctx * gqa};
        }
        s->h_layers = hl;
        B200_CHECK(cudaMalloc(&s->d_layers, hl.size() * sizeof(DecodeLayer)));
        B200_CHECK(cudaMemcpy(s->d_layers, hl.data(), hl.size() * sizeof(DecodeLayer), cudaMemcpyHostToDevice));
    }
    DecodeParams &P = s->dp;
    P.layers = s->d_layers; P.n_layer = hp.n_layer; P.wte = m->wte; P.output = m->output; P.norm = m->norm;
    P.e = (int)e; P.f = (int)f; P.hd = m->hd; P.gqa = m->gqa; P.n_head = hp.n_head; P.n_head_kv = hp.n_head_kv; P.n_ctx = (int)n_ctx; P.n_vocab = hp.n_vocab;
    P.kq_scale = 1.0f / sqrtf((float)hp.n_embd / (float)hp.n_head); P.eps = 5e-6f;
    P.rope_cs = rt_.cs; P.rope_half = rt_.half;
    P.lut_silu = luts().silu; P.lut_exp = luts().exp;
    P.token = s->d_tokens; P.n_past = s->d_n_past;
    P.x = s->x; P.q = s->qbuf; P.kq = s->kq; P.attn = s->attn; P.ff = s->ff; P.h13 = s->h13; P.logits = s->logits;
    P.bar = s->d_bar;
    B200_CHECK(cudaMalloc(&s->xpack_d, (e / QK) * 64));
    B200_CHECK(cudaMalloc(&s->xpack_f, (f / QK) * 64));
    P.xpack_d = s->xpack_d; P.xpack_f = s->xpack_f;
    B200_CHECK(cudaMalloc(&s->xpack_a, (e / QK) * 64));
    P.scratch_bytes = decode_scratch_bytes((int)e, (int)f, m->hd, (int)n_ctx);
    B200_CHECK(cudaMalloc(&s->d_prof, B200_PROF_SLOTS * 9 * sizeof(unsigned long long)));
    B200_CHECK(cudaMemset(s->d_prof, 0, B200_PROF_SLOTS * 9 * sizeof(unsigned long long)));
    P.prof = getenv("B200_DECODE_PROF") ? s->d_prof : nullptr;
    s->mega_ok = hp.n_rot == m->hd && (m->hd == 64 || m->hd == 128) && decode_supported(P, hp.wtype);
    B200_CHECK(cudaDeviceSynchronize());   // the memsets / copies above ran on the legacy stream: order them before anything on the backend's non-blocking stream
    return s;
}

int32_t b200_session_n_past(const b200_session *s) { return s ? s->n_past : -1; }
int b200_session_set_n_past(b200_session *s, int32_t n_past) {
    if (!s || n_past < 0 || n_past > s->n_past) return B200_ERR_BAD_ARG;
    s->n_past = n_past;
    return B200_OK;
}
int32_t b200_session_last_launches(const b200_session *s) { return s ? s->last_launches : 0; }

int b200_session_evaluate_device(b200_session *s, const int32_t *d_tokens, int32_t n) {
    if (!s || n < 1 || n > s->cfg.n_batch) return B200_ERR_BAD_ARG;
    if (s->n_past + n > s->m->hp.context_size) return B200_ERR_CONTEXT_FULL;
    if (d_tokens && d_tokens != s->d_tokens)
        B200_CHECK(cudaMemcpyAsync(s->d_tokens, d_tokens, (size_t)n * 4, cudaMemcpyDeviceToDevice, rt().stream));
    forward(s, n);
    return B200_OK;
}
const float *b200_session_device_logits(b200_session *s) { return s ? s->logits : nullptr; }

int b200_session_evaluate(b200_session *s, const int32_t *tokens, int32_t n, float *logits_out, int32_t all_logits) {
    if (!s || !tokens || n < 1 || n > s->cfg.n_batch) return B200_ERR_BAD_ARG;
    if (s->n_past + n > s->m->hp.context_size) return B200_ERR_CONTEXT_FULL;
    if (s->m->tp_world > 1 && n > 1) {                  // tensor-parallel sessions have the decode schedule only: a batch is fed token by token
        const size_t V = s->m->hp.n_vocab;
        for (int i = 0; i < n; i++) {
            float *out = !logits_out ? nullptr : all_logits ? logits_out + (size_t)i * V : (i == n - 1 ? logits_out : nullptr);
            const int rc = b200_session_evaluate(s, tokens + i, 1, out, 0);
            if (rc != B200_OK) return rc;
        }
        return B200_OK;
    }
    for (int i = 0; i < n; i++) if (tokens[i] < 0 || tokens[i] >= s->m->hp.n_vocab) return B200_ERR_BAD_ARG;
    cudaStream_t st = rt().stream;
    B200_CHECK(cudaEventSynchronize(s->tokens_uploaded));       // the previous (feed-only) call may still be reading the staging buffer
    memcpy(s->h_tokens, tokens, (size_t)n * 4);
    B200_CHECK(cudaMemcpyAsync(s->d_tokens, s->h_tokens, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    B200_CHECK(cudaEventRecord(s->tokens_uploaded, st));
    forward(s, n, all_logits != 0);
    const size_t V = s->m->hp.n_vocab;
    if (logits_out) {
        const size_t rows = all_logits ? n : 1;
        const float *src = all_logits ? s->logits : s->logits + (size_t)(n - 1) * V;
        B200_CHECK(cudaMemcpyAsync(s->h_logits, src, rows * V * 4, cudaMemcpyDeviceToHost, st));
        B200_CHECK(cudaStreamSynchronize(st));
        memcpy(logits_out, s->h_logits, rows * V * 4);
    }
    return B200_OK;
}

// Sampler hand-off (SURVEY.md §8f-3): the k largest logits of the last evaluated row, selected on the device; 8 k bytes cross PCIe instead of
// n_vocab floats.  Order = descending logit, ties by ascending token id (what a stable descending sort of (id, logit) pairs yields: llm-samplers top-k).
int b200_session_top_k(b200_session *s, int32_t k, int32_t *ids_out, float *logits_out) {
    if (!s || !ids_out || !logits_out || k < 1 || k > 1024 || k > s->m->hp.n_vocab || s->last_n < 1) return B200_ERR_BAD_ARG;
    cudaStream_t st = rt().stream;
    const size_t V = s->m->hp.n_vocab;
    int32_t *d_ids = s->topk;
    float *d_vals = (float *)(s->topk + 1024);
    top_k_rows(s->logits + (size_t)(s->last_n - 1) * V, (int64_t)V, k, d_ids, d_vals, st);
    B200_CHECK(cudaMemcpyAsync(s->h_topk, d_ids, (size_t)k * 4, cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaMemcpyAsync(s->h_topk + 1024, d_vals, (size_t)k * 4, cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaStreamSynchronize(st));
    memcpy(ids_out, s->h_topk, (size_t)k * 4);
    memcpy(logits_out, s->h_topk + 1024, (size_t)k * 4);
    return B200_OK;
}

int b200_session_feed_prompt(b200_session *s, const int32_t *tokens, int32_t n, float *last_logits_out) {
    if (!s || !tokens || n < 0) return B200_ERR_BAD_ARG;
    if (s->n_past + n > s->m->hp.context_size) return B200_ERR_CONTEXT_FULL;          // inference_session.rs:311-313
    for (int i = 0; i < n; i += s->cfg.n_batch) {                                     // :315-316 chunks(n_batch)
        const int c = (n - i) < s->cfg.n_batch ? (n - i) : s->cfg.n_batch;
        const bool last = i + c >= n;
        const int rc = b200_session_evaluate(s, tokens + i, c, last ? last_logits_out : nullptr, 0);
        if (rc != B200_OK) return rc;
    }
    return B200_OK;
}

int b200_session_read_kv(b200_session *s, int32_t which, void *host_out, size_t nbytes) {
    if (!s || !host_out) return B200_ERR_BAD_ARG;
    const size_t kv_bytes = (size_t)s->m->hp.n_layer * s->m->hp.context_size * (s->m->tp_world > 1 ? s->m->gqa_loc : s->m->gqa) * 2;   // tensor-parallel: this rank's heads
    if (nbytes != kv_bytes) return B200_ERR_TENSOR_SHAPE;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    B200_CHECK(cudaMemcpy(host_out, which ? s->memory_v : s->memory_k, kv_bytes, cudaMemcpyDeviceToHost));
    return B200_OK;
}

int b200_session_set_tap(b200_session *s, int32_t layer, int32_t stage) {
    if (!s || s->m->tp_world > 1) return B200_ERR_BAD_ARG;
    s->tap_layer = layer; s->tap_stage = stage; s->tap_count = 0;
    return B200_OK;
}
int64_t b200_session_read_tap(b200_session *s, float *host_out, int64_t max_count) {
    if (!s || !host_out) return B200_ERR_BAD_ARG;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    const size_t c = s->tap_count < (size_t)max_count ? s->tap_count : (size_t)max_count;
    if (c) B200_CHECK(cudaMemcpy(host_out, s->tap, c * 4, cudaMemcpyDeviceToHost));
    return (int64_t)c;
}

int b200_session_decode_profile(b200_session *s, unsigned long long *out128) {
    if (!s || !out128) return B200_ERR_BAD_ARG;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    B200_CHECK(cudaMemcpy(out128, s->d_prof, 128 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return B200_OK;
}

// Per-kernel timeline of the graph decode schedule (B200_DECODE_PROF=1): slot i = the i-th launch of the token;
// out = 9 arrays of n (%globaltimer, ns): CTA begin min, CTA end max, prologue-done min, begin max, prologue-done max, first stage landed min / max,
// last stage landed max (mat-vec kernels only for the last three), unused by the mat-vecs.  The fused attention stamps its phases into arrays
// 2 / 4 (past pdl_wait, first / last CTA), 5 / 6 (KQ share done), 7 (scores exchanged, last CTA) and 8 (soft_max done, last CTA).
// reset != 0 re-arms the slots.
int b200_session_decode_timeline(b200_session *s, unsigned long long *out, int n, int reset) {
    if (!s || n < 0 || n > B200_PROF_SLOTS) return B200_ERR_BAD_ARG;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    if (out && n) {
        for (int k = 0; k < 9; k++)
            B200_CHECK(cudaMemcpy(out + (size_t)k * n, s->d_prof + (size_t)k * B200_PROF_SLOTS, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    if (reset) {                                                  // arrays 0, 2, 5 hold minima, the others maxima
        for (int k = 0; k < 9; k++)
            B200_CHECK(cudaMemset(s->d_prof + (size_t)k * B200_PROF_SLOTS, (k == 0 || k == 2 || k == 5) ? 0xFF : 0, B200_PROF_SLOTS * sizeof(unsigned long long)));
        B200_CHECK(cudaDeviceSynchronize());
    }
    return B200_OK;
}

int b200_session_sync(b200_session *s) { (void)s; B200_CHECK(cudaStreamSynchronize(rt().stream)); return B200_OK; }

// ---- tensor-parallel plumbing: exchange-slab handles (CUDA IPC; one process per GPU, handles travel over the host's own channel) --------
int b200_session_tp_handle(b200_session *s, void *handle_out64) {
    if (!s || !s->tp_slab || !handle_out64) return B200_ERR_BAD_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    B200_CHECK(cudaIpcGetMemHandle(&h, s->tp_slab));
    memcpy(handle_out64, &h, 64);
    return B200_OK;
}
int b200_session_tp_connect(b200_session *s, const void *handles_by_rank) {
    if (!s || !s->tp_slab || !handles_by_rank) return B200_ERR_BAD_ARG;
    TpCtx &T = s->dp.tp;
    for (int p = 0; p < T.world; p++) {
        if (p == T.rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles_by_rank + (size_t)p * 64, 64);
        void *ptr = nullptr;
        const cudaError_t err = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (err != cudaSuccess) { fprintf(stderr, "llm_b200: cudaIpcOpenMemHandle(rank %d): %s\n", p, cudaGetErrorString(err)); return B200_ERR_IO; }
        s->tp_peer_map[p] = ptr;
        T.peer[p] = (char *)ptr;
    }
    s->tp_connected = true;
    decode_set_tp(T, rt().stream);
    return B200_OK;
}
int b200_session_tp_set_nowait(b200_session *s, int32_t nowait) {     // measurement aid: the captured graphs carry the flag, so they are dropped
    if (!s || !s->tp_slab) return B200_ERR_BAD_ARG;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    s->dp.tp.nowait = nowait < 0 ? 0 : nowait > 2 ? 2 : nowait;
    decode_set_tp(s->dp.tp, rt().stream);
    for (auto &g : s->graphs) cudaGraphExecDestroy(g.exec);
    s->graphs.clear();
    return B200_OK;
}
int32_t b200_session_tp_timeouts(b200_session *s) {      // number of flag waits that gave up (a peer stopped): must be 0
    if (!s || !s->tp_state) return -1;
    unsigned v[2] = {0, 0};
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    B200_CHECK(cudaMemcpy(v, s->tp_state, sizeof(v), cudaMemcpyDeviceToHost));
    return (int32_t)v[1];
}

void b200_session_free(b200_session *s) {
    if (!s) return;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    if (s->h_n_past) B200_CHECK(cudaFreeHost(s->h_n_past));
    for (auto &g : s->graphs) cudaGraphExecDestroy(g.exec);
    if (s->tp_slab) {                                    // tensor-parallel session: the exchange slab and the peers' mappings
        for (int p = 0; p < TP_MAX; p++) if (s->tp_peer_map[p]) cudaIpcCloseMemHandle(s->tp_peer_map[p]);
        B200_CHECK(cudaFree(s->tp_slab)); B200_CHECK(cudaFree(s->tp_state));
    }
    void *dev[] = {s->xpack_a, s->xpack_d, s->xpack_f, s->d_prof, s->d_layers, s->d_bar, s->d_n_past, s->qbuf, s->attn, s->tap, s->memory_k, s->memory_v, s->d_tokens, s->x, s->cur, s->ff, s->qkv, s->kq, s->h13, s->hmul, s->logits, s->xq, s->xds, s->xpack, s->xh, s->topk};
    for (void *p : dev) if (p) B200_CHECK(cudaFree(p));
    if (s->h_tokens) B200_CHECK(cudaFreeHost(s->h_tokens));
    if (s->h_logits) B200_CHECK(cudaFreeHost(s->h_logits));
    if (s->h_topk) B200_CHECK(cudaFreeHost(s->h_topk));
    if (s->tokens_uploaded) B200_CHECK(cudaEventDestroy(s->tokens_uploaded));
    delete s;
}

// ---- single-op entry points on host buffers ---------------------------------------------------------------------------------
int b200_op_quantize_act(int32_t vdt, const float *x, int64_t K, int64_t B, int8_t *qs_out, float *d_out, float *aux_out) {
    if (!x || K % QK || (vdt != T_Q8_0 && vdt != T_Q8_1)) return B200_ERR_BAD_ARG;
    Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
    cudaStream_t st = R.stream;
    const size_t nblk = (size_t)B * (K / QK);
    float *dx = (float *)R.op_arena.get((size_t)B * K * 4, st);
    int8_t *dq = (int8_t *)R.op_arena.get((size_t)B * K, st);
    float2 *dds = (float2 *)R.op_arena.get(nblk * sizeof(float2), st);
    B200_CHECK(cudaMemcpyAsync(dx, x, (size_t)B * K * 4, cudaMemcpyHostToDevice, st));
    quantize_act(vdt, dx, K, dq, dds, K, B, st);
    std::vector<float2> h(nblk);
    B200_CHECK(cudaMemcpyAsync(qs_out, dq, (size_t)B * K, cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaMemcpyAsync(h.data(), dds, nblk * sizeof(float2), cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < nblk; i++) { if (d_out) d_out[i] = h[i].x; if (aux_out) aux_out[i] = h[i].y; }
    return B200_OK;
}

int b200_op_quantize_q8_K(const float *x, int64_t K, int64_t B, void *blocks_out) {      // quantize_row_q8_K of B rows -> B * K/256 block_q8_K (292 bytes each)
    if (!x || !blocks_out || K % 256) return B200_ERR_BAD_ARG;
    Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
    cudaStream_t st = R.stream;
    float *dx = (float *)R.op_arena.get((size_t)B * K * 4, st);
    void *xq = R.op_arena.get(q8k_bytes(K, B), st);
    B200_CHECK(cudaMemcpyAsync(dx, x, (size_t)B * K * 4, cudaMemcpyHostToDevice, st));
    quantize_act_q8k(dx, K, xq, K, B, st);
    B200_CHECK(cudaMemcpyAsync(blocks_out, xq, q8k_bytes(K, B), cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaStreamSynchronize(st));
    return B200_OK;
}
int b200_op_mul_mat(int32_t wtype, const void *w_ggml, int64_t K, int64_t N, const float *x, int64_t B, float *dst, int32_t impl) {
    if (is_kquant(wtype)) {                              // Q2_K .. Q6_K: one exact kernel (kquants.cu); `impl` must be AUTO or EXACT
        if (!w_ggml || !x || !dst || K % 256 || (impl != B200_MM_AUTO && impl != B200_MM_EXACT)) return B200_ERR_BAD_ARG;
        Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
        cudaStream_t st = R.stream;
        const size_t raw_bytes = (size_t)N * (K / 256) * kquant_block_bytes(wtype);
        void *raw = R.op_arena.get(raw_bytes, st);
        float *dx = (float *)R.op_arena.get((size_t)B * K * 4, st);
        float *dd = (float *)R.op_arena.get((size_t)B * N * 4, st);
        void *xq = R.op_arena.get(q8k_bytes(K, B), st);
        B200_CHECK(cudaMemcpyAsync(raw, w_ggml, raw_bytes, cudaMemcpyHostToDevice, st));
        B200_CHECK(cudaMemcpyAsync(dx, x, (size_t)B * K * 4, cudaMemcpyHostToDevice, st));
        quantize_act_q8k(dx, K, xq, K, B, st);
        mul_mat_kq_exact(wtype, raw, xq, dd, N, K, N, B, nullptr, 0, st);
        B200_CHECK(cudaMemcpyAsync(dst, dd, (size_t)B * N * 4, cudaMemcpyDeviceToHost, st));
        B200_CHECK(cudaStreamSynchronize(st));
        return B200_OK;
    }
    if (!is_quant(wtype) || !w_ggml || !x || !dst || K % 64) return B200_ERR_BAD_ARG;
    Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
    cudaStream_t st = R.stream;
    const size_t raw_bytes = (size_t)N * (K / QK) * ggml_block_bytes(wtype);
    void *raw = R.op_arena.get(raw_bytes, st);
    B200_CHECK(cudaMemcpyAsync(raw, w_ggml, raw_bytes, cudaMemcpyHostToDevice, st));
    QWeight w;
    const size_t pb = qweight_layout(w, wtype, K, N, nullptr);
    qweight_layout(w, wtype, K, N, R.op_arena.get(pb, st));
    repack_weights(w, raw, st);
    float *dx = (float *)R.op_arena.get((size_t)B * K * 4, st);
    float *dd = (float *)R.op_arena.get((size_t)B * N * 4, st);
    int8_t *xq = (int8_t *)R.op_arena.get((size_t)B * K, st);
    float2 *xds = (float2 *)R.op_arena.get((size_t)B * (K / QK) * sizeof(float2), st);
    B200_CHECK(cudaMemcpyAsync(dx, x, (size_t)B * K * 4, cudaMemcpyHostToDevice, st));
    quantize_act(vec_dot_type(wtype), dx, K, xq, xds, K, B, st);
    if (impl == B200_MM_AUTO) impl = B200_MM_EXACT;
    if (impl == B200_MM_EXACT_MMA) {
        __half *xh = (__half *)R.op_arena.get((size_t)xh_bytes(K, B), st);
        quantize_act_f16(vec_dot_type(wtype), dx, K, xh, xds, K, B, st);
        mul_mat_q_exact_mma(w, xh, xds, dd, N, B, nullptr, 0, st);
    } else if (impl == B200_MM_EXACT_TC5) {
        __half *xh = (__half *)R.op_arena.get((size_t)B * K * 2 + 16, st);
        quantize_act_f16_rm(vec_dot_type(wtype), dx, K, xh, xds, K, B, st);
        mul_mat_q_exact_tc5(w, xh, xds, dd, N, B, nullptr, 0, st);
        B200_CHECK(cudaStreamSynchronize(st));
        if (exact_tc5_check_timeout() != 0) return B200_ERR_IO;
    } else if (impl == B200_MM_FAST_TC5) {
        __half *xh = (__half *)R.op_arena.get((size_t)B * K * 2 + 16, st);
        cvt_act_f16(dx, K, xh, K, B, st);
        mul_mat_q_fast_tc5(w, xh, dd, N, B, nullptr, 0, st);
        B200_CHECK(cudaStreamSynchronize(st));
        if (fast_tc5_check_timeout() != 0) return B200_ERR_IO;
    } else if (impl == B200_MM_EXACT_STREAM) {
        if (!mmv_exact_stream_supported(w)) return B200_ERR_BAD_ARG;
        int4 *pack = (int4 *)R.op_arena.get((size_t)(K / QK) * 64, st);
        for (int64_t b = 0; b < B; b++) { quantize_act_pack(wtype, dx + b * K, pack, K, st); mul_mat_vec_q_exact_stream(w, pack, dd + b * N, nullptr, st); }
    } else if (impl == B200_MM_EXACT) mul_mat_q_exact(w, xq, xds, dd, N, B, nullptr, 0, st);
    else if (impl == B200_MM_VEC) { for (int64_t b = 0; b < B; b++) mul_mat_vec_q(w, xq + b * K, xds + b * (K / QK), dd + b * N, nullptr, st); }
    else if (impl == B200_MM_SIMPLE) mul_mat_q_simple(w, xq, xds, dd, N, B, nullptr, 0, st);
    else mul_mat_q(w, xq, xds, dd, N, B, nullptr, 0, st);
    B200_CHECK(cudaMemcpyAsync(dst, dd, (size_t)B * N * 4, cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaStreamSynchronize(st));
    return B200_OK;
}

// ggml_quantize_q{4_0,4_1,5_0,5_1,8_0} on the GPU (crates/llm-base/src/quantize.rs:320-414 calls them per tensor): f32 rows in, GGML blocks out
int b200_op_quantize_weights(int32_t wtype, const float *w_host, int64_t K, int64_t N, void *ggml_blocks_out) {
    if (!is_quant(wtype) || !w_host || !ggml_blocks_out || K % QK) return B200_ERR_BAD_ARG;
    Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
    cudaStream_t st = R.stream;
    float *dw = (float *)R.op_arena.get((size_t)N * K * 4, st);
    B200_CHECK(cudaMemcpyAsync(dw, w_host, (size_t)N * K * 4, cudaMemcpyHostToDevice, st));
    QWeight w;
    const size_t pb = qweight_layout(w, wtype, K, N, nullptr);
    qweight_layout(w, wtype, K, N, R.op_arena.get(pb, st));
    quantize_weights(w, dw, st);
    const size_t raw_bytes = (size_t)N * (K / QK) * ggml_block_bytes(wtype);
    void *raw = R.op_arena.get(raw_bytes, st);
    unpack_weights(w, raw, st);
    B200_CHECK(cudaMemcpyAsync(ggml_blocks_out, raw, raw_bytes, cudaMemcpyDeviceToHost, st));
    B200_CHECK(cudaStreamSynchronize(st));
    return B200_OK;
}

// Kernel-only timing of one weight mat-mul on device-resident synthetic operands (seeded random weights and activations): used by
// tools/prefill_gemm_bench.py and bench.py's prefill roofline; impl = B200_MM_EXACT_MMA / B200_MM_EXACT_TC5 / B200_MM_TENSOR
int b200_op_bench_mul_mat(int32_t wtype, int64_t K, int64_t N, int64_t B, int32_t impl, int32_t iters, float *ms_out) {
    if (!is_quant(wtype) || K % 64 || !ms_out || iters < 1) return B200_ERR_BAD_ARG;
    Runtime &R = rt(); R.ensure_init(); R.op_arena.reset();
    cudaStream_t st = R.stream;
    QWeight w;
    const size_t pb = qweight_layout(w, wtype, K, N, nullptr);
    void *base = R.op_arena.get(pb, st);
    qweight_layout(w, wtype, K, N, base);
    synth_qweight(w, 777u, st);
    float *dx = (float *)R.op_arena.get((size_t)B * K * 4, st);
    float *dd = (float *)R.op_arena.get((size_t)B * N * 4, st);
    float2 *xds = (float2 *)R.op_arena.get((size_t)B * (K / QK) * sizeof(float2), st);
    __half *xh = (__half *)R.op_arena.get(xh_bytes(K, B) + 16, st);
    int8_t *xq = (int8_t *)R.op_arena.get((size_t)B * K, st);
    synth_gain(dx, B * K, 12345u, st);
    if (impl == B200_MM_FAST_TC5) cvt_act_f16(dx, K, xh, K, B, st);
    else if (impl == B200_MM_EXACT_TC5) quantize_act_f16_rm(vec_dot_type(wtype), dx, K, xh, xds, K, B, st);
    else if (impl == B200_MM_EXACT_MMA) quantize_act_f16(vec_dot_type(wtype), dx, K, xh, xds, K, B, st);
    else quantize_act(vec_dot_type(wtype), dx, K, xq, xds, K, B, st);
    auto run = [&]() {
        if (impl == B200_MM_FAST_TC5) mul_mat_q_fast_tc5(w, xh, dd, N, B, nullptr, 0, st);
        else if (impl == B200_MM_EXACT_TC5) mul_mat_q_exact_tc5(w, xh, xds, dd, N, B, nullptr, 0, st);
        else if (impl == B200_MM_EXACT_MMA) mul_mat_q_exact_mma(w, xh, xds, dd, N, B, nullptr, 0, st);
        else mul_mat_q(w, xq, xds, dd, N, B, nullptr, 0, st);
    };
    for (int i = 0; i < 2; i++) run();
    cudaEvent_t e0, e1;
    B200_CHECK(cudaEventCreate(&e0)); B200_CHECK(cudaEventCreate(&e1));
    B200_CHECK(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; i++) run();
    B200_CHECK(cudaEventRecord(e1, st));
    B200_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    B200_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    *ms_out = ms / iters;
    B200_CHECK(cudaEventDestroy(e0)); B200_CHECK(cudaEventDestroy(e1));
    if (impl == B200_MM_EXACT_TC5 && exact_tc5_check_timeout() != 0) return B200_ERR_IO;
    if (impl == B200_MM_FAST_TC5 && fast_tc5_check_timeout() != 0) return B200_ERR_IO;
    return B200_OK;
}

}  // extern "C"
