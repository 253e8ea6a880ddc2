// llm_b200/csrc/neox.cu -- native host runtime for GPT-NeoX and GPT-2 (include/llm_b200.h: b200_neox_*): model + InferenceSession on the B200.
//
// Mirrors   GptNeoX::new / TensorLoader         crates/models/gptneox/src/lib.rs:36-140
//           GptNeoX::evaluate (the graph)       crates/models/gptneox/src/lib.rs:156-350   (feed-forward: :487-515)
//           Gpt2::new / Gpt2::evaluate          crates/models/gpt2/src/lib.rs:43-136, 138-329   (hp.arch == 1: c_attn rows in thirds, no RoPE, learned positions,
//                                                                                               sequential residual, lm_head optional -> tied to wte)
//           InferenceSession::compute           crates/llm-base/src/inference_session.rs:114-295
// Batches (prefill) run node by node on the bit-exact kernels of this directory (LayerNorm, bias adds, RoPE mode 2 on n_rot of the head size, gelu table,
// exact quantized mat-muls incl. the tcgen05 GEMM, exact f16 attention mat-muls); single tokens run the fused 8-kernels-per-layer schedule of
// decode_ops.cu::neox_decode_enqueue from one CUDA graph per context bucket, up to the largest bucket its attention holds (attn_fused_fits: 3072
// positions), and node by node past it.  Logits are bit-identical to the reference's CPU path (tests/test_gpu_neox.py, tests/test_gpu_long_context.py).
#include <string.h>

#include <string>
#include <vector>

#include "../../include/llm_b200.h"
#include "decode.h"
#include "kernels.cuh"
#include "runtime.h"

using namespace b200;

struct b200_neox_model {
    b200_neox_hparams hp;
    int hd = 0;
    char *slab = nullptr;
    size_t slab_bytes = 0, weight_bytes = 0;
    QWeight wte, lm_head;
    float *lnf_g = nullptr, *lnf_b = nullptr, *wpe = nullptr;     // wpe: GPT-2 learned positions [n_ctx][e] f32
    bool gpt2() const { return hp.arch == 1; }
    struct Layer { QWeight wqkv, wdense, wfc, wproj; float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *bqkv, *bdense, *bfc, *bproj; };
    std::vector<Layer> layers;
    std::vector<uint8_t> loaded;
    int n_loaded = 0;
    int n_slots() const { return 4 + 12 * hp.n_layer + (gpt2() && hp.has_lm_head ? 1 : 0); }   // GPT-2: slot 3 = wpe, lm_head (if present) last
    struct Slot { QWeight q; float *f = nullptr; int64_t n = 0; bool is_q = false; };
    bool lookup(const char *name, Slot &s, int &id);
};

struct b200_neox_session {
    b200_neox_model *m = nullptr;
    int n_batch = 0, n_past = 0, dev_n_past = -1, last_launches = 0, graph_nodes = 0;
    __half *memory_k = nullptr, *memory_v = nullptr;            // [n_layer][n_ctx][e], [n_layer][e][n_ctx]
    int32_t *d_tokens = nullptr, *h_tokens = nullptr;
    float *x = nullptr, *cur = nullptr, *qkv = nullptr, *kq = nullptr, *attn = nullptr, *h4 = nullptr, *hact = nullptr, *t = nullptr, *logits = nullptr, *h_logits = nullptr;
    float *qdec = nullptr;
    int8_t *xq = nullptr; float2 *xds = nullptr; int4 *xpack = nullptr; __half *xh = nullptr;
    int4 *xpack_a = nullptr, *xpack_d = nullptr, *xpack_f = nullptr;
    int *d_n_past = nullptr, *h_n_past = nullptr;
    bool decode_ok = false, decode_warm = false;
    std::vector<NeoxLayer> dl;
    NeoxParams dp;
    std::vector<std::pair<int, cudaGraphExec_t>> graphs;
};

bool b200_neox_model::lookup(const char *name, Slot &s, int &id) {
    const int e = hp.n_embd;
    s = Slot();
    if (gpt2()) {                                                         // tensor names of crates/models/gpt2/src/lib.rs:59-107
        if (!strcmp(name, "model/wte")) { s.q = wte; s.is_q = true; id = 0; return true; }
        if (!strcmp(name, "model/ln_f/g")) { s.f = lnf_g; s.n = e; id = 1; return true; }
        if (!strcmp(name, "model/ln_f/b")) { s.f = lnf_b; s.n = e; id = 2; return true; }
        if (!strcmp(name, "model/wpe")) { s.f = wpe; s.n = (int64_t)hp.context_size * e; id = 3; return true; }
        if (!strcmp(name, "model/lm_head")) { if (!hp.has_lm_head) return false; s.q = lm_head; s.is_q = true; id = 4 + 12 * hp.n_layer; return true; }
        int il = -1; char sub[96];
        if (sscanf(name, "model/h%d/%95s", &il, sub) != 2 || il < 0 || il >= hp.n_layer) return false;
        Layer &L = layers[il];
        struct { const char *n; QWeight *q; float *f; int64_t len; } tab[] = {
            {"ln_1/g", nullptr, L.ln1_g, e}, {"ln_1/b", nullptr, L.ln1_b, e}, {"ln_2/g", nullptr, L.ln2_g, e}, {"ln_2/b", nullptr, L.ln2_b, e},
            {"attn/c_attn/w", &L.wqkv, nullptr, 0}, {"attn/c_attn/b", nullptr, L.bqkv, 3 * (int64_t)e}, {"attn/c_proj/w", &L.wdense, nullptr, 0}, {"attn/c_proj/b", nullptr, L.bdense, e},
            {"mlp/c_fc/w", &L.wfc, nullptr, 0}, {"mlp/c_fc/b", nullptr, L.bfc, 4 * (int64_t)e}, {"mlp/c_proj/w", &L.wproj, nullptr, 0}, {"mlp/c_proj/b", nullptr, L.bproj, e}};
        for (int k = 0; k < 12; k++)
            if (!strcmp(sub, tab[k].n)) {
                if (tab[k].q) { s.q = *tab[k].q; s.is_q = true; } else { s.f = tab[k].f; s.n = tab[k].len; }
                id = 4 + 12 * il + k;
                return true;
            }
        return false;
    }
    if (!strcmp(name, "gpt_neox.embed_in.weight")) { s.q = wte; s.is_q = true; id = 0; return true; }
    if (!strcmp(name, "gpt_neox.final_layer_norm.weight")) { s.f = lnf_g; s.n = e; id = 1; return true; }
    if (!strcmp(name, "gpt_neox.final_layer_norm.bias")) { s.f = lnf_b; s.n = e; id = 2; return true; }
    if (!strcmp(name, "embed_out.weight")) { s.q = lm_head; s.is_q = true; id = 3; return true; }
    int il = -1; char sub[96];
    if (sscanf(name, "gpt_neox.layers.%d.%95s", &il, sub) != 2 || il < 0 || il >= hp.n_layer) return false;
    Layer &L = layers[il];
    const int base = 4 + 12 * il;
    struct { const char *n; QWeight *q; float *f; int64_t len; } tab[] = {
        {"input_layernorm.weight", nullptr, L.ln1_g, e}, {"input_layernorm.bias", nullptr, L.ln1_b, e},
        {"post_attention_layernorm.weight", nullptr, L.ln2_g, e}, {"post_attention_layernorm.bias", nullptr, L.ln2_b, e},
        {"attention.query_key_value.weight", &L.wqkv, nullptr, 0}, {"attention.query_key_value.bias", nullptr, L.bqkv, 3 * (int64_t)e},
        {"attention.dense.weight", &L.wdense, nullptr, 0}, {"attention.dense.bias", nullptr, L.bdense, e},
        {"mlp.dense_h_to_4h.weight", &L.wfc, nullptr, 0}, {"mlp.dense_h_to_4h.bias", nullptr, L.bfc, 4 * (int64_t)e},
        {"mlp.dense_4h_to_h.weight", &L.wproj, nullptr, 0}, {"mlp.dense_4h_to_h.bias", nullptr, L.bproj, e}};
    for (int k = 0; k < 12; k++)
        if (!strcmp(sub, tab[k].n)) {
            if (tab[k].q) { s.q = *tab[k].q; s.is_q = true; } else { s.f = tab[k].f; s.n = tab[k].len; }
            id = base + k;
            return true;
        }
    return false;
}

namespace {

// ggml_mul_mat(w, x) for B rows: INIT-phase quantization + the bit-exact kernel for the batch size
void matmul(b200_neox_session *s, const QWeight &w, const float *x, float *dst, int64_t ldd, int64_t B, cudaStream_t st, int &n) {
    if (B == 1 && mmv_exact_stream_supported(w)) {
        quantize_act_pack(w.type, x, s->xpack, w.K, st);
        mul_mat_vec_q_exact_stream(w, s->xpack, dst, nullptr, st);
    } else if (B >= 16) {
        if (prefill_gemm_tc5() && B >= 96) {
            quantize_act_f16_rm(vec_dot_type(w.type), x, w.K, s->xh, s->xds, w.K, B, st);
            mul_mat_q_exact_tc5(w, s->xh, s->xds, dst, ldd, B, nullptr, 0, st);
        } else {
            quantize_act_f16(vec_dot_type(w.type), x, w.K, s->xh, s->xds, w.K, B, st);
            mul_mat_q_exact_mma(w, s->xh, s->xds, dst, ldd, B, nullptr, 0, st);
        }
    } else {
        quantize_act(vec_dot_type(w.type), x, w.K, s->xq, s->xds, w.K, B, st);
        mul_mat_q_exact(w, s->xq, s->xds, dst, ldd, B, nullptr, 0, st);
    }
    n += 2;
}

void forward(b200_neox_session *s, int n, bool all_rows) {
    b200_neox_model *m = s->m;
    const b200_neox_hparams &hp = m->hp;
    cudaStream_t st = rt().stream;
    const int e = hp.n_embd, hd = m->hd, n_head = hp.n_head, n_ctx = hp.context_size, n_past = s->n_past, n_kv = n_past + n;
    int L = 0;
    int bucket = ((n_kv + 255) / 256) * 256; if (bucket > n_ctx) bucket = n_ctx;
    // a bucket the cluster attention cannot hold (past 3072 positions) decodes through the per-op schedule below, which leaves d_n_past alone
    if (n == 1 && s->decode_ok && attn_fused_fits(bucket, hd)) {
        if (s->dev_n_past != n_past) {
            B200_CHECK(cudaStreamSynchronize(st));
            *s->h_n_past = n_past;
            B200_CHECK(cudaMemcpyAsync(s->d_n_past, s->h_n_past, sizeof(int), cudaMemcpyHostToDevice, st));
        }
        int nodes = 0;
        if (!s->decode_warm) {
            neox_decode_enqueue(s->dp, s->dl, hp.wtype, bucket, st, &nodes);
            s->decode_warm = true; s->graph_nodes = nodes;
        } else {
            cudaGraphExec_t exec = nullptr;
            for (auto &g : s->graphs) if (g.first == bucket) exec = g.second;
            if (!exec) {
                cudaGraph_t graph;
                B200_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                neox_decode_enqueue(s->dp, s->dl, hp.wtype, bucket, st, &nodes);
                B200_CHECK(cudaStreamEndCapture(st, &graph));
                B200_CHECK(cudaGraphInstantiate(&exec, graph, 0));
                B200_CHECK(cudaGraphDestroy(graph));
                s->graphs.emplace_back(bucket, exec);
                s->graph_nodes = nodes;
            }
            B200_CHECK(cudaGraphLaunch(exec, st));
        }
        s->dev_n_past = n_past + 1;
        s->last_launches = s->graph_nodes; s->n_past += 1;
        return;
    }
    const float kq_scale = 1.0f / sqrtf((float)e / (float)n_head);                                                  // :270-273
    const bool g2 = m->gpt2(), parallel = !g2 && hp.use_parallel_residual;
    const RopeTable *rope = g2 ? nullptr : &rope_table(hp.n_rot, 2, 10000.0f, 1.0f, hd, n_ctx);
    const int64_t ld3 = 3 * (int64_t)e;
    // where q / k / v of head h live inside a row of the fused projection: NeoX per head [q | k | v], GPT-2 the three thirds of the row
    const int64_t hs = g2 ? hd : 3 * hd, koff = g2 ? e : hd, voff = g2 ? 2 * (int64_t)e : 2 * hd;
    get_rows_q(m->wte, s->d_tokens, s->x, n, st); L++;                                                               // :178
    if (g2) { add_f32(s->x, m->wpe + (size_t)n_past * e, s->x, (int64_t)n * e, (int64_t)n * e, st); L++; }             // gpt2 lib.rs:164-172: + wpe[n_past + i]
    for (int il = 0; il < hp.n_layer; il++) {
        const b200_neox_model::Layer &ly = m->layers[il];
        __half *Kl = s->memory_k + (size_t)il * n_ctx * e, *Vl = s->memory_v + (size_t)il * n_ctx * e;
        layer_norm(s->x, s->cur, ly.ln1_g, ly.ln1_b, e, n, st); L++;                                                  // :192-196
        matmul(s, ly.wqkv, s->cur, s->qkv, ld3, n, st, L);                                                             // :199
        add_f32(s->qkv, ly.bqkv, s->qkv, (int64_t)n * ld3, ld3, st); L++;                                             // :200
        if (!g2) {   // RoPE mode 2 in place on q and k                                                                       :205-228
            rope_f32(s->qkv, s->qkv, hd, n_head, n, hs, ld3, hs, ld3, n_past, *rope, st); L++;
            rope_f32(s->qkv + koff, s->qkv + koff, hd, n_head, n, hs, ld3, hs, ld3, n_past, *rope, st); L++;
        }
        {   // k -> cache rows n_past.., v -> cache columns (transposed; GPT-2's v_trans copy of every evaluate is this layout)       :231-247
            StridedDesc sk{{hd, n_head, n, 1}, {4, hs * 4, ld3 * 4, 0}}, dk{{hd, n_head, n, 1}, {2, (int64_t)hd * 2, (int64_t)e * 2, 0}};
            cpy_strided(s->qkv + koff, T_F32, sk, Kl + (size_t)n_past * e, T_F16, dk, st); L++;
            StridedDesc dv{{hd, n_head, n, 1}, {(int64_t)n_ctx * 2, (int64_t)hd * n_ctx * 2, 2, 0}};
            cpy_strided(s->qkv + voff, T_F32, sk, Vl + n_past, T_F16, dv, st); L++;
        }
        mul_mat_f16_exact(Kl, hd, n_kv, n_head, (int64_t)e * 2, (int64_t)hd * 2, s->qkv, n, n_head, ld3 * 4, hs * 4,
                          s->kq, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4, n_past, st); L++;                          // :250-267
        soft_max(s->kq, s->kq, n_kv, (int64_t)n_head * n, n, kq_scale, true, n_past, true, true, st); L++;            // :270-279
        mul_mat_f16_exact(Vl, n_kv, hd, n_head, (int64_t)n_ctx * 2, (int64_t)n_ctx * hd * 2, s->kq, n, n_head, (int64_t)n_kv * 4, (int64_t)n_kv * n * 4,
                          s->cur, (int64_t)e * 4, (int64_t)hd * 4, -1, st); L++;                                      // :282-298
        matmul(s, ly.wdense, s->cur, s->attn, e, n, st, L);                                                            // :301
        add_f32(s->attn, ly.bdense, s->attn, (int64_t)n * e, e, st); L++;                                             // :302
        const float *ff_in = s->x;
        if (!parallel) { add_f32(s->attn, s->x, s->attn, (int64_t)n * e, (int64_t)n * e, st); L++; ff_in = s->attn; }   // :308-309 / gpt2 :279
        layer_norm(ff_in, s->cur, ly.ln2_g, ly.ln2_b, e, n, st); L++;                                                 // feed_forward :487-493
        matmul(s, ly.wfc, s->cur, s->h4, 4 * (int64_t)e, n, st, L);
        add_f32(s->h4, ly.bfc, s->h4, (int64_t)n * 4 * e, 4 * (int64_t)e, st); L++;
        unary_lut(UNARY_GELU, s->h4, s->hact, (int64_t)n * 4 * e, st); L++;
        matmul(s, ly.wproj, s->hact, s->t, e, n, st, L);
        add_f32(s->t, ly.bproj, s->t, (int64_t)n * e, e, st); L++;
        add_f32(s->t, s->attn, s->t, (int64_t)n * e, (int64_t)n * e, st); L++;                                        // parallel: ffn + attn; sequential: ffn + ff_in
        if (parallel) { add_f32(s->t, s->x, s->x, (int64_t)n * e, (int64_t)n * e, st); L++; }        // :324
        else { B200_CHECK(cudaMemcpyAsync(s->x, s->t, (size_t)n * e * 4, cudaMemcpyDeviceToDevice, st)); }
    }
    if (all_rows || n == 1) {
        layer_norm(s->x, s->cur, m->lnf_g, m->lnf_b, e, n, st); L++;                                                   // :332-334
        matmul(s, m->lm_head, s->cur, s->logits, hp.n_vocab, n, st, L);                                                // :342
    } else {
        const size_t last = (size_t)(n - 1);
        layer_norm(s->x + last * e, s->cur + last * e, m->lnf_g, m->lnf_b, e, 1, st); L++;
        matmul(s, m->lm_head, s->cur + last * e, s->logits + last * hp.n_vocab, hp.n_vocab, 1, st, L);
    }
    s->last_launches = L;
    s->n_past += n;
}

}  // namespace

extern "C" {

b200_neox_model *b200_neox_new(const b200_neox_hparams *hp) {
    if (!hp || !is_quant(hp->wtype) || hp->n_embd % 64 || hp->n_head <= 0 || hp->n_embd % hp->n_head || hp->n_layer <= 0 || hp->context_size <= 0 || hp->arch < 0 || hp->arch > 1 ||
        (hp->arch == 0 && (hp->n_rot <= 0 || hp->n_rot % 2 || hp->n_rot > hp->n_embd / hp->n_head))) return nullptr;
    rt().ensure_init();
    b200_neox_model *m = new b200_neox_model();
    m->hp = *hp;
    const int e = hp->n_embd, v = hp->n_vocab, t = hp->wtype;
    m->hd = e / hp->n_head;
    m->layers.resize(hp->n_layer);
    for (int pass = 0; pass < 2; pass++) {
        size_t off = 0;
        auto cq = [&](QWeight &w, int64_t K, int64_t N) {
            off += qweight_layout(w, t, K, N, pass ? m->slab + off : nullptr);
            if (pass) m->weight_bytes += (size_t)N * (K / QK) * ggml_block_bytes(t);
        };
        auto cf = [&](float *&p, int64_t n) { if (pass) p = (float *)(m->slab + off); off += ((size_t)n * 4 + 255) & ~(size_t)255; };
        cq(m->wte, e, v);
        if (!m->gpt2() || hp->has_lm_head) cq(m->lm_head, e, v);
        cf(m->lnf_g, e); cf(m->lnf_b, e);
        if (m->gpt2()) cf(m->wpe, (int64_t)hp->context_size * e);
        for (auto &L : m->layers) {
            cf(L.ln1_g, e); cf(L.ln1_b, e); cf(L.ln2_g, e); cf(L.ln2_b, e); cf(L.bqkv, 3 * e); cf(L.bdense, e); cf(L.bfc, 4 * e); cf(L.bproj, e);
            cq(L.wqkv, e, 3 * e); cq(L.wdense, e, e); cq(L.wfc, e, 4 * e); cq(L.wproj, 4 * e, e);
        }
        if (!pass) { m->slab_bytes = off; B200_CHECK(cudaMalloc(&m->slab, off)); }
    }
    if (m->gpt2() && !hp->has_lm_head) m->lm_head = m->wte;              // tied output projection (gpt2 lib.rs:319-320): wte is streamed as the lm_head
    else m->weight_bytes -= (size_t)v * (e / QK) * ggml_block_bytes(t);  // the embedding table is gathered from, not streamed
    m->loaded.assign(m->n_slots(), 0);
    return m;
}

size_t b200_neox_weight_bytes(b200_neox_model *m) { return m ? m->weight_bytes : 0; }

int b200_neox_load_tensor(b200_neox_model *m, const char *name, int32_t type, const void *host_data, size_t nbytes) {
    if (!m || !name || !host_data) return B200_ERR_BAD_ARG;
    b200_neox_model::Slot s; int id;
    if (!m->lookup(name, s, id)) return B200_ERR_UNKNOWN_TENSOR;
    Runtime &R = rt();
    if (s.is_q) {
        if (type != s.q.type || nbytes != (size_t)s.q.N * s.q.nb * ggml_block_bytes(type)) return B200_ERR_TENSOR_SHAPE;
        R.op_arena.reset();
        void *raw = R.op_arena.get(nbytes, R.stream);
        B200_CHECK(cudaMemcpyAsync(raw, host_data, nbytes, cudaMemcpyHostToDevice, R.stream));
        repack_weights(s.q, raw, R.stream);
        B200_CHECK(cudaStreamSynchronize(R.stream));
    } else {
        if (type != T_F32 || nbytes != (size_t)s.n * 4) return B200_ERR_TENSOR_SHAPE;
        B200_CHECK(cudaMemcpy(s.f, host_data, nbytes, cudaMemcpyHostToDevice));
        B200_CHECK(cudaDeviceSynchronize());
    }
    if (!m->loaded[id]) { m->loaded[id] = 1; m->n_loaded++; }
    return B200_OK;
}

// seeded synthetic weights generated in HBM (bench): N(0, 1/K) quantized by the reference's rule, LayerNorm gains 1 + 0.1 N(0,1), biases = gains - 1 (small)
int b200_neox_synthesize(b200_neox_model *m, uint64_t seed) {
    if (!m) return B200_ERR_BAD_ARG;
    cudaStream_t st = rt().stream;
    uint64_t id = 0;
    auto q = [&](const QWeight &w) { synth_qweight(w, seed + 0x1000003ull * (++id), st); };
    auto g = [&](float *p, int64_t n) { synth_gain(p, n, seed + 0x1000003ull * (++id), st); };
    auto b = [&](float *p, int64_t n) { synth_gain(p, n, seed + 0x1000003ull * (++id), st); scale_shift_f32(p, n, 0.1f, -0.1f, st); };   // 0.01 N(0,1)
    const int e = m->hp.n_embd;
    q(m->wte); if (!m->gpt2() || m->hp.has_lm_head) q(m->lm_head); g(m->lnf_g, e); b(m->lnf_b, e);
    if (m->gpt2()) b(m->wpe, (int64_t)m->hp.context_size * e);
    for (auto &L : m->layers) {
        g(L.ln1_g, e); b(L.ln1_b, e); g(L.ln2_g, e); b(L.ln2_b, e); b(L.bqkv, 3 * e); b(L.bdense, e); b(L.bfc, 4 * e); b(L.bproj, e);
        q(L.wqkv); q(L.wdense); q(L.wfc); q(L.wproj);
    }
    B200_CHECK(cudaStreamSynchronize(st));
    m->loaded.assign(m->n_slots(), 1); m->n_loaded = m->n_slots();
    return B200_OK;
}

void b200_neox_free(b200_neox_model *m) {
    if (!m) return;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    if (m->slab) B200_CHECK(cudaFree(m->slab));
    delete m;
}

b200_neox_session *b200_neox_start_session(b200_neox_model *m, int32_t n_batch) {
    if (!m || n_batch < 1) return nullptr;
    if (m->n_loaded != m->n_slots()) { fprintf(stderr, "llm_b200: neox start_session: %d of %d tensors loaded\n", m->n_loaded, m->n_slots()); return nullptr; }
    b200_neox_session *s = new b200_neox_session();
    s->m = m; s->n_batch = n_batch;
    const b200_neox_hparams &hp = m->hp;
    const size_t e = hp.n_embd, B = n_batch, n_ctx = hp.context_size, V = hp.n_vocab;
    const size_t kv = (size_t)hp.n_layer * n_ctx * e;
    B200_CHECK(cudaMalloc(&s->memory_k, kv * 2)); B200_CHECK(cudaMalloc(&s->memory_v, kv * 2));
    B200_CHECK(cudaMemset(s->memory_k, 0, kv * 2)); B200_CHECK(cudaMemset(s->memory_v, 0, kv * 2));
    B200_CHECK(cudaMalloc(&s->d_tokens, B * 4)); B200_CHECK(cudaMallocHost(&s->h_tokens, B * 4));
    B200_CHECK(cudaMalloc(&s->x, B * e * 4)); B200_CHECK(cudaMalloc(&s->cur, B * e * 4)); B200_CHECK(cudaMalloc(&s->qkv, B * 3 * e * 4));
    B200_CHECK(cudaMalloc(&s->kq, (size_t)hp.n_head * B * n_ctx * 4)); B200_CHECK(cudaMalloc(&s->attn, B * e * 4));
    B200_CHECK(cudaMalloc(&s->h4, B * 4 * e * 4)); B200_CHECK(cudaMalloc(&s->hact, B * 4 * e * 4)); B200_CHECK(cudaMalloc(&s->t, B * e * 4));
    B200_CHECK(cudaMalloc(&s->logits, B * V * 4)); B200_CHECK(cudaMallocHost(&s->h_logits, B * V * 4));
    B200_CHECK(cudaMalloc(&s->xq, B * 4 * e)); B200_CHECK(cudaMalloc(&s->xds, B * (4 * e / QK) * sizeof(float2)));
    B200_CHECK(cudaMalloc(&s->xpack, (4 * e / QK) * 64)); B200_CHECK(cudaMalloc(&s->xh, xh_bytes(4 * e, B)));
    B200_CHECK(cudaMalloc(&s->qdec, e * 4));
    B200_CHECK(cudaMalloc(&s->xpack_a, (e / QK) * 64)); B200_CHECK(cudaMalloc(&s->xpack_d, (e / QK) * 64)); B200_CHECK(cudaMalloc(&s->xpack_f, (4 * e / QK) * 64));
    B200_CHECK(cudaMalloc(&s->d_n_past, sizeof(int))); B200_CHECK(cudaMallocHost(&s->h_n_past, sizeof(int)));
    const RopeTable *rt_ = m->gpt2() ? nullptr : &rope_table(hp.n_rot, 2, 10000.0f, 1.0f, m->hd, (int)n_ctx);
    s->dl.resize(hp.n_layer);
    for (int il = 0; il < hp.n_layer; il++) {
        const b200_neox_model::Layer &L = m->layers[il];
        s->dl[il] = NeoxLayer{L.wqkv, L.wdense, L.wfc, L.wproj, L.ln1_g, L.ln1_b, L.ln2_g, L.ln2_b, L.bqkv, L.bdense, L.bfc, L.bproj,
                              s->memory_k + (size_t)il * n_ctx * e, s->memory_v + (size_t)il * n_ctx * e};
    }
    NeoxParams &P = s->dp;
    P.n_layer = hp.n_layer; P.e = (int)e; P.hd = m->hd; P.n_head = hp.n_head; P.n_ctx = (int)n_ctx; P.n_vocab = hp.n_vocab; P.n_rot = hp.n_rot;
    P.parallel_residual = !m->gpt2() && hp.use_parallel_residual; P.gpt2 = m->gpt2() ? 1 : 0; P.wpe = m->wpe; P.wte = m->wte; P.lm_head = m->lm_head; P.lnf_g = m->lnf_g; P.lnf_b = m->lnf_b;
    P.kq_scale = 1.0f / sqrtf((float)e / (float)hp.n_head); P.rope_cs = rt_ ? rt_->cs : nullptr; P.rope_half = rt_ ? rt_->half : 0;
    P.lut_gelu = luts().gelu; P.lut_exp = luts().exp; P.token = s->d_tokens; P.n_past = s->d_n_past;
    P.x = s->x; P.qkv = s->qkv; P.q = s->qdec; P.attn_out = s->attn; P.logits = s->logits;
    P.xpack_a = s->xpack_a; P.xpack_d = s->xpack_d; P.xpack_f = s->xpack_f;
    QWeight p1; p1.nb = (int64_t)e / QK; QWeight p2; p2.nb = 4 * (int64_t)e / QK;
    s->decode_ok = m->hd % 32 == 0 && m->hd <= 128 && e % 128 == 0 && e <= 8192 && n_ctx % 8 == 0 && mmv_exact_stream_supported(p1) && mmv_exact_stream_supported(p2) &&
                   !getenv("B200_NEOX_UNFUSED");
    B200_CHECK(cudaDeviceSynchronize());
    return s;
}

int32_t b200_neox_n_past(const b200_neox_session *s) { return s ? s->n_past : -1; }
int b200_neox_set_n_past(b200_neox_session *s, int32_t n_past) {
    if (!s || n_past < 0 || n_past > s->n_past) return B200_ERR_BAD_ARG;
    s->n_past = n_past;
    return B200_OK;
}
int32_t b200_neox_last_launches(const b200_neox_session *s) { return s ? s->last_launches : 0; }
int b200_neox_sync(b200_neox_session *s) { if (!s) return B200_ERR_BAD_ARG; B200_CHECK(cudaStreamSynchronize(rt().stream)); return B200_OK; }

// tokens already in HBM (left there by the last b200_neox_evaluate), logits stay in HBM
int b200_neox_evaluate_device(b200_neox_session *s, int32_t n) {
    if (!s || n < 1 || n > s->n_batch) return B200_ERR_BAD_ARG;
    if (s->n_past + n > s->m->hp.context_size) return B200_ERR_CONTEXT_FULL;
    forward(s, n, true);
    return B200_OK;
}

int b200_neox_evaluate(b200_neox_session *s, const int32_t *tokens, int32_t n, float *logits_out, int32_t all_logits) {
    if (!s || !tokens || n < 1 || n > s->n_batch) return B200_ERR_BAD_ARG;
    if (s->n_past + n > s->m->hp.context_size) return B200_ERR_CONTEXT_FULL;
    for (int i = 0; i < n; i++) if (tokens[i] < 0 || tokens[i] >= s->m->hp.n_vocab) return B200_ERR_BAD_ARG;
    cudaStream_t st = rt().stream;
    B200_CHECK(cudaStreamSynchronize(st));
    memcpy(s->h_tokens, tokens, (size_t)n * 4);
    B200_CHECK(cudaMemcpyAsync(s->d_tokens, s->h_tokens, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    forward(s, n, all_logits != 0);
    if (logits_out) {
        const size_t V = s->m->hp.n_vocab, rows = all_logits ? n : 1;
        const float *src = all_logits ? s->logits : s->logits + (size_t)(n - 1) * V;
        B200_CHECK(cudaMemcpyAsync(s->h_logits, src, rows * V * 4, cudaMemcpyDeviceToHost, st));
        B200_CHECK(cudaStreamSynchronize(st));
        memcpy(logits_out, s->h_logits, rows * V * 4);
    }
    return B200_OK;
}

void b200_neox_session_free(b200_neox_session *s) {
    if (!s) return;
    B200_CHECK(cudaStreamSynchronize(rt().stream));
    for (auto &g : s->graphs) cudaGraphExecDestroy(g.second);
    void *dev[] = {s->memory_k, s->memory_v, s->d_tokens, s->x, s->cur, s->qkv, s->kq, s->attn, s->h4, s->hact, s->t, s->logits, s->xq, s->xds, s->xpack, s->xh, s->qdec,
                   s->xpack_a, s->xpack_d, s->xpack_f, s->d_n_past};
    for (void *p : dev) if (p) B200_CHECK(cudaFree(p));
    if (s->h_tokens) B200_CHECK(cudaFreeHost(s->h_tokens));
    if (s->h_logits) B200_CHECK(cudaFreeHost(s->h_logits));
    if (s->h_n_past) B200_CHECK(cudaFreeHost(s->h_n_past));
    delete s;
}

}  // extern "C"
