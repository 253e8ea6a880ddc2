// llm_b200/csrc/decode.h -- parameters of the one-launch-per-token decode kernel (decode.cu)
#pragma once
#include <vector>

#include "kernels.cuh"
#include "tp.cuh"

#ifndef B200_PROF_SLOTS
#define B200_PROF_SLOTS 1024
#endif

namespace b200 {

struct DecodeLayer {
    QWeight wqkv, wo, w13, w2;
    const float *attn_norm, *ffn_norm;
    __half *K, *V;                      // this layer's slice of memory_k ([n_ctx][gqa]) / memory_v ([gqa][n_ctx], transposed)
};

struct DecodeParams {
    const DecodeLayer *layers;
    int n_layer;
    QWeight wte, output;
    const float *norm;
    int e, f, hd, gqa, n_head, n_head_kv, n_ctx, n_vocab;
    float kq_scale, eps;
    const float2 *rope_cs; int rope_half;
    const uint16_t *lut_silu, *lut_exp;
    const int32_t *token;
    int *n_past;                        // device copy of InferenceSession::n_past; incremented at the end of the kernel
    float *x, *q, *kq, *attn, *ff, *h13, *logits;
    int scratch_bytes;                  // decode_scratch_bytes(): per-CTA shared memory behind the weight ring
    int4 *xpack_d, *xpack_f;            // activation records produced by phase C (for wo) and phase E (for w2)
    // tensor-parallel decode (tp.cuh): dims above are THIS RANK's (n_head, n_head_kv, gqa = local heads / cache width; f = local n_ff / G;
    // n_vocab = local rows of the lm_head) except e = the full n_embd; e_loc = n_embd / G (q rows, rows of wo / w2 owned here)
    TpCtx tp;
    int e_loc = 0, head0 = 0;           // first global head of this rank
    int n_vocab_full = 0;               // rows of the whole lm_head (the gathered logits)
    int64_t row0_e = 0, row0_w13 = 0, row0_v = 0;   // first row of this rank in the full wo / w2 output, the interleaved [w1|w3] rows, the lm_head
    unsigned int *bar;                  // [0] arrival count, [1] generation
    unsigned long long *prof;   /* graph schedule: 3 x B200_PROF_SLOTS timeline slots (begin | end | prologue done) */           // optional: %globaltimer stamps of CTA 0 at phase boundaries (debug / tuning), 128 slots
};

// ---- GPT-NeoX (crates/models/gptneox/src/lib.rs:156-350) fused decode schedule: 8 kernels per layer, same mat-vec core -------------------------
struct NeoxLayer {
    QWeight wqkv, wdense, wfc, wproj;   // query_key_value [3e x e] (rows per head: q | k | v), attention.dense, mlp.dense_h_to_4h, mlp.dense_4h_to_h
    const float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *bqkv, *bdense, *bfc, *bproj;
    __half *K, *V;                      // [n_ctx][e] by position / [e][n_ctx] transposed, as the reference lays out memory_k / memory_v (:233-247)
};
struct NeoxParams {
    int n_layer, e, hd, n_head, n_ctx, n_vocab, n_rot, parallel_residual;
    int gpt2;                                   // GPT-2 (crates/models/gpt2/src/lib.rs:138-329): c_attn rows are [q | k | v] thirds, no RoPE, learned positions wpe, sequential residual
    const float *wpe;                           // [n_ctx][e] f32 (GPT-2), else nullptr
    QWeight wte, lm_head;
    const float *lnf_g, *lnf_b;
    float kq_scale;
    const float2 *rope_cs; int rope_half;
    const uint16_t *lut_gelu, *lut_exp;
    const int32_t *token; int *n_past;
    float *x, *qkv, *q, *attn_out, *logits;     // residual stream [e], raw qkv [3e], roped q [e], attention branch output [e]
    int4 *xpack_a, *xpack_d, *xpack_f;          // records: layer-norm output (K = e), attention rows (K = e), gelu output (K = 4e)
};
void decode_set_tp(const TpCtx &T, cudaStream_t st);   // uploads the tensor-parallel context the decode kernels read (constant memory)
void neox_decode_enqueue(const NeoxParams &P, const std::vector<NeoxLayer> &layers, int wtype, int n_kv_bucket, cudaStream_t st, int *launches);

int decode_scratch_bytes(int e, int f, int hd, int n_ctx);
bool decode_supported(const DecodeParams &P, int wtype);
// cooperative launch on `st`; returns false if the kernel cannot be made resident (caller falls back to the per-op schedule)
bool launch_decode(const DecodeParams &P, int wtype, cudaStream_t st, int *grid_out);

// whether the cluster attention kernel of the fused decode schedules (decode_ops.cu) holds a context bucket of n_kv_bucket positions in shared
// memory at head size hd: true up to a bucket of 3072 (and for a last bucket, capped at n_ctx, of up to 3264).  LLaMA decodes the larger buckets
// through the two-kernel attention, GPT-NeoX / GPT-2 through the per-op schedule; a tensor-parallel session needs every bucket to fit.
bool attn_fused_fits(int n_kv_bucket, int hd);

// default decode schedule: 8 fused kernels per layer on `st` (decode_ops.cu); position read from *P.n_past on the device
void decode_ops_enqueue(const DecodeParams &P, const std::vector<DecodeLayer> &layers, int wtype, int n_kv_bucket, int4 *xpack_a, cudaStream_t st, int *launches);

}  // namespace b200
