// llm_b200/csrc/decode_ops.cu -- the default decode schedule: 7 fused kernels per layer, replayed from ONE CUDA graph per token.
//
//   1 norm_pack        rms_norm(x) * attn_norm -> Q8 activation records                       (llama lib.rs:183-186 + mul_mat INIT)
//   2 mmv<QKV>         [wq|wk|wv] x, epilogue: RoPE on Q/K rows, K/V rows -> f16 cache at n_past (:190-244)
//   3 attn_fused       KQ = K . f16(Q), scale + soft_max, V^T . f16(P), epilogue: quantize the merged row -- one cluster of hd/32 CTAs per
//                      head, scores exchanged through distributed shared memory                (:246-307)
//                      (B200_ATTN_FUSED=0, and context buckets past 3072 positions: the two-kernel variant attn_kq + attn_sv)
//   4 mmv<RES>         wo x + inpSA                                                           (:310-314)
//   5 norm_pack        rms_norm(inpFF) * ffn_norm                                             (:318-321)
//   6 mmv<SILU>        [w1|w3] x (rows interleaved in 32-row pieces), epilogue: silu(w1 x) * (w3 x) quantized (:323-330)
//   7 mmv<RES>         w2 h + inpFF                                                           (:332-334)
// Everything that depends on the position reads n_past from DEVICE memory, so the captured graph is valid for every token; the
// last node increments it.  All arithmetic is the bit-exact arithmetic of exact.cu / rowops.cu (same device functions as decode.cu).
// What was tried on top of this and measured slower (PDL, norm fusion, tiled weights + TMA, L2 prefetch, ...): profiles/r01_notes.md.
#include <cooperative_groups.h>
#include <stdlib.h>

#include <array>
#include <map>
#include <vector>

#include "decode.h"
#include "stream_core.cuh"
#include "tp.cuh"

namespace b200 {

using namespace stream;

// the tensor-parallel context of this process's session (tp.cuh): one copy in constant memory instead of ~120 bytes in every kernel's argument block
// (the single-GPU decode graph must not pay for it: 227 launches per token).  world == 0 / 1: single GPU.
__constant__ TpCtx c_tp;

namespace {

// Programmatic dependent launch.  Every kernel of the chain touches nothing a predecessor of the same token writes (and writes nothing at
// all) before `pdl_wait`.  What runs ahead of the wait reads the constant weights (the producer warp of the next mat-vec fills its ring)
// and, in the fused attention, n_past and the layer's K rows / V columns below n_past: within one token n_past changes only in the last
// node (EPI_LOGITS, EPI_BIAS with n_past_inc), which starts after every attention launch has completed, and the only writer of a layer's
// cache is the launch right before its attention (mmv<EPI_QKV>, or neox_rope_store_kernel for GPT-NeoX / GPT-2), which writes K row and
// V column n_past and nothing else.  Everything below n_past was written by earlier tokens or batches, which are stream-ordered before
// this token's graph (its first node is an ordinary launch).  Tensor-parallel ranks hold their own heads of the cache: the same holds.
// WHERE the dependents are released matters (B200, LLaMA-7B decode, ms/token): trigger at kernel entry 2.41 (the successors sit on SM
// resources the running kernel's tail needs), no PDL 1.757, trigger after the last tile is consumed 1.729, trigger from the producer warp
// as soon as every byte of the CTA is requested 1.705 -> that is the default.
// tuning aid: per-launch timeline (DecodeParams::prof), see b200_session_decode_timeline
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void prof_begin(unsigned long long *p) { if (p && threadIdx.x == 0) { const unsigned long long t = gtime(); atomicMin(p, t); atomicMax(p + 3 * B200_PROF_SLOTS, t); } }
__device__ __forceinline__ void prof_ready(unsigned long long *p) { if (p && threadIdx.x == 0) { const unsigned long long t = gtime(); atomicMin(p + 2 * B200_PROF_SLOTS, t); atomicMax(p + 4 * B200_PROF_SLOTS, t); } }
__device__ __forceinline__ void prof_end(unsigned long long *p) { if (p && threadIdx.x == 0) atomicMax(p + B200_PROF_SLOTS, gtime()); }
// a phase boundary: earliest CTA into array kmin (one that holds minima, or -1 for none), latest into array kmax
__device__ __forceinline__ void prof_stamp(unsigned long long *p, int kmin, int kmax) {
    if (p && threadIdx.x == 0) { const unsigned long long t = gtime(); if (kmin >= 0) atomicMin(p + kmin * B200_PROF_SLOTS, t); atomicMax(p + kmax * B200_PROF_SLOTS, t); }
}

__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// B200_PDL: bit 0 = the weight mat-vecs are launched as programmatic dependents, bit 1 = the small kernels between them too (default 3)
int pdl_mask() {
    static int mask = -1;
    if (mask < 0) { const char *e = getenv("B200_PDL"); mask = e ? atoi(e) : 3; }
    return mask;
}
// B200_ATTN_PREFETCH: 1 (default) = the fused attention streams the cached K/V below n_past ahead of its pdl_wait, 0 = every load after it
int attn_prefetch() {
    static int on = -1;
    if (on < 0) { const char *e = getenv("B200_ATTN_PREFETCH"); on = e ? (atoi(e) != 0) : 1; }
    return on;
}

template <int CLASS = 2, typename... KArgs, typename... Args>
void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = (pdl_mask() & CLASS) ? 1 : 0;
    B200_CHECK(cudaLaunchKernelEx(&cfg, kern, KArgs(args)...));
}

__device__ __forceinline__ float lutf(const uint16_t *t, float x) { return f16_bits_to_f32(__ldg(t + f32_to_f16_bits(x))); }
__device__ __forceinline__ float f16dot_tree(float s) {          // ggml_vec_dot_f16 reduction order, see exact.cu
    s = __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 16));
    s = __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 8));
    s = __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 4));
    s = __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 1));
    s = __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 2));
    return s;
}

// ---- 1 / 6: rms_norm * gain -> records.  grid = e/128 CTAs of 256 threads; every CTA reduces the whole row (16 KB from L2) and
//      quantizes its own 4 blocks per warp pass. ------------------------------------------------------------------------------------
template <bool TP>
__device__ __forceinline__ void norm_pack_body(const float *__restrict__ x, const float *__restrict__ gain, int4 *__restrict__ pack,
                                               int e, float eps, int q81, int off, int scale16, unsigned long long *prof, const TpSync &S) {
    const TpCtx &T = c_tp;
    __shared__ double shd[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_trigger();                                              // 4 CTAs: the next mat-vec fits beside this kernel and streams its first stages meanwhile
    // Tensor-parallel: the row arrives as tagged units and the records this kernel overwrites were last read by a mat-vec whose outputs the producers of
    // those units needed (tp.cuh): nothing here depends on the predecessor grid having COMPLETED, only on its units -- do not wait for its peer stores to be acknowledged.
    if (!(TP && (T.relax & 1))) pdl_wait();
    constexpr bool tp = TP;                                    // tensor-parallel: the row is an array of {value, tag} units filled by every rank (tp.cuh)
    const unsigned tag = tp ? tp_tag(T, S.in_v) : 0u;

    prof_begin(prof);
    // this CTA's 32 blocks are float4s [blockIdx.x * 256, +256) of the row: thread tid packs float4 blockIdx.x * 256 + tid, which is also
    // one of the values it sums -- the row is read once, all loads (row and gains) are in flight before the first use (one L2 round trip)
    const int mine = blockIdx.x * 256 + tid, nv = e / 4;
    const bool active = mine < nv;
    const float4 gv = active ? __ldg((const float4 *)gain + mine) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
    double s = 0.0;
    constexpr int U = 4;
    if (tp && (T.relax & 1)) {                                  // launched ahead of the data: warp 0 watches a sample of the row, the others sleep on the barrier
        if (warp == 0) tp_wait_sample(T, S.in_buf, (int64_t)e, tag, lane);
        __syncthreads();
    }
    for (int i0 = tid; i0 < nv; i0 += 256 * U) {
        float4 v[U];
        if (!tp) {
#pragma unroll
            for (int k = 0; k < U; k++) { const int i = i0 + 256 * k; v[k] = i < nv ? __ldcg((const float4 *)x + i) : make_float4(0.f, 0.f, 0.f, 0.f); }   // written by a predecessor: L2-coherent load
        } else {                                                // float4 i = units 4i .. 4i+3 = pairs 2i, 2i+1: all loads first, then the tag checks
            uint4 ra[U], rb[U];
#pragma unroll
            for (int k = 0; k < U; k++) { const int i = i0 + 256 * k; if (i < nv) { ra[k] = tp_ld2(T, S.in_buf, 2 * (int64_t)i); rb[k] = tp_ld2(T, S.in_buf, 2 * (int64_t)i + 1); } }
#pragma unroll
            for (int k = 0; k < U; k++) {
                const int i = i0 + 256 * k;
                if (i < nv) {
                    tp_fix2(T, S.in_buf, 2 * (int64_t)i, tag, ra[k]); tp_fix2(T, S.in_buf, 2 * (int64_t)i + 1, tag, rb[k]);
                    v[k] = make_float4(__uint_as_float(ra[k].x), __uint_as_float(ra[k].z), __uint_as_float(rb[k].x), __uint_as_float(rb[k].z));
                } else v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int k = 0; k < U; k++) {
            if (i0 + 256 * k == mine) xv = v[k];
            s += (double)__fmul_rn(v[k].x, v[k].x); s += (double)__fmul_rn(v[k].y, v[k].y); s += (double)__fmul_rn(v[k].z, v[k].z); s += (double)__fmul_rn(v[k].w, v[k].w);
        }
    }
    s = warp_sum(s);
    if (lane == 0) shd[warp] = s;
    __syncthreads();
    const double tot = ((shd[0] + shd[1]) + (shd[2] + shd[3])) + ((shd[4] + shd[5]) + (shd[6] + shd[7]));
    const float mean = (float)(tot / (double)e);
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, eps)));
    float4 v;
    v.x = __fmul_rn(__fmul_rn(xv.x, scale), gv.x); v.y = __fmul_rn(__fmul_rn(xv.y, scale), gv.y);
    v.z = __fmul_rn(__fmul_rn(xv.z, scale), gv.z); v.w = __fmul_rn(__fmul_rn(xv.w, scale), gv.w);
    pack_quad(v, pack + (active ? mine >> 3 : 0) * 4, lane, active, q81, off, scale16);
    prof_end(prof);
}
// Two entry points: the single-GPU kernel does not carry the 24 bytes of TpSync, so its argument block stays inside ONE 64-byte line of the constant bank
// (56 B; with them, 80 B, the 4-CTA kernel measured +0.2..0.4 us per launch, 64 launches per token: profiles/r02m_timeline*.txt).
__global__ void __launch_bounds__(256) norm_pack_kernel(const float *__restrict__ x, const float *__restrict__ gain, int4 *__restrict__ pack,
                                                        int e, float eps, int q81, int off, int scale16, unsigned long long *prof) {
    norm_pack_body<false>(x, gain, pack, e, eps, q81, off, scale16, prof, TpSync{});
}
__global__ void __launch_bounds__(256) norm_pack_tp_kernel(const float *__restrict__ x, const float *__restrict__ gain, int4 *__restrict__ pack,
                                                           int e, float eps, int q81, int off, int scale16, unsigned long long *prof, const TpSync S) {
    norm_pack_body<true>(x, gain, pack, e, eps, q81, off, scale16, prof, S);
}

// ---- mat-vec with fused epilogues --------------------------------------------------------------------------------------------------
enum { EPI_RES = 0, EPI_QKV = 1, EPI_SILU = 2, EPI_LOGITS = 3, EPI_BIAS = 4, EPI_GELU = 5 };   // BIAS / GELU: GPT-NeoX (bias adds, gelu table)

struct MmvArgs {
    const int4 *xpack;            // input records
    float *dst; const float *addend;                       // EPI_RES / EPI_LOGITS
    // Two pointer groups that no launch uses together share their 32 bytes: the argument block (QWeight 72 B + this struct) then stays within four 64-byte
    // lines of the constant bank (248 B; 280 B with both groups measured +0.2..0.4 us on every launch of the decode graph, profiles/r02_notes.md).
    union {
        struct { float *q; __half *K, *V; const float2 *rope_cs; };                            // EPI_QKV (LLaMA: RoPE + KV store)
        // EPI_BIAS: dst = ((W x + bias) [+ add1]) [+ add2] in that order (ggml_add nodes of gptneox lib.rs:200,302,308-325); EPI_GELU: gelu(W x + bias) quantized
        struct { const float *bias, *add1, *add2; const uint16_t *lut_gelu; };
    };
    int rope_half, hd, e, gqa, n_ctx; const int *n_past;                                      // EPI_QKV
    // EPI_SILU
    int4 *xpack_out; const uint16_t *lut_silu;
    int q81, off, scale16;
    int *n_past_inc;              // EPI_LOGITS: the last node of the token increments InferenceSession::n_past on the device
    int nst;                      // ring depth chosen by launch_mmv
    int pdl_early;                // trigger the dependents from the producer warp once every byte is requested (B200_PDL_EARLY, default 1)
    unsigned long long *prof;
    // tensor-parallel decode (tp.cuh): this rank owns rows [row0, row0 + w.N) of the full matrix; results go to buffer dst_buf of every rank
    TpSync ts; int64_t row0;
};
static_assert(sizeof(QWeight) + sizeof(MmvArgs) <= 256, "mat-vec argument block: at most four 64-byte lines of the constant bank (see the union above)");

template <int TYPE, int EPI, bool TP>
__global__ void __launch_bounds__(STHREADS) mmv_fused_kernel(const QWeight w, const MmvArgs A) {
    const bool pdl_early = A.pdl_early != 0;
    using T = St<TYPE>;
    extern __shared__ __align__(128) uint8_t smem[];
    Ring R{(uint64_t *)smem, (uint64_t *)smem + SST_MAX, smem + 256, 0u, (uint32_t)A.nst};
    int4 *sx = (int4 *)(R.base + T::ring_bytes(A.nst));
    const int tid = threadIdx.x;
    constexpr int G = EPI == EPI_SILU ? 2 : 1;
    prof_begin(A.prof);
    if (tid == 0) ring_init(R.full, R.empty, A.nst);
    __syncthreads();
    if (tid >= SCOMPUTE) {                                      // weights only: runs ahead of the predecessors
        produce_matvec<TYPE>(w, R, blockIdx.x, gridDim.x, tid & 31, G);
        if (pdl_early) pdl_trigger();                           // every byte of this CTA is requested: let the successor's CTAs take the free slots
        return;
    }
    if (!(TP && (c_tp.relax & 2) && A.ts.in_buf >= 0)) pdl_wait();    // records and addend arrive as tagged units: no dependence on the predecessor's completion (tp.cuh)
    if (TP && A.ts.in_buf >= 0) {                 // tensor-parallel: the input records arrive from every rank as {word, tag} units (tp.cuh)
        const unsigned tag = tp_tag(c_tp, A.ts.in_v);
        if (c_tp.relax & 2) {                                   // launched ahead of the data: warp 0 watches a sample, the others sleep on the barrier
            if (tid < 32) tp_wait_sample(c_tp, A.ts.in_buf, (int64_t)w.nb * 16, tag, tid);
            compute_sync();
        }
        const int npair = (int)w.nb * 8;                        // a 16-byte record = 4 units = 2 pairs
        constexpr int U = 8;                                    // 16-byte loads in flight per thread
        for (int i0 = tid; i0 < npair; i0 += SCOMPUTE * U) {
            uint4 v[U];
#pragma unroll
            for (int k = 0; k < U; k++) { const int i = i0 + k * SCOMPUTE; if (i < npair) v[k] = tp_ld2(c_tp, A.ts.in_buf, i); }
#pragma unroll
            for (int k = 0; k < U; k++) {
                const int i = i0 + k * SCOMPUTE;
                if (i < npair) { tp_fix2(c_tp, A.ts.in_buf, i, tag, v[k]); ((uint2 *)sx)[i] = make_uint2(v[k].x, v[k].z); }
            }
        }
    } else {
        for (int i = tid; i < (int)w.nb * 4; i += SCOMPUTE) cp16(smem_u32(sx + i), A.xpack + i);   // all 16-byte copies in flight at once
        asm volatile("cp.async.wait_all;" ::: "memory");
    }
    float *stash = (float *)(sx + (size_t)w.nb * 4);      // 64 floats behind the records (EPI_SILU)
    compute_sync();
    prof_ready(A.prof);
    const int lane = tid & 31, warp = tid >> 5;
    if (EPI == EPI_RES || EPI == EPI_LOGITS) {
        consume_matvec<TYPE>(w, sx, R, blockIdx.x, gridDim.x, tid, [&](int64_t row, float v) {
            if ((tid & 3) != 0 || row >= w.N) return;
            const int64_t g = A.row0 + row;                      // row of the full matrix (row0 = 0 on a single GPU)
            if (TP) {                                            // addend: this rank's own slice of the gathered vector; result: to every rank
                const float out = A.ts.add_buf >= 0 ? __fadd_rn(v, tp_get_f32(c_tp, A.ts.add_buf, g, tp_tag(c_tp, A.ts.add_v))) : v;
                tp_put_f32(c_tp, A.ts.out_buf, g, out, tp_tag(c_tp, A.ts.out_v));
            } else A.dst[g] = A.addend ? __fadd_rn(v, __ldcg(A.addend + g)) : v;
        }, 1, A.prof);
        if (EPI == EPI_LOGITS && blockIdx.x == 0 && tid == 0) *A.n_past_inc = *A.n_past_inc + 1;
    } else if (EPI == EPI_QKV) {
        const int p = __ldcg(A.n_past);
        consume_matvec<TYPE>(w, sx, R, blockIdx.x, gridDim.x, tid, [&](int64_t row, float v) {
            const float other = __shfl_xor_sync(0xffffffffu, v, 4);              // rotation partner: rows 2i, 2i+1 sit in adjacent quads
            if ((tid & 3) != 0 || row >= w.N) return;
            if (row < A.e + A.gqa) {                                               // ggml_rope mode 0 (LC/ggml.c:11859-11874)
                const int within = (int)(row < A.e ? row : row - A.e);
                const float2 cs = __ldg(A.rope_cs + (int64_t)p * A.rope_half + (within % A.hd) / 2);
                const bool even = (row & 1) == 0;
                const float x0 = even ? v : other, x1 = even ? other : v;
                const float out = even ? __fmaf_rn(x0, cs.x, -__fmul_rn(x1, cs.y)) : __fmaf_rn(x0, cs.y, __fmul_rn(x1, cs.x));
                if (row < A.e) A.q[row] = out;
                else A.K[(int64_t)p * A.gqa + within] = __float2half_rn(out);
            } else {
                A.V[(int64_t)(row - A.e - A.gqa) * A.n_ctx + p] = __float2half_rn(v);
            }
        });
    } else if (EPI == EPI_BIAS) {
        consume_matvec<TYPE>(w, sx, R, blockIdx.x, gridDim.x, tid, [&](int64_t row, float v) {
            if ((tid & 3) != 0 || row >= w.N) return;
            float out = A.bias ? __fadd_rn(v, __ldg(A.bias + row)) : v;
            if (A.add1) out = __fadd_rn(out, __ldcg(A.add1 + row));
            if (A.add2) out = __fadd_rn(out, __ldcg(A.add2 + row));
            A.dst[row] = out;
        }, 1, A.prof);
        if (A.n_past_inc && blockIdx.x == 0 && tid == 0) *A.n_past_inc = *A.n_past_inc + 1;
    } else if (EPI == EPI_GELU) {   // one 32-row tile = one quant block of the next mat-vec's input (rows past N: zero activations)
        consume_matvec<TYPE>(w, sx, R, blockIdx.x, gridDim.x, tid, [&](int64_t row, float v) {
            if ((tid & 3) == 0) stash[row & 31] = row < w.N ? __fadd_rn(v, __ldg(A.bias + row)) : 0.f;
            compute_sync();
            if (warp == 0) {
                const float4 a = ((const float4 *)stash)[lane & 7];
                float4 hm;
                hm.x = lutf(A.lut_gelu, a.x); hm.y = lutf(A.lut_gelu, a.y); hm.z = lutf(A.lut_gelu, a.z); hm.w = lutf(A.lut_gelu, a.w);
                pack_quad(hm, A.xpack_out + (row >> 5) * 4, lane, lane < 8, A.q81, A.off, A.scale16);
            }
            compute_sync();
        }, 1, A.prof);
    } else {   // EPI_SILU
        consume_matvec<TYPE>(w, sx, R, blockIdx.x, gridDim.x, tid, [&](int64_t row, float v) {
            if ((tid & 3) == 0) stash[row & 63] = v;
            if (((row >> 5) & 1) == 0) return;
            compute_sync();
            if (warp == 0) {
                const int w8 = lane & 7;
                const float4 a = ((const float4 *)stash)[w8], b = ((const float4 *)stash)[8 + w8];
                float4 hm;
                hm.x = __fmul_rn(lutf(A.lut_silu, a.x), b.x); hm.y = __fmul_rn(lutf(A.lut_silu, a.y), b.y);
                hm.z = __fmul_rn(lutf(A.lut_silu, a.z), b.z); hm.w = __fmul_rn(lutf(A.lut_silu, a.w), b.w);
                const int64_t blk = (A.row0 >> 6) + (row >> 6);     // block of w2's input (row0 counts this rank's interleaved w1|w3 rows)
                int4 rec;
                if (pack_quad_rec(hm, lane, lane < 8, A.q81, A.off, A.scale16, rec)) {
                    if (TP) tp_put_rec(c_tp, TPB_XF, blk * 4 + (lane & 7), rec, tp_tag(c_tp, A.ts.out_v)); else A.xpack_out[blk * 4 + (lane & 7)] = rec;
                }
            }
            compute_sync();
        }, G, A.prof);
    }
    pdl_trigger();                                              // late: this CTA has consumed its last tile
    prof_end(A.prof);
}

// ---- 3: KQ.  CTA = (64 cached positions, head); CTAs past n_kv exit at once (the grid is sized for the context bucket).  All
//      16-byte loads of the K tile are issued before the first one is consumed. ---------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(128) attn_kq_kernel(const float *__restrict__ q, const __half *__restrict__ Kl, float *__restrict__ kq,
                                                      const int *__restrict__ n_past, int gqa, int n_head, int n_head_kv, int n_ctx, unsigned long long *prof) {
    __shared__ __align__(16) __half q16[HD];
    __shared__ __align__(16) __half kt[64 * HD];
    pdl_trigger();
    pdl_wait();
    prof_begin(prof);
    const int n_kv = __ldcg(n_past) + 1;
    const int j0 = blockIdx.x * 64, h = blockIdx.y;
    if (j0 >= n_kv) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int hk = h / (n_head / n_head_kv);
    const int rows = n_kv - j0 < 64 ? n_kv - j0 : 64;
    constexpr int VPR = HD / 8;                       // 16-byte vectors per K row
    constexpr int NV = 64 * VPR / 128;                // vectors per thread
    int4 v[NV];
#pragma unroll
    for (int u = 0; u < NV; u++) {
        const int i = tid + u * 128, rr = i / VPR, cc = i % VPR;
        v[u] = rr < rows ? __ldcg((const int4 *)(Kl + (int64_t)(j0 + rr) * gqa + hk * HD) + cc) : make_int4(0, 0, 0, 0);
    }
    for (int i = tid; i < HD; i += 128) q16[i] = __float2half_rn(__ldcg(q + h * HD + i));
#pragma unroll
    for (int u = 0; u < NV; u++) ((int4 *)kt)[tid + u * 128] = v[u];
    __syncthreads();
    for (int jj = warp; jj < rows; jj += 4) {
        const __half *krow = kt + jj * HD;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < HD; k += 32) s = __fmaf_rn(__half2float(krow[k + lane]), __half2float(q16[k + lane]), s);
        s = f16dot_tree(s);
        if (lane == 0) kq[(int64_t)h * n_ctx + j0 + jj] = (float)(double)s;
    }
    prof_end(prof);
}

// ---- 4: scale + soft_max + KQV for 32 channels of one head, then quantize those 32 outputs (one block of wo's input) ---------------
constexpr int KC = 128;
__global__ void __launch_bounds__(128) attn_sv_kernel(const float *__restrict__ kq, const __half *__restrict__ Vl, int4 *__restrict__ xpack_out,
                                                      const int *__restrict__ n_past, const uint16_t *__restrict__ lut_exp, float kq_scale,
                                                      int hd, int n_head, int n_head_kv, int n_ctx, int q81, int off, int scale16, unsigned long long *prof) {
    extern __shared__ __align__(16) uint8_t sm[];
    __shared__ double shd[8];
    __shared__ float shf[4], stash[32];
    pdl_trigger();
    pdl_wait();
    prof_begin(prof);
    const int n_kv = __ldcg(n_past) + 1;
    const int per_head = hd / 32, h = blockIdx.x / per_head, c0 = (blockIdx.x - h * per_head) * 32;
    const int hk = h / (n_head / n_head_kv);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *sc = (float *)sm;
    __half *p16 = (__half *)(sm + (size_t)n_ctx * 4);
    __half *vt = (__half *)(sm + (size_t)n_ctx * 6);
    __half *vleft = vt + 32 * KC;
    // leftover V columns and the first V tile are requested before anything else so that their latency hides behind the soft_max
    const int np = n_kv & ~31;
    if (np < n_kv) {
        const int rr = tid >> 2, part = tid & 3;
        ((int4 *)vleft)[tid] = __ldcg((const int4 *)(Vl + (int64_t)(hk * hd + c0 + rr) * n_ctx + np) + part);
    }
    int4 pre[KC / 32];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int u = 0; u < KC / 32; u++) {
            const int i = tid + u * 128, rr = i / (KC / 8), cc = i - rr * (KC / 8);
            pre[u] = __ldcg((const int4 *)(Vl + (int64_t)(hk * hd + c0 + rr) * n_ctx + k0) + cc);
        }
    };
    if (np > 0) fetch(0);
    float mx = -INFINITY;
    constexpr int SB = 8;                              // scores per thread per pass: 8 loads in flight
    for (int jb = 0; jb < n_kv; jb += SB * 128) {
        float sv[SB];
#pragma unroll
        for (int u = 0; u < SB; u++) { const int j = jb + tid + u * 128; sv[u] = j < n_kv ? __ldcg(kq + (int64_t)h * n_ctx + j) : 0.f; }
#pragma unroll
        for (int u = 0; u < SB; u++) { const int j = jb + tid + u * 128; if (j < n_kv) { const float v = __fmul_rn(sv[u], kq_scale); sc[j] = v; mx = fmaxf(mx, v); } }
    }
    mx = warp_max(mx);
    if (lane == 0) shf[warp] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(shf[0], shf[1]), fmaxf(shf[2], shf[3]));
    double s = 0.0;
    for (int jb = 0; jb < n_kv; jb += SB * 128) {
        uint16_t ev16[SB];
#pragma unroll
        for (int u = 0; u < SB; u++) { const int j = jb + tid + u * 128; ev16[u] = j < n_kv ? __ldg(lut_exp + f32_to_f16_bits(__fsub_rn(sc[j], mx))) : (uint16_t)0; }
#pragma unroll
        for (int u = 0; u < SB; u++) { const int j = jb + tid + u * 128; if (j < n_kv) { const float ev = f16_bits_to_f32(ev16[u]); sc[j] = ev; s += (double)ev; } }
    }
    s = warp_sum(s);
    if (lane == 0) shd[warp] = s;
    __syncthreads();
    const float inv = (float)(1.0 / ((shd[0] + shd[1]) + (shd[2] + shd[3])));
    for (int j = tid; j < n_kv; j += 128) p16[j] = __float2half_rn(__fmul_rn(sc[j], inv));
    float acc[8];
#pragma unroll
    for (int cc = 0; cc < 8; cc++) acc[cc] = 0.f;
    for (int k0 = 0; k0 < np; k0 += KC) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < KC / 32; u++) ((int4 *)vt)[tid + u * 128] = pre[u];
        __syncthreads();
        if (k0 + KC < np) fetch(k0 + KC);
        const int kend = np - k0 < KC ? np - k0 : KC;
#pragma unroll
        for (int cc = 0; cc < 8; cc++) {
            const __half *vrow = vt + (warp * 8 + cc) * KC;
            for (int k = lane; k < kend; k += 32) acc[cc] = __fmaf_rn(__half2float(vrow[k]), __half2float(p16[k0 + k]), acc[cc]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < 8; cc++) {
        const float a = f16dot_tree(acc[cc]);
        if (lane == 0) {
            const __half *vrow = vleft + (warp * 8 + cc) * 32;
            double sumf = (double)a;
            for (int k = np; k < n_kv; k++) sumf += (double)__fmul_rn(__half2float(vrow[k - np]), __half2float(p16[k]));
            stash[warp * 8 + cc] = (float)sumf;
        }
    }
    __syncthreads();
    if (warp == 0) pack_quad(((const float4 *)stash)[lane & 7], xpack_out + (int64_t)((h * hd + c0) / QK) * 4, lane, lane < 8, q81, off, scale16);
    prof_end(prof);
}

// ---- 3+4 fused: KQ, scale, soft_max, KQV and the quantize epilogue for one head, as ONE cluster of hd/32 CTAs ----------------------------
// CTA `part` of the cluster owns 32 channels of the head (its V rows are staged by cp.async at kernel entry, long before they are needed)
// and 1/(hd/32) of the cached positions for KQ; the scaled scores are written straight into every CTA's shared memory (DSMEM) and one
// cluster barrier later each CTA runs the soft_max on the full row and its own 32 KQV dots.  No global round trip between the phases.
//
// ggml_vec_dot_f16 (LC/ggml.c:1573-1610) keeps 32 f32 chains, chain l over elements k = l (mod 32); here thread u (0..3) of a quad owns
// chains 8u..8u+7 of one dot, so every load is a 16-byte vector, and the reduction tree (offsets 16, 8, 4, 1, 2) is two quad shuffles plus
// in-thread adds in exactly that association.
__device__ __forceinline__ float quad_tree(float (&acc)[8]) {
#pragma unroll
    for (int e = 0; e < 8; e++) acc[e] = __fadd_rn(acc[e], __shfl_xor_sync(0xffffffffu, acc[e], 2));     // chain l += chain l + 16
#pragma unroll
    for (int e = 0; e < 8; e++) acc[e] = __fadd_rn(acc[e], __shfl_xor_sync(0xffffffffu, acc[e], 1));     // l += l + 8   (valid in u == 0)
    const float r0 = __fadd_rn(acc[0], acc[4]), r1 = __fadd_rn(acc[1], acc[5]), r2 = __fadd_rn(acc[2], acc[6]), r3 = __fadd_rn(acc[3], acc[7]);   // l += l + 4
    return __fadd_rn(__fadd_rn(r0, r1), __fadd_rn(r2, r3));                                                // down 1, down 2
}
__device__ __forceinline__ void fma8(float (&acc)[8], const int4 &a, const int4 &b) {
    const __half2 *ah = (const __half2 *)&a, *bh = (const __half2 *)&b;
#pragma unroll
    for (int e = 0; e < 4; e++) {
        const float2 af = __half22float2(ah[e]), bf = __half22float2(bh[e]);
        acc[2 * e] = __fmaf_rn(af.x, bf.x, acc[2 * e]); acc[2 * e + 1] = __fmaf_rn(af.y, bf.y, acc[2 * e + 1]);
    }
}

constexpr int ATH = 256;
template <bool TP>
__global__ void __launch_bounds__(ATH) attn_fused_kernel(const float *__restrict__ q, const __half *__restrict__ Kl, const __half *__restrict__ Vl,
                                                         int4 *__restrict__ xpack_out, const int *__restrict__ n_past, const uint16_t *__restrict__ lut_exp,
                                                         float kq_scale, int hd, int n_head, int n_head_kv, int gqa, int n_ctx, int nlay, int q81, int off, int scale16,
                                                         unsigned long long *prof, const TpSync S, int head0, int prefetch) {
    const TpCtx &T = c_tp;
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) uint8_t sm[];
    __shared__ double shd[ATH / 32];
    __shared__ float shf[ATH / 32], stash[32];
    prof_begin(prof);
    const int per_head = hd / 32, h = blockIdx.x / per_head, part = blockIdx.x - h * per_head, c0 = part * 32;
    const int hk = h / (n_head / n_head_kv);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, u = tid & 3;
    // shared-memory layout for nlay >= n_kv positions (the context bucket the graph was captured for, a multiple of 64: small enough that the
    // next mat-vec's CTAs fit beside this kernel's and stream their weights while it runs)
    const int vstride = nlay + 32;                              // halves; (nlay + 32) * 2 B = 64 B mod 128 B: the two columns of a quarter-warp hit different banks
    float *sc = (float *)sm;
    __half *p16 = (__half *)(sm + (size_t)nlay * 4);
    __half *q16 = p16 + nlay;
    __half *vs = (__half *)(sm + (((size_t)nlay * 6 + (size_t)hd * 2 + 127) & ~(size_t)127));
    pdl_trigger();                                              // the successor (wo) only needs shared memory beside us: let it prefetch its tiles now
    if (!prefetch) { pdl_wait(); prof_ready(prof); }
    // With `prefetch`, everything up to the pdl_wait below runs while the QKV launch is still finishing: it reads only what that launch does
    // not write (the rule at the top of this file).  The K row and the V column at n_past are the QKV launch's output: loaded after the wait.
    const int n_kv = __ldcg(n_past) + 1, p = n_kv - 1;
    const int np = n_kv & ~31;

    // V rows of this CTA's 32 channels: all copies in flight at once, consumed after the soft_max
    const int cpr = (n_kv + 7) / 8;                              // 16-byte chunks per row
    auto copy_v = [&](int c_lo, int c_hi) {
        const int nc = c_hi - c_lo;
        for (int i = tid; i < 32 * nc; i += ATH) {
            const int rr = i / nc, cc = c_lo + i - rr * nc;
            cp16(smem_u32(vs + rr * vstride + cc * 8), Vl + (int64_t)(hk * hd + c0 + rr) * n_ctx + cc * 8);
        }
    };
    const int vpre = prefetch ? p / 8 : 0;                       // chunks that lie entirely below column n_past

    // KQ for this CTA's share [j0, j1) of the positions, one pass = PU positions per quad; pass 0's K rows below n_past are loaded now
    const int per = (n_kv + per_head - 1) / per_head, j0 = part * per, j1 = n_kv < j0 + per ? n_kv : j0 + per;
    const int nvec = hd / 32;                                    // 16-byte loads per thread per position (chunks i = 0..nvec-1)
    constexpr int PU = 4;                                        // positions per quad per pass: up to 4 * nvec 16-byte loads in flight per thread
    int4 kv[PU][4];
    auto load_k = [&](int jb, int jend) {                        // rows j < jend (<= j1) of the pass at jb, zeros from there on
#pragma unroll
        for (int pu = 0; pu < PU; pu++) {
            const int j = jb + pu * (ATH / 4) + (tid >> 2);
            const __half *krow = Kl + (int64_t)(j < jend ? j : j0) * gqa + hk * hd + 8 * u;
#pragma unroll
            for (int i = 0; i < 4; i++) if (i < nvec) kv[pu][i] = j < jend ? __ldcg((const int4 *)(krow + 32 * i)) : make_int4(0, 0, 0, 0);
        }
    };
    // K first: the scores need it long before KQV needs V, and loads issued behind the V burst queue behind it
    load_k(j0, prefetch ? (p < j1 ? p : j1) : 0);
    copy_v(0, vpre);
    // every CTA of the cluster is running before its shared memory is written remotely (no data is exchanged yet, so the cluster barrier
    // can be the relaxed one: no fence)
    asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
    if (prefetch) { pdl_wait(); prof_ready(prof); }

    float qv = 0.f;
    if (tid < hd) qv = __ldcg(q + h * hd + tid);               // hd <= 256 = ATH
    if (!prefetch) load_k(j0, j1);
    else {                                                       // row n_past, if it lies in pass 0 (past j1 too: that score is not stored, and
#pragma unroll                                                   // the guard would cost 16 registers)
        for (int pu = 0; pu < PU; pu++)
            if (j0 + pu * (ATH / 4) + (tid >> 2) == p) {
                const __half *krow = Kl + (int64_t)p * gqa + hk * hd + 8 * u;
#pragma unroll
                for (int i = 0; i < 4; i++) if (i < nvec) kv[pu][i] = __ldcg((const int4 *)(krow + 32 * i));
            }
    }
    copy_v(vpre, cpr);
    if (tid < hd) q16[tid] = __float2half_rn(qv);
    __syncthreads();                                             // q16 visible inside the CTA

    for (int jb = j0; jb < j1; jb += PU * (ATH / 4)) {
        if (jb != j0) load_k(jb, j1);
#pragma unroll
        for (int pu = 0; pu < PU; pu++) {
            const int j = jb + pu * (ATH / 4) + (tid >> 2);
            float acc[8];
#pragma unroll
            for (int e = 0; e < 8; e++) acc[e] = 0.f;
#pragma unroll
            for (int i = 0; i < 4; i++) if (i < nvec) fma8(acc, kv[pu][i], *(const int4 *)(q16 + 32 * i + 8 * u));
            const float s = quad_tree(acc);
            if (j < j1 && u < per_head) cluster.map_shared_rank(sc, u)[j] = __fmul_rn(s, kq_scale);   // thread u of the quad feeds CTA u
        }
    }
    prof_stamp(prof, 5, 6);                                      // this CTA's K rows have landed and its scores are out
    cluster.sync();
    prof_stamp(prof, -1, 7);

    // ---- soft_max over sc[0, n_kv) (ggml_compute_forward_soft_max_f32, LC/ggml.c:11700-11770: fp16 exp table, double row sum) ----
    float mx = -INFINITY;
    for (int j = tid; j < n_kv; j += ATH) mx = fmaxf(mx, sc[j]);
    mx = warp_max(mx);
    if (lane == 0) shf[warp] = mx;
    __syncthreads();
    mx = shf[0];
#pragma unroll
    for (int i = 1; i < ATH / 32; i++) mx = fmaxf(mx, shf[i]);
    double s = 0.0;
    constexpr int SB = 4;                                        // table look-ups in flight per thread
    for (int jb = 0; jb < n_kv; jb += SB * ATH) {
        uint16_t ev16[SB];
#pragma unroll
        for (int k = 0; k < SB; k++) { const int j = jb + tid + k * ATH; ev16[k] = j < n_kv ? __ldg(lut_exp + f32_to_f16_bits(__fsub_rn(sc[j], mx))) : (uint16_t)0; }
#pragma unroll
        for (int k = 0; k < SB; k++) { const int j = jb + tid + k * ATH; if (j < n_kv) { const float ev = f16_bits_to_f32(ev16[k]); sc[j] = ev; s += (double)ev; } }
    }
    s = warp_sum(s);
    if (lane == 0) shd[warp] = s;
    __syncthreads();
    const float inv = (float)(1.0 / (((shd[0] + shd[1]) + (shd[2] + shd[3])) + ((shd[4] + shd[5]) + (shd[6] + shd[7]))));
    for (int j = tid; j < n_kv; j += ATH) p16[j] = __float2half_rn(__fmul_rn(sc[j], inv));
    prof_stamp(prof, -1, 8);
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    // ---- KQV: 32 channels x 4 threads ----
    if (tid < 128) {
        const int col = tid >> 2;
        const __half *vrow = vs + col * vstride;
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; e++) acc[e] = 0.f;
#pragma unroll 4
        for (int k = 0; k < np; k += 32) fma8(acc, *(const int4 *)(vrow + k + 8 * u), *(const int4 *)(p16 + k + 8 * u));
        const float a = quad_tree(acc);
        if (u == 0) {
            double sumf = (double)a;
            for (int k = np; k < n_kv; k++) sumf += (double)__fmul_rn(__half2float(vrow[k]), __half2float(p16[k]));
            stash[col] = (float)sumf;
        }
    }
    __syncthreads();
    if (warp == 0) {
        int4 rec;
        const int64_t blk = (int64_t)(((head0 + h) * hd + c0) / QK);       // block of wo's input: heads are global (head0 = first head of this rank)
        if (pack_quad_rec(((const float4 *)stash)[lane & 7], lane, lane < 8, q81, off, scale16, rec)) {
            if (TP) tp_put_rec(T, TPB_XD, blk * 4 + (lane & 7), rec, tp_tag(T, S.out_v)); else xpack_out[blk * 4 + (lane & 7)] = rec;
        }
    }
    prof_end(prof);
}

template <int TYPE, int EPI, bool TP = false>
void launch_mmv(const QWeight &w, MmvArgs A, cudaStream_t st) {
    constexpr int ROWS = SR, CB = SCB;
    using T = St<TYPE>;
    static int smem_set = 0, sms = 0, depth_cap = -1;
    static std::map<int, std::array<int, SST_MAX + 1>> occ_by_nb;
    if (!sms) { int dev; B200_CHECK(cudaGetDevice(&dev)); B200_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)); }
    if (depth_cap < 0) { const char *e = getenv("B200_RING_DEPTH"); depth_cap = e ? atoi(e) : SST_MAX; if (depth_cap < 2) depth_cap = 2; if (depth_cap > SST_MAX) depth_cap = SST_MAX; }
    auto smem_of = [&](int nst) { return 256 + T::ring_bytes(nst) + (int)w.nb * 64 + 256; };
    if (smem_of(SST_MAX) > smem_set) {
        const int want = smem_of(SST_MAX) < 227 * 1024 ? smem_of(SST_MAX) : 227 * 1024;
        B200_CHECK(cudaFuncSetAttribute(mmv_fused_kernel<TYPE, EPI, TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, want));
        smem_set = smem_of(SST_MAX);
    }
    auto it = occ_by_nb.find((int)w.nb);
    if (it == occ_by_nb.end()) {                                          // CTAs per SM for every ring depth at this activation length
        std::array<int, SST_MAX + 1> o{};
        for (int nst = 2; nst <= SST_MAX; nst++)
            if (smem_of(nst) <= 227 * 1024) B200_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o[nst], mmv_fused_kernel<TYPE, EPI, TP>, STHREADS, smem_of(nst)));
        it = occ_by_nb.emplace((int)w.nb, o).first;
    }
    const std::array<int, SST_MAX + 1> &occ = it->second;
    constexpr int G = EPI == EPI_SILU ? 2 : 1;
    const int64_t groups = ((w.N + ROWS - 1) / ROWS + G - 1) / G;
    // Ring depth: the deepest ring that still keeps every row group resident at once (more bytes in flight per CTA: the small matrices
    // -- 128 groups for 148 SMs -- are bound by HBM round trips per CTA, not by bandwidth); never deeper than one group's chunk count.
    const int chunks = (int)((w.nb + CB - 1) / CB) * G;
    const int base = SST < depth_cap ? SST : depth_cap;
    int nst = base;
    B200_ASSERT(occ[nst] > 0);
    const int64_t need = groups < (int64_t)sms * occ[base] ? groups : (int64_t)sms * occ[base];
    for (int c = base + 1; c <= depth_cap && c <= chunks; c++)
        if (occ[c] > 0 && (int64_t)sms * occ[c] >= need) nst = c;
    A.nst = nst;
    { static int pe = -1; if (pe < 0) { const char *e = getenv("B200_PDL_EARLY"); pe = e ? atoi(e) : 1; } A.pdl_early = pe; }
    const int64_t slots = (int64_t)sms * occ[nst];
    launch_k<1>(mmv_fused_kernel<TYPE, EPI, TP>, dim3((unsigned)(groups < slots ? groups : slots)), dim3(STHREADS), (size_t)smem_of(nst), st, w, A);
}

// dynamic shared memory of the cluster attention kernel for a context bucket (attn_fused_kernel's layout): f32 scores, f16 probabilities and q16,
// rounded to 128 B, then 32 staged V rows of nlay + 32 halves
size_t attn_fused_smem(int n_kv_bucket, int hd) {
    const size_t nlay = (size_t)(n_kv_bucket + 63) / 64 * 64;
    return ((nlay * 6 + (size_t)hd * 2 + 127) & ~(size_t)127) + (size_t)32 * (nlay + 32) * 2;
}

// dynamic shared memory opt-in of the cluster attention kernel: one high-water mark for both instantiations (the attribute is per function, not per caller)
static void attn_fused_reserve(size_t bytes) {
    static size_t set = 48 * 1024;
    if (bytes <= set) return;
    B200_CHECK(cudaFuncSetAttribute(attn_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    B200_CHECK(cudaFuncSetAttribute(attn_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    set = bytes;
}

// tensor-parallel helpers (tp.cuh).  spread: the embedding row every rank computed for itself -> the X exchange buffer's unit form (stamp 0);
// collect: the gathered logits units -> the plain f32 logits array the host reads; bump: the token is complete, the epoch moves on.
__global__ void __launch_bounds__(256) tp_spread_kernel(const float *__restrict__ x, int n) {
    const TpCtx &T = c_tp;
    pdl_wait();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    uint2 *dst = (uint2 *)(T.peer[T.rank] + T.off[TPB_X]) + i;
    *dst = make_uint2(__float_as_uint(__ldcg(x + i)), tp_tag(T, 0));
}
__global__ void __launch_bounds__(256) tp_collect_kernel(float *__restrict__ logits, int n) {
    const TpCtx &T = c_tp;
    pdl_wait();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) logits[i] = tp_get_f32(T, TPB_LOGITS, i, tp_tag(T, 0));
}
__global__ void tp_bump_kernel() {
    const TpCtx &T = c_tp;
    pdl_wait();
    if (threadIdx.x == 0) *T.epoch = *(volatile unsigned *)T.epoch + 1;
}

template <int TYPE, bool TP>
void decode_ops_t(const DecodeParams &P, const std::vector<DecodeLayer> &layers, int n_kv_bucket, int4 *xpack_a, cudaStream_t st, int *launches) {
    const int q81 = has_min(TYPE) ? 1 : 0, off = TYPE == T_Q5_0 ? 16 : 0, s16 = TYPE == T_Q4_0 ? 1 : 0;
    const int e = P.e, f = P.f;
    const TpCtx &T = P.tp;
    constexpr bool tp = TP;
    B200_ASSERT(tp == (T.world > 1));
    const int e_loc = tp ? P.e_loc : e;
    // layer stamps (tp.cuh): X carries stamp il when it enters layer il (0 = the embedding), il + 1 when layer il leaves it; FF / XD / XF of layer il carry il + 1
    auto ts = [&](int in_buf, unsigned in_v, int add_buf, unsigned add_v, int out_buf, unsigned out_v) {
        TpSync S;
        if (tp) { S.in_buf = in_buf; S.in_v = in_v; S.add_buf = add_buf; S.add_v = add_v; S.out_buf = out_buf; S.out_v = out_v; }
        return S;
    };
    int n = 0;
    auto pr = [&]() -> unsigned long long * { return P.prof && n < B200_PROF_SLOTS ? P.prof + n : nullptr; };   // timeline slot of the next launch
    auto launch_norm = [&](const float *x, const float *gain, const TpSync &S) {               // rms_norm * gain -> records of the next mat-vec
        const dim3 grid((e / QK + 31) / 32), block(256);
        if constexpr (TP) launch_k(norm_pack_tp_kernel, grid, block, 0, st, x, gain, xpack_a, e, P.eps, q81, off, s16, pr(), S);
        else { (void)S; launch_k(norm_pack_kernel, grid, block, 0, st, x, gain, xpack_a, e, P.eps, q81, off, s16, pr()); }
        n++;
    };
    get_rows_q(P.wte, P.token, P.x, 1, st); n++;
    if (tp) { launch_k(tp_spread_kernel, dim3((e + 255) / 256), dim3(256), 0, st, (const float *)P.x, e); n++; }
    // attention: one cluster launch per layer (default) or the two-kernel variant (B200_ATTN_FUSED=0, head sizes a cluster cannot cover, or a
    // context bucket whose scores and V rows do not fit one CTA's shared memory: past 3072 positions)
    static const bool fused_env = !(getenv("B200_ATTN_FUSED") && getenv("B200_ATTN_FUSED")[0] == '0');
    const int nlay = (n_kv_bucket + 63) / 64 * 64;
    const size_t fa_smem = attn_fused_smem(n_kv_bucket, P.hd);
    const bool fused_attn = (fused_env || tp) && P.hd % 32 == 0 && P.hd <= 128 && P.n_ctx % 8 == 0 && attn_fused_fits(n_kv_bucket, P.hd);
    // the tensor-parallel exchange lives in the fused attention kernel's epilogue; start_session_tp refuses a context whose buckets do not all fit
    B200_ASSERT(fused_attn || !tp);
    if (fused_attn) attn_fused_reserve(fa_smem);
    const size_t sv_smem = (size_t)P.n_ctx * 6 + 32 * KC * 2 + 32 * 32 * 2;
    static size_t sv_set = 48 * 1024;
    if (sv_smem > sv_set) { B200_CHECK(cudaFuncSetAttribute(attn_sv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sv_smem)); sv_set = sv_smem; }
    for (int il = 0; il < P.n_layer; il++) {
        const DecodeLayer &L = layers[il];
        const unsigned v = (unsigned)il + 1;                     // flag value of this layer's exchanges (tp.cuh)
        launch_norm(P.x, L.attn_norm, ts(TPB_X, (unsigned)il, -1, 0, -1, 0));
        MmvArgs A{}; A.xpack = xpack_a; A.q = P.q; A.K = L.K; A.V = L.V; A.rope_cs = P.rope_cs; A.rope_half = P.rope_half; A.hd = P.hd; A.e = e_loc; A.gqa = P.gqa;
        A.n_ctx = P.n_ctx; A.n_past = P.n_past;
        A.prof = pr(); launch_mmv<TYPE, EPI_QKV, TP>(L.wqkv, A, st); n++;
        if (fused_attn) {
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(P.n_head * (P.hd / 32)); cfg.blockDim = dim3(ATH); cfg.dynamicSmemBytes = fa_smem; cfg.stream = st;
            cudaLaunchAttribute at[2];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = P.hd / 32; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[1].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at; cfg.numAttrs = (pdl_mask() & 2) ? 2 : 1;
            B200_CHECK(cudaLaunchKernelEx(&cfg, attn_fused_kernel<TP>, (const float *)P.q, (const __half *)L.K, (const __half *)L.V, P.xpack_d, (const int *)P.n_past,
                                          (const uint16_t *)P.lut_exp, P.kq_scale, P.hd, P.n_head, P.n_head_kv, P.gqa, P.n_ctx, nlay, q81, off, s16, pr(),
                                          ts(-1, 0, -1, 0, TPB_XD, v), tp ? P.head0 : 0, attn_prefetch()));
            n++;
        } else {
            launch_k(P.hd == 128 ? attn_kq_kernel<128> : attn_kq_kernel<64>, dim3((n_kv_bucket + 63) / 64, P.n_head), dim3(128), 0, st,
                     P.q, L.K, P.kq, P.n_past, P.gqa, P.n_head, P.n_head_kv, P.n_ctx, pr());
            n++;
            launch_k(attn_sv_kernel, dim3(P.n_head * (P.hd / 32)), dim3(128), sv_smem, st, P.kq, L.V, P.xpack_d, P.n_past, P.lut_exp, P.kq_scale, P.hd, P.n_head,
                     P.n_head_kv, P.n_ctx, q81, off, s16, pr()); n++;
        }
        MmvArgs Bo{}; Bo.xpack = P.xpack_d; Bo.dst = P.ff; Bo.addend = P.x;
        Bo.ts = ts(TPB_XD, v, TPB_X, (unsigned)il, TPB_FF, v); Bo.row0 = tp ? P.row0_e : 0;
        Bo.prof = pr(); launch_mmv<TYPE, EPI_RES, TP>(L.wo, Bo, st); n++;
        launch_norm(P.ff, L.ffn_norm, ts(TPB_FF, v, -1, 0, -1, 0));
        MmvArgs C{}; C.xpack = xpack_a; C.xpack_out = P.xpack_f; C.lut_silu = P.lut_silu; C.q81 = q81; C.off = off; C.scale16 = s16;
        C.ts = ts(-1, 0, -1, 0, TPB_XF, v); C.row0 = tp ? P.row0_w13 : 0;
        C.prof = pr(); launch_mmv<TYPE, EPI_SILU, TP>(L.w13, C, st); n++;
        MmvArgs D{}; D.xpack = P.xpack_f; D.dst = P.x; D.addend = P.ff;
        D.ts = ts(TPB_XF, v, TPB_FF, v, TPB_X, v); D.row0 = tp ? P.row0_e : 0;
        D.prof = pr(); launch_mmv<TYPE, EPI_RES, TP>(L.w2, D, st); n++;
    }
    launch_norm(P.x, P.norm, ts(TPB_X, (unsigned)P.n_layer, -1, 0, -1, 0));
    MmvArgs Z{}; Z.xpack = xpack_a; Z.dst = P.logits; Z.addend = nullptr; Z.n_past_inc = P.n_past;
    Z.ts = ts(-1, 0, -1, 0, TPB_LOGITS, 0); Z.row0 = tp ? P.row0_v : 0;
    Z.prof = pr(); launch_mmv<TYPE, EPI_LOGITS, TP>(P.output, Z, st); n++;
    if (tp) {                                                    // gathered logits -> the plain array the host reads; then the epoch moves on
        launch_k(tp_collect_kernel, dim3((P.n_vocab_full + 255) / 256), dim3(256), 0, st, P.logits, P.n_vocab_full); n++;
        launch_k(tp_bump_kernel, dim3(1), dim3(32), 0, st); n++;
    }
    B200_CHECK(cudaGetLastError());
    (void)f;
    if (launches) *launches = n;
}

// ---- GPT-NeoX --------------------------------------------------------------------------------------------------------------------------------
// LayerNorm (ggml_compute_forward_norm_f32, LC/ggml.c:10063-10111) * gain + bias -> Q8 records.  Same shape as norm_pack_kernel: every CTA reduces
// the whole row from registers (two passes: mean, then the variance of the centred values) and packs its own 32 blocks.
__global__ void __launch_bounds__(256) ln_pack_kernel(const float *__restrict__ x, const float *__restrict__ gain, const float *__restrict__ bias, int4 *__restrict__ pack,
                                                      int e, int q81, int off, int scale16) {
    __shared__ double shd[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_trigger();
    pdl_wait();
    constexpr int MAXV = 8;                                     // n_embd <= 8192
    const int nv = e / 4, mine = blockIdx.x * 256 + tid;
    float4 v[MAXV];
#pragma unroll
    for (int k = 0; k < MAXV; k++) { const int i = tid + k * 256; v[k] = i < nv ? __ldcg((const float4 *)x + i) : make_float4(0.f, 0.f, 0.f, 0.f); }
    const bool active = mine < nv;
    const float4 gv = active ? __ldg((const float4 *)gain + mine) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 bv = active ? __ldg((const float4 *)bias + mine) : make_float4(0.f, 0.f, 0.f, 0.f);
    auto total = [&](double s) {
        s = warp_sum(s);
        __syncthreads();
        if (lane == 0) shd[warp] = s;
        __syncthreads();
        return ((shd[0] + shd[1]) + (shd[2] + shd[3])) + ((shd[4] + shd[5]) + (shd[6] + shd[7]));
    };
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < MAXV; k++) if (tid + k * 256 < nv) { s += (double)v[k].x; s += (double)v[k].y; s += (double)v[k].z; s += (double)v[k].w; }
    const float mean = (float)(total(s) / (double)e);
    double s2 = 0.0;
    float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < MAXV; k++) if (tid + k * 256 < nv) {
        float4 c;
        c.x = __fsub_rn(v[k].x, mean); c.y = __fsub_rn(v[k].y, mean); c.z = __fsub_rn(v[k].z, mean); c.w = __fsub_rn(v[k].w, mean);
        s2 += (double)__fmul_rn(c.x, c.x); s2 += (double)__fmul_rn(c.y, c.y); s2 += (double)__fmul_rn(c.z, c.z); s2 += (double)__fmul_rn(c.w, c.w);
        if (k == (int)blockIdx.x) xv = c;                       // float4 index tid + k * 256 == mine
    }
    const float variance = (float)(total(s2) / (double)e);
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(variance, 1e-5f)));
    float4 y;
    y.x = __fadd_rn(__fmul_rn(__fmul_rn(xv.x, scale), gv.x), bv.x); y.y = __fadd_rn(__fmul_rn(__fmul_rn(xv.y, scale), gv.y), bv.y);
    y.z = __fadd_rn(__fmul_rn(__fmul_rn(xv.z, scale), gv.z), bv.z); y.w = __fadd_rn(__fmul_rn(__fmul_rn(xv.w, scale), gv.w), bv.w);
    pack_quad(y, pack + (active ? mine >> 3 : 0) * 4, lane, active, q81, off, scale16);
}

// qkv [3e] (bias added) -> q [e], k -> f16 cache row n_past, v -> f16 cache column n_past.  GPT-NeoX (gptneox lib.rs:205-247): rows per head are q | k | v
// (head stride 3 hd) and q, k get RoPE mode 2 -- the ggml neox branch (LC/ggml.c:11876-11897) rotates EVERY block of n_rot dims of the head, pairs
// (c, c + n_rot/2).  GPT-2 (gpt2 lib.rs:190-210): the three thirds of the row, no rotation (n_rot = 0).  One thread per channel.
__global__ void __launch_bounds__(256) neox_rope_store_kernel(const float *__restrict__ qkv, float *__restrict__ q, __half *__restrict__ Kl, __half *__restrict__ Vl,
                                                              const int *__restrict__ n_past, const float2 *__restrict__ rope_cs, int rope_half, int n_rot, int hd, int e, int n_ctx,
                                                              int head_stride, int k_off, int v_off) {
    pdl_trigger();
    pdl_wait();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= e) return;
    const int p = __ldcg(n_past);
    const int h = i / hd, c = i - h * hd;
    const float *base = qkv + (int64_t)h * head_stride;
    float qo = __ldcg(base + c), ko = __ldcg(base + k_off + c);
    if (n_rot > 0) {
        const int hb = n_rot / 2, ib = c / n_rot, r = c - ib * n_rot;
        if (ib < hd / n_rot) {
            const bool lo = r < hb;
            const int partner = lo ? c + hb : c - hb;
            const float2 cs = __ldg(rope_cs + (int64_t)p * rope_half + ib * hb + (lo ? r : r - hb));
            const float qp = __ldcg(base + partner), kp = __ldcg(base + k_off + partner);
            // x0 = element of the lower half, x1 = upper: out0 = fma(x0, cos, -(x1 sin)), out1 = fma(x0, sin, x1 cos)  (rowops.cu::rope_kernel)
            qo = lo ? __fmaf_rn(qo, cs.x, -__fmul_rn(qp, cs.y)) : __fmaf_rn(qp, cs.y, __fmul_rn(qo, cs.x));
            ko = lo ? __fmaf_rn(ko, cs.x, -__fmul_rn(kp, cs.y)) : __fmaf_rn(kp, cs.y, __fmul_rn(ko, cs.x));
        }
    }
    q[i] = qo;
    Kl[(int64_t)p * e + i] = __float2half_rn(ko);
    Vl[(int64_t)i * n_ctx + p] = __float2half_rn(__ldcg(base + v_off + c));
}

// GPT-2: inpL = wte[token] + wpe[n_past]  (gpt2 lib.rs:164-172), position read from device memory
__global__ void __launch_bounds__(256) gpt2_add_pos_kernel(float *__restrict__ x, const float *__restrict__ wpe, const int *__restrict__ n_past, int e) {
    pdl_wait();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < e) x[i] = __fadd_rn(x[i], __ldg(wpe + (int64_t)__ldcg(n_past) * e + i));
}

template <int TYPE>
void neox_ops_t(const NeoxParams &P, const std::vector<NeoxLayer> &layers, int n_kv_bucket, cudaStream_t st, int *launches) {
    const int q81 = has_min(TYPE) ? 1 : 0, off = TYPE == T_Q5_0 ? 16 : 0, s16 = TYPE == T_Q4_0 ? 1 : 0;
    const int e = P.e;
    int n = 0;
    get_rows_q(P.wte, P.token, P.x, 1, st); n++;
    if (P.wpe) { launch_k(gpt2_add_pos_kernel, dim3((e + 255) / 256), dim3(256), 0, st, P.x, P.wpe, (const int *)P.n_past, e); n++; }
    const int nlay = (n_kv_bucket + 63) / 64 * 64;
    const size_t fa_smem = attn_fused_smem(n_kv_bucket, P.hd);
    // neox.cu decodes a token whose bucket does not fit through the per-op schedule instead
    B200_ASSERT(P.hd % 32 == 0 && P.hd <= 128 && P.n_ctx % 8 == 0 && attn_fused_fits(n_kv_bucket, P.hd) && e <= 8192);
    attn_fused_reserve(fa_smem);
    const dim3 ln_grid((e / 4 + 255) / 256);
    const TpSync S{};
    for (int il = 0; il < P.n_layer; il++) {
        const NeoxLayer &L = layers[il];
        launch_k(ln_pack_kernel, ln_grid, dim3(256), 0, st, (const float *)P.x, L.ln1_g, L.ln1_b, P.xpack_a, e, q81, off, s16); n++;          // :192-196
        MmvArgs A{}; A.xpack = P.xpack_a; A.dst = P.qkv; A.bias = L.bqkv;
        launch_mmv<TYPE, EPI_BIAS>(L.wqkv, A, st); n++;                                                                                      // :199-200
        launch_k(neox_rope_store_kernel, dim3((e + 255) / 256), dim3(256), 0, st, (const float *)P.qkv, P.q, L.K, L.V, (const int *)P.n_past, P.rope_cs, P.rope_half,
                 P.gpt2 ? 0 : P.n_rot, P.hd, e, P.n_ctx, P.gpt2 ? P.hd : 3 * P.hd, P.gpt2 ? e : P.hd, P.gpt2 ? 2 * e : 2 * P.hd); n++;               // :205-247
        {
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(P.n_head * (P.hd / 32)); cfg.blockDim = dim3(ATH); cfg.dynamicSmemBytes = fa_smem; cfg.stream = st;
            cudaLaunchAttribute at[2];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = P.hd / 32; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[1].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at; cfg.numAttrs = (pdl_mask() & 2) ? 2 : 1;
            B200_CHECK(cudaLaunchKernelEx(&cfg, attn_fused_kernel<false>, (const float *)P.q, (const __half *)L.K, (const __half *)L.V, P.xpack_d, (const int *)P.n_past,
                                          (const uint16_t *)P.lut_exp, P.kq_scale, P.hd, P.n_head, P.n_head, e, P.n_ctx, nlay, q81, off, s16,
                                          (unsigned long long *)nullptr, S, 0, attn_prefetch()));                                                           // :250-298
            n++;
        }
        // attention.dense (+bias); sequential residual: ff_in = that + inpL                                                                    :301-312
        MmvArgs Bo{}; Bo.xpack = P.xpack_d; Bo.dst = P.attn_out; Bo.bias = L.bdense; Bo.add1 = P.parallel_residual ? nullptr : P.x;
        launch_mmv<TYPE, EPI_BIAS>(L.wdense, Bo, st); n++;
        // mlp: LayerNorm of inpL (parallel residual) or of ff_in                                                                                :313-316 / ffn
        launch_k(ln_pack_kernel, ln_grid, dim3(256), 0, st, (const float *)(P.parallel_residual ? P.x : P.attn_out), L.ln2_g, L.ln2_b, P.xpack_a, e, q81, off, s16); n++;
        MmvArgs C{}; C.xpack = P.xpack_a; C.xpack_out = P.xpack_f; C.bias = L.bfc; C.lut_gelu = P.lut_gelu; C.q81 = q81; C.off = off; C.scale16 = s16;
        launch_mmv<TYPE, EPI_GELU>(L.wfc, C, st); n++;
        // parallel: inpL = ((proj + bias) + attn) + inpL; sequential: inpL = (proj + bias) + ff_in                                              :317-325
        MmvArgs D{}; D.xpack = P.xpack_f; D.dst = P.x; D.bias = L.bproj; D.add1 = P.attn_out; D.add2 = P.parallel_residual ? P.x : nullptr;
        launch_mmv<TYPE, EPI_BIAS>(L.wproj, D, st); n++;
    }
    launch_k(ln_pack_kernel, ln_grid, dim3(256), 0, st, (const float *)P.x, P.lnf_g, P.lnf_b, P.xpack_a, e, q81, off, s16); n++;                     // :332-334
    MmvArgs Z{}; Z.xpack = P.xpack_a; Z.dst = P.logits; Z.n_past_inc = P.n_past;
    launch_mmv<TYPE, EPI_BIAS>(P.lm_head, Z, st); n++;                                                                                        // :342
    B200_CHECK(cudaGetLastError());
    if (launches) *launches = n;
}

}  // namespace

bool attn_fused_fits(int n_kv_bucket, int hd) { return attn_fused_smem(n_kv_bucket, hd) <= 227 * 1024; }

void neox_decode_enqueue(const NeoxParams &P, const std::vector<NeoxLayer> &layers, int wtype, int n_kv_bucket, cudaStream_t st, int *launches) {
    switch (wtype) {
        case T_Q4_0: neox_ops_t<T_Q4_0>(P, layers, n_kv_bucket, st, launches); break;
        case T_Q4_1: neox_ops_t<T_Q4_1>(P, layers, n_kv_bucket, st, launches); break;
        case T_Q5_0: neox_ops_t<T_Q5_0>(P, layers, n_kv_bucket, st, launches); break;
        case T_Q5_1: neox_ops_t<T_Q5_1>(P, layers, n_kv_bucket, st, launches); break;
        case T_Q8_0: neox_ops_t<T_Q8_0>(P, layers, n_kv_bucket, st, launches); break;
        default: B200_ASSERT(!"neox_decode_enqueue: unsupported weight type");
    }
}

// the process's tensor-parallel context (session.cu calls it after the slabs are connected and when the measurement switch flips); not inside a stream capture
void decode_set_tp(const TpCtx &T, cudaStream_t st) {
    B200_CHECK(cudaStreamSynchronize(st));
    B200_CHECK(cudaMemcpyToSymbol(c_tp, &T, sizeof(TpCtx)));
    B200_CHECK(cudaDeviceSynchronize());
}

// Enqueue one decode step (position read from *P.n_past on the device) on `st`.  n_kv_bucket >= n_past + 1 sizes the KQ grid.
void decode_ops_enqueue(const DecodeParams &P, const std::vector<DecodeLayer> &layers, int wtype, int n_kv_bucket, int4 *xpack_a, cudaStream_t st, int *launches) {
    const bool tp = P.tp.world > 1;
    switch (wtype) {
        case T_Q4_0: if (tp) decode_ops_t<T_Q4_0, true>(P, layers, n_kv_bucket, xpack_a, st, launches); else decode_ops_t<T_Q4_0, false>(P, layers, n_kv_bucket, xpack_a, st, launches); break;
        case T_Q4_1: if (tp) decode_ops_t<T_Q4_1, true>(P, layers, n_kv_bucket, xpack_a, st, launches); else decode_ops_t<T_Q4_1, false>(P, layers, n_kv_bucket, xpack_a, st, launches); break;
        case T_Q5_0: if (tp) decode_ops_t<T_Q5_0, true>(P, layers, n_kv_bucket, xpack_a, st, launches); else decode_ops_t<T_Q5_0, false>(P, layers, n_kv_bucket, xpack_a, st, launches); break;
        case T_Q5_1: if (tp) decode_ops_t<T_Q5_1, true>(P, layers, n_kv_bucket, xpack_a, st, launches); else decode_ops_t<T_Q5_1, false>(P, layers, n_kv_bucket, xpack_a, st, launches); break;
        case T_Q8_0: if (tp) decode_ops_t<T_Q8_0, true>(P, layers, n_kv_bucket, xpack_a, st, launches); else decode_ops_t<T_Q8_0, false>(P, layers, n_kv_bucket, xpack_a, st, launches); break;
        default: B200_ASSERT(!"decode_ops_enqueue: unsupported weight type");
    }
}

}  // namespace b200
