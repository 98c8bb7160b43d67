// encoder.cu -- encoder forwards of the three BERT-base towers (HF BertModel semantics restated in SURVEY.md Appendix B):
//   query side: two independent towers on the same tokens, hidden state at position 0 of each (Encoder.forward(return_query=True)
//     -> embed_query, /root/reference/densephrases/encoder.py:146-152, 101-118).  Both towers run as one grouped problem: every
//     GEMM is one launch of the tcgen05 kernels (gemm_tf32.cu / gemm_bf16x3.cu) with blockIdx.z = tower.
//   phrase side: the phrase tower over every token, its last LayerNorm fused with the filter head and the int8 dump quantisation
//     (Encoder.forward(input_ids=..., return_phrase=True) -> embed_phrase + filter_linear, encoder.py:92-99, 130-144).
// Both run through one tower body (run_towers) parameterised by the tower set and by what the last layer keeps.
#include "common.cuh"
#include "../../include/dph_b200.h"
#include <cuda_bf16.h>

#define ENC_H 768
#define ENC_HEADS 12
#define ENC_DH 64
#define ENC_LAYERS 12
#define ENC_FF 3072
#define ENC_MAX_S 384          // Makefile:357-375 uses max_query_length 384 for KILT; attention keeps K,V of one head in smem

int dph_launch_gemm_tf32(int group, const float* const* A, const float* const* W, const float* const* bias, const float* const* residual,
                         float* const* out, int M, int N, int K, int act, cudaStream_t st, const float* const* A_lo, const float* const* W_lo);
int dph_launch_split_tf32(const float* x, float* hi, float* lo, long long n, cudaStream_t st);
int dph_launch_split_bf16(const float* x, void* hi, void* lo, long long n, cudaStream_t st);                                                  // gemm_bf16x3.cu
int dph_launch_gemm_bf16x3(int group, const void* const* A_hi, const void* const* A_lo, const void* const* W_hi, const void* const* W_lo,
                           const float* const* bias, const float* const* residual, float* const* out, void* const* out_hi, void* const* out_lo,
                           int M, int N, int K, int act, cudaStream_t st);
int dph_launch_attention_tc(const float* const qkv[2], float* const ctx[2], const long long* mask, int B, int S, long long T, cudaStream_t st, int split,
                            unsigned short* const* ctx_hi, unsigned short* const* ctx_lo, int ntw);   // attention_tc.cu
int dph_launch_attention_long(const float* qkv, float* ctx, const long long* mask, int B, int S, cudaStream_t st, int split,
                              unsigned short* ctx_hi, unsigned short* ctx_lo);                        // attention_long.cu
#define ENC_MAX_S_LONG 512     // the tensor-core long-sequence attention (attention_long.cu); max_seq_length of the phrase dump
#define ENC_TOWERS 3           // 0 query_start_encoder, 1 query_end_encoder, 2 phrase_encoder

struct LayerW { const float *Wqkv, *bqkv, *Wo, *bo, *ln1g, *ln1b, *Wi, *bi, *Wo2, *bo2, *ln2g, *ln2b; };
struct TowerW { const float *word, *pos, *type, *embg, *embb; LayerW L[ENC_LAYERS]; };

struct dph_encoder {
    int device = 0; int vocab = 0, max_pos = 512, type_vocab = 2;
    cudaStream_t stream = 0;
    float* blob[ENC_TOWERS] = {};
    TowerW tw[ENC_TOWERS];
    float* filt = nullptr;                       // filter_linear: W [2, 768] (row 0 start, row 1 end) | b [2]
    // 3xTF32 mode: (hi, lo) copies of the four GEMM weight matrices of every layer, made lazily on the first precise forward
    int precise = 0;                             // 0: 1xTF32, 1: 3xTF32 split (fp32 planes), 2: bf16x3 split (bf16 planes, gemm_bf16x3.cu)
    unsigned short* wbf[ENC_TOWERS] = {};        // bf16x3 mode: per tower, per layer [Wqkv_hi, Wqkv_lo, Wo_hi, Wo_lo, Wi_hi, Wi_lo, Wo2_hi, Wo2_lo]
    int attention_tc = 1;                        // S <= 64 and not precise: attention on the tensor cores (attention_tc.cu); 0: SIMT fp32 kernels below
    float* wsplit[ENC_TOWERS] = {};              // per tower: for each layer [Wqkv_hi, Wqkv_lo, Wo_hi, Wo_lo, Wi_hi, Wi_lo, Wo2_hi, Wo2_lo]
    float *act_hi[2] = {}, *act_lo[2] = {};      // split copy of the current GEMM input activation (up to T x 3072)
    // workspace: one slot per tower of a forward (query: slots 0, 1; phrase: slot 0 only), each for cap_slot[s] tokens
    int64_t cap_tokens = 0, cap_slot[2] = {0, 0};
    float *x[2] = {}, *qkv[2] = {}, *ctx[2] = {}, *a[2] = {}, *ffn[2] = {};
    long long *ids = nullptr, *mask = nullptr, *tt = nullptr;
    float *out_s = nullptr, *out_e = nullptr;
    int64_t cap_b = 0;
    int* bad_ids = nullptr;                      // device flag: an input id / token type was outside the embedding tables
    bool bad_pending = false;                    // an asynchronous (device-buffer) forward has not had its flag checked yet
};

static int64_t tower_floats(const dph_encoder* e) {
    int64_t n = (int64_t)e->vocab * ENC_H + (int64_t)e->max_pos * ENC_H + (int64_t)e->type_vocab * ENC_H + 2 * ENC_H;
    int64_t per_layer = (int64_t)3 * ENC_H * ENC_H + 3 * ENC_H + (int64_t)ENC_H * ENC_H + ENC_H + 2 * ENC_H + (int64_t)ENC_FF * ENC_H + ENC_FF +
                        (int64_t)ENC_H * ENC_FF + ENC_H + 2 * ENC_H;
    return n + ENC_LAYERS * per_layer;
}
static void carve(dph_encoder* e, int t) {
    const float* p = e->blob[t];
    TowerW& w = e->tw[t];
    auto take = [&](int64_t n) { const float* r = p; p += n; return r; };
    w.word = take((int64_t)e->vocab * ENC_H); w.pos = take((int64_t)e->max_pos * ENC_H); w.type = take((int64_t)e->type_vocab * ENC_H);
    w.embg = take(ENC_H); w.embb = take(ENC_H);
    for (int l = 0; l < ENC_LAYERS; l++) {
        LayerW& L = w.L[l];
        L.Wqkv = take((int64_t)3 * ENC_H * ENC_H); L.bqkv = take(3 * ENC_H); L.Wo = take((int64_t)ENC_H * ENC_H); L.bo = take(ENC_H);
        L.ln1g = take(ENC_H); L.ln1b = take(ENC_H); L.Wi = take((int64_t)ENC_FF * ENC_H); L.bi = take(ENC_FF);
        L.Wo2 = take((int64_t)ENC_H * ENC_FF); L.bo2 = take(ENC_H); L.ln2g = take(ENC_H); L.ln2b = take(ENC_H);
    }
}

// ---- LayerNorm helpers: one 256-thread block per token row, 3 elements per thread, eps inside the sqrt (torch.nn.LayerNorm) ----
__device__ __forceinline__ float block_sum_256(float v, float* red) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) t += red[i];
    return t;
}
__device__ __forceinline__ void ln_row_256(float v[3], const float* g, const float* b, float* out, float* red) {
    const float mean = block_sum_256(v[0] + v[1] + v[2], red) * (1.0f / ENC_H);
    const float d0 = v[0] - mean, d1 = v[1] - mean, d2 = v[2] - mean;
    const float var = block_sum_256(d0 * d0 + d1 * d1 + d2 * d2, red) * (1.0f / ENC_H);
    const float rstd = rsqrtf(var + 1e-12f);
    const int t = threadIdx.x;
    out[t] = d0 * rstd * g[t] + b[t];
    out[t + 256] = d1 * rstd * g[t + 256] + b[t + 256];
    out[t + 512] = d2 * rstd * g[t + 512] + b[t + 512];
}

// (hi, lo) bf16 planes with x ~= hi + lo (gemm_bf16x3.cu); hardware converts, round to nearest even
__device__ __forceinline__ void enc_split(float x, unsigned short& hi, unsigned short& lo) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    hi = __bfloat16_as_ushort(h);
    lo = __bfloat16_as_ushort(__float2bfloat16_rn(x - __bfloat162float(h)));
}
__device__ __forceinline__ void enc_split2(float x0, float x1, unsigned& hi, unsigned& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const unsigned*>(&h);
    lo = *reinterpret_cast<const unsigned*>(&l);
}

struct EmbedArgs { const long long* ids; const long long* tt; int S; const float* word[2]; const float* pos[2]; const float* type[2];
                   const float* g[2]; const float* b[2]; float* out[2]; long long vocab, type_vocab; int* bad;
                   unsigned short* out_hi[2]; unsigned short* out_lo[2]; };      // nullable: bf16 planes of the output for the first bf16x3 GEMM
__global__ void __launch_bounds__(256) embed_ln_kernel(EmbedArgs a) {
    __shared__ float red[8];
    const long long tok = blockIdx.x; const int tw = blockIdx.y, t = threadIdx.x;
    long long id = a.ids[tok], ty = a.tt[tok]; const int s = (int)(tok % a.S);
    // torch.nn.Embedding raises IndexError on an out-of-range id; here the row is clamped (no out-of-bounds read) and a sticky
    // device flag makes the host call fail (host buffers: this call; device buffers: the next call that synchronises)
    if (id < 0 || id >= a.vocab || ty < 0 || ty >= a.type_vocab) {
        if (t == 0) atomicExch(a.bad, 1);
        id = id < 0 ? 0 : (id >= a.vocab ? a.vocab - 1 : id);
        ty = ty < 0 ? 0 : (ty >= a.type_vocab ? a.type_vocab - 1 : ty);
    }
    const float* w = a.word[tw] + id * ENC_H; const float* p = a.pos[tw] + (long long)s * ENC_H; const float* y = a.type[tw] + ty * ENC_H;
    float v[3];
#pragma unroll
    for (int i = 0; i < 3; i++) v[i] = (w[t + 256 * i] + y[t + 256 * i]) + p[t + 256 * i];   // inputs_embeds + token_type, + position (HF order)
    ln_row_256(v, a.g[tw], a.b[tw], a.out[tw] + tok * ENC_H, red);
    if (a.out_hi[tw]) {
        const float* o = a.out[tw] + tok * ENC_H;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            unsigned short h, l;
            enc_split(o[t + 256 * i], h, l);          // this thread's own three outputs (written just above)
            a.out_hi[tw][tok * ENC_H + t + 256 * i] = h;
            a.out_lo[tw][tok * ENC_H + t + 256 * i] = l;
        }
    }
}
struct LnArgs { const float* in[2]; const float* g[2]; const float* b[2]; float* out[2]; long long rows; long long in_stride, out_stride;
                unsigned short* out_hi[2]; unsigned short* out_lo[2]; };          // nullable: dense [rows, 768] bf16 planes of the output
// One warp per row, 24 elements per lane as six float4: no shared memory, no block barrier; two-pass mean / variance like
// torch.nn.LayerNorm.  in/out row strides allow normalising only the [CLS] rows of the last layer.
__global__ void __launch_bounds__(256) layernorm_kernel(LnArgs a) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int tw = blockIdx.y, lane = threadIdx.x & 31;
    if (row >= a.rows) return;
    const float4* x = reinterpret_cast<const float4*>(a.in[tw] + row * a.in_stride);
    float4 v[6];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 6; i++) { v[i] = x[lane + 32 * i]; s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float mean = s * (1.0f / ENC_H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
    const float rstd = rsqrtf(q * (1.0f / ENC_H) + 1e-12f);
    const float4* g = reinterpret_cast<const float4*>(a.g[tw]);
    const float4* b = reinterpret_cast<const float4*>(a.b[tw]);
    float4* o = reinterpret_cast<float4*>(a.out[tw] + row * a.out_stride);
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const float4 gg = g[lane + 32 * i], bb = b[lane + 32 * i];
        const float4 r4 = make_float4(v[i].x * rstd * gg.x + bb.x, v[i].y * rstd * gg.y + bb.y, v[i].z * rstd * gg.z + bb.z, v[i].w * rstd * gg.w + bb.w);
        o[lane + 32 * i] = r4;
        if (a.out_hi[tw]) {
            uint2 h4, l4;
            enc_split2(r4.x, r4.y, h4.x, l4.x); enc_split2(r4.z, r4.w, h4.y, l4.y);
            reinterpret_cast<uint2*>(a.out_hi[tw] + row * ENC_H)[lane + 32 * i] = h4;
            reinterpret_cast<uint2*>(a.out_lo[tw] + row * ENC_H)[lane + 32 * i] = l4;
        }
    }
}
// gather rows b*S of [B*S, 768] into a dense [B, 768] buffer (the [CLS] rows the last layer's output actually needs)
__global__ void gather_cls_kernel(const float* in0, const float* in1, float* out0, float* out1, int S, long long B) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * (ENC_H / 4)) return;
    const long long b = i / (ENC_H / 4); const int c = (int)(i % (ENC_H / 4));
    const float* in = blockIdx.y ? in1 : in0; float* out = blockIdx.y ? out1 : out0;
    reinterpret_cast<float4*>(out)[b * (ENC_H / 4) + c] = reinterpret_cast<const float4*>(in)[b * S * (ENC_H / 4) + c];
}

// ---- self attention: one CTA per (head, batch row, tower); K (padded rows) and V of the head in shared memory; a warp per
// query row: lanes = keys for QK^T and softmax, lanes = output dims for P V.  scores/8 + (1-mask)*-10000, softmax in fp32.
struct AttnArgs { const float* qkv[2]; float* ctx[2]; const long long* mask; int S; };
__global__ void __launch_bounds__(256) attention_kernel(AttnArgs a) {
    extern __shared__ float asm_[];
    const int S = a.S, h = blockIdx.x, b = blockIdx.y, tw = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    float* Ks = asm_;                       // [S][65]
    float* Vs = Ks + (size_t)S * 65;        // [S][64]
    float* mb = Vs + (size_t)S * 64;        // [S] additive mask
    float* qs = mb + S;                     // [nw][64]
    float* ps = qs + nw * 64;               // [nw][S]
    const float* base = a.qkv[tw] + (long long)b * S * (3 * ENC_H) + h * ENC_DH;
    for (int i = threadIdx.x; i < S * 64; i += blockDim.x) {
        const int j = i >> 6, d = i & 63;
        Ks[j * 65 + d] = base[(long long)j * (3 * ENC_H) + ENC_H + d];
        Vs[j * 64 + d] = base[(long long)j * (3 * ENC_H) + 2 * ENC_H + d];
    }
    for (int j = threadIdx.x; j < S; j += blockDim.x) mb[j] = (1.0f - (float)a.mask[(long long)b * S + j]) * -10000.0f;
    __syncthreads();
    const int nj = (S + 31) >> 5;
    for (int i = warp; i < S; i += nw) {
        float* q = qs + warp * 64;
        q[lane] = base[(long long)i * (3 * ENC_H) + lane];
        q[lane + 32] = base[(long long)i * (3 * ENC_H) + lane + 32];
        __syncwarp();
        float sc[ENC_MAX_S / 32];
        float mx = -3.0e38f;
#pragma unroll
        for (int jj = 0; jj < ENC_MAX_S / 32; jj++) {
            if (jj < nj) {
                const int j = jj * 32 + lane;
                float dot = 0.f;
                if (j < S) {
                    const float* kr = Ks + j * 65;
#pragma unroll 16
                    for (int d = 0; d < 64; d++) dot = fmaf(q[d], kr[d], dot);
                    dot = dot * 0.125f + mb[j];
                } else dot = -3.0e38f;
                sc[jj] = dot;
                mx = fmaxf(mx, dot);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        float sum = 0.f;
#pragma unroll
        for (int jj = 0; jj < ENC_MAX_S / 32; jj++) {
            if (jj < nj) {
                const int j = jj * 32 + lane;
                const float e = (j < S) ? expf(sc[jj] - mx) : 0.f;
                sc[jj] = e;
                sum += e;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
        const float inv = 1.0f / sum;
        float* p = ps + (size_t)warp * S;
#pragma unroll
        for (int jj = 0; jj < ENC_MAX_S / 32; jj++)
            if (jj < nj) { const int j = jj * 32 + lane; if (j < S) p[j] = sc[jj] * inv; }
        __syncwarp();
        float o0 = 0.f, o1 = 0.f;
        for (int j = 0; j < S; j++) {
            const float pj = p[j];
            o0 = fmaf(pj, Vs[j * 64 + lane], o0);
            o1 = fmaf(pj, Vs[j * 64 + lane + 32], o1);
        }
        float* out = a.ctx[tw] + ((long long)b * S + i) * ENC_H + h * ENC_DH;
        out[lane] = o0;
        out[lane + 32] = o1;
        __syncwarp();
    }
}

// ---- register-tiled attention for S <= 128 (the query path: max_query_length 24/32/64, options.py:38, Makefile:441) ----------------
// One CTA per (head x 64-row tile, batch row, tower), 256 threads as 16 x 16: thread (ty,tx) owns rows 4ty..4ty+3 and keys
// tx + 16 c (c < KT) of the score tile, then rows 4ty.. and dims 4tx..4tx+3 of the context tile.  Q and K are staged transposed
// ([d][row]) so every inner step is two LDS.128 for 16 (scores) / 16 (context) FMAs; the softmax row reduction is a 16-lane
// shuffle.  Same arithmetic as the reference: scores/8 + (1-mask)*-10000, fp32 softmax, P V.
template <int KT>
__global__ void __launch_bounds__(256) attention_tile_kernel(AttnArgs a) {
    extern __shared__ __align__(16) float asm2_[];
    constexpr int SP = 16 * KT;                       // padded key count
    const int S = a.S, h = blockIdx.x % ENC_HEADS, rt = blockIdx.x / ENC_HEADS, b = blockIdx.y, tw = blockIdx.z;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    float* Qt = asm2_;                                // [64 d][68]      rows of this tile
    float* Kt = Qt + 64 * 68;                         // [64 d][SP + 4]
    float* Vs = Kt + 64 * (SP + 4);                   // [SP][64]
    float* Pt = Vs + SP * 64;                         // [SP keys][68]   probabilities, transposed
    float* mb = Pt + SP * 68;                         // [SP]
    const float* base = a.qkv[tw] + (long long)b * S * (3 * ENC_H) + h * ENC_DH;
    const int row0 = rt * 64;
    for (int i = tid; i < 64 * 64; i += 256) {        // Q tile, transposed
        const int r = i >> 6, d = i & 63;
        Qt[d * 68 + r] = (row0 + r < S) ? base[(long long)(row0 + r) * (3 * ENC_H) + d] : 0.f;
    }
    for (int i = tid; i < SP * 64; i += 256) {        // K transposed, V as is
        const int j = i >> 6, d = i & 63;
        const bool ok = j < S;
        Kt[d * (SP + 4) + j] = ok ? base[(long long)j * (3 * ENC_H) + ENC_H + d] : 0.f;
        Vs[j * 64 + d] = ok ? base[(long long)j * (3 * ENC_H) + 2 * ENC_H + d] : 0.f;
    }
    for (int j = tid; j < SP; j += 256) mb[j] = (j < S) ? (1.0f - (float)a.mask[(long long)b * S + j]) * -10000.0f : -3.0e38f;
    __syncthreads();
    float acc[4][KT];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int c = 0; c < KT; c++) acc[i][c] = 0.f;
#pragma unroll 8
    for (int d = 0; d < 64; d++) {
        const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * 68 + ty * 4);
        const float q[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
        for (int c = 0; c < KT; c++) {
            const float kv = Kt[d * (SP + 4) + tx + 16 * c];
#pragma unroll
            for (int i = 0; i < 4; i++) acc[i][c] = fmaf(q[i], kv, acc[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float mx = -3.0e38f;
#pragma unroll
        for (int c = 0; c < KT; c++) { acc[i][c] = acc[i][c] * 0.125f + mb[tx + 16 * c]; mx = fmaxf(mx, acc[i][c]); }
#pragma unroll
        for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        float sum = 0.f;
#pragma unroll
        for (int c = 0; c < KT; c++) { const float e = (tx + 16 * c < S) ? expf(acc[i][c] - mx) : 0.f; acc[i][c] = e; sum += e; }
#pragma unroll
        for (int off = 8; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
        const float inv = 1.0f / sum;
#pragma unroll
        for (int c = 0; c < KT; c++) Pt[(tx + 16 * c) * 68 + ty * 4 + i] = acc[i][c] * inv;
    }
    __syncthreads();
    float o[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int e = 0; e < 4; e++) o[i][e] = 0.f;
    for (int j = 0; j < S; j++) {
        const float4 p4 = *reinterpret_cast<const float4*>(Pt + j * 68 + ty * 4);
        const float4 v4 = *reinterpret_cast<const float4*>(Vs + j * 64 + tx * 4);
        const float p[4] = {p4.x, p4.y, p4.z, p4.w}, v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int e = 0; e < 4; e++) o[i][e] = fmaf(p[i], v[e], o[i][e]);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = row0 + ty * 4 + i;
        if (r < S) *reinterpret_cast<float4*>(a.ctx[tw] + ((long long)b * S + r) * ENC_H + h * ENC_DH + tx * 4) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
    }
}
template <int KT> static int launch_attention_tile(const AttnArgs& aa, int B, int ng, cudaStream_t st) {
    constexpr int SP = 16 * KT;
    const size_t smem = (size_t)(64 * 68 + 64 * (SP + 4) + SP * 64 + SP * 68 + SP) * 4;
    static DphPerDeviceOnce once;
    if (once.first()) { DPH_CUDA(cudaFuncSetAttribute(attention_tile_kernel<KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }
    attention_tile_kernel<KT><<<dim3(ENC_HEADS * ((aa.S + 63) / 64), (unsigned)B, (unsigned)ng), 256, smem, st>>>(aa);
    DPH_CUDA(cudaGetLastError());
    return 0;
}
// ng: towers of the grouped problem (blockIdx.z), 1 or 2
static int launch_attention(const AttnArgs& aa, int B, int ng, cudaStream_t st) {
    const int S = aa.S;
    if (S <= 16) return launch_attention_tile<1>(aa, B, ng, st);
    if (S <= 32) return launch_attention_tile<2>(aa, B, ng, st);
    if (S <= 64) return launch_attention_tile<4>(aa, B, ng, st);
    if (S <= 96) return launch_attention_tile<6>(aa, B, ng, st);
    if (S <= 128) return launch_attention_tile<8>(aa, B, ng, st);
    const int attn_warps = 8;      // long sequences (max_query_length 384 for KILT entity linking): K,V of the head in shared memory
    const size_t attn_smem = ((size_t)S * 65 + (size_t)S * 64 + S + attn_warps * 64 + (size_t)attn_warps * S) * 4;
    static DphPerDeviceOnce once;
    if (once.first()) { DPH_CUDA(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); }
    attention_kernel<<<dim3(ENC_HEADS, (unsigned)B, (unsigned)ng), attn_warps * 32, attn_smem, st>>>(aa);
    DPH_CUDA(cudaGetLastError());
    return 0;
}

// ---- C ABI ---------------------------------------------------------------------------------------------
DPH_API int dph_encoder_create(dph_encoder** out, int device, int vocab_size, int max_pos, int type_vocab) {
    DPH_CHECK(out && vocab_size > 0 && max_pos > 0 && type_vocab > 0, "bad encoder geometry");
    DPH_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    DPH_CUDA(cudaGetDeviceProperties(&prop, device));
    DPH_CHECK(prop.major == 10, "libdph_b200 is built for sm_100a (B200) only");
    dph_encoder* e = new dph_encoder();
    e->device = device; e->vocab = vocab_size; e->max_pos = max_pos; e->type_vocab = type_vocab;
    *out = e;
    return 0;
}
DPH_API void dph_encoder_free(dph_encoder* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    for (int t = 0; t < ENC_TOWERS; t++) {
        float* w[] = {e->blob[t], e->wsplit[t], (float*)e->wbf[t]};
        for (float* p : w) if (p) cudaFree(p);
    }
    for (int t = 0; t < 2; t++) {
        float* ws[] = {e->x[t], e->qkv[t], e->ctx[t], e->a[t], e->ffn[t], e->act_hi[t], e->act_lo[t]};
        for (float* p : ws) if (p) cudaFree(p);
    }
    void* misc[] = {e->ids, e->mask, e->tt, e->out_s, e->out_e, e->bad_ids, e->filt};
    for (void* p : misc) if (p) cudaFree(p);
    delete e;
}
DPH_API int dph_encoder_set_stream(dph_encoder* e, void* s) { e->stream = (cudaStream_t)s; return 0; }
DPH_API int dph_encoder_set_precision(dph_encoder* e, int precise) {
    DPH_CHECK(precise >= 0 && precise <= 2, "precision mode: 0 (1xTF32), 1 (3xTF32) or 2 (bf16x3)");
    e->precise = precise;
    return 0;
}
DPH_API int dph_encoder_set_attention(dph_encoder* e, int tensor_core) { e->attention_tc = tensor_core ? 1 : 0; return 0; }
// (the encoder's attention setting: S <= 64 -> attention_tc.cu, 64 < S <= 512 in the phrase forward -> attention_long.cu)

// C ABI (test / standalone use): one BERT self-attention over a [B*S, 2304] QKV activation (device pointers) -> ctx [B*S, 768].
// tensor_core 1 / 2: S <= 64 -> attention_tc.cu, 64 < S <= 512 -> attention_long.cu; 0: the SIMT kernels, S <= 384.
DPH_API int dph_attention_bert(const float* qkv, const int64_t* mask, int B, int S, float* ctx, int tensor_core, void* cuda_stream) {
    DPH_CHECK(tensor_core >= 0 && tensor_core <= 2, "tensor_core: 0 SIMT fp32, 1 tcgen05 TF32, 2 tcgen05 bf16x3 planes (fp32-accurate)");
    DPH_CHECK(qkv && mask && ctx && B >= 1 && S >= 1 && S <= (tensor_core ? ENC_MAX_S_LONG : ENC_MAX_S), "attention: bad arguments");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc;
    if (tensor_core && S > 64) {
        rc = dph_launch_attention_long(qkv, ctx, (const long long*)mask, B, S, st, tensor_core == 2, nullptr, nullptr);
    } else if (tensor_core) {
        const float* q2[2] = {qkv, qkv}; float* c2[2] = {ctx, ctx};
        rc = dph_launch_attention_tc(q2, c2, (const long long*)mask, B, S, (long long)B * S, st, tensor_core == 2, nullptr, nullptr, 1);
    } else {
        AttnArgs aa; aa.qkv[0] = qkv; aa.qkv[1] = qkv; aa.ctx[0] = ctx; aa.ctx[1] = ctx; aa.mask = (const long long*)mask; aa.S = S;
        rc = launch_attention(aa, B, 1, st);
    }
    cudaStreamSynchronize(st);
    return rc;
}

static const int64_t kGemmW[4] = {(int64_t)3 * ENC_H * ENC_H, (int64_t)ENC_H * ENC_H, (int64_t)ENC_FF * ENC_H, (int64_t)ENC_H * ENC_FF};
static int64_t split_layer_floats() { return 2 * (kGemmW[0] + kGemmW[1] + kGemmW[2] + kGemmW[3]); }
static int ensure_split_weights(dph_encoder* e, const int* towers, int ng) {
    for (int g = 0; g < ng; g++) {
        const int t = towers[g];
        if (e->wsplit[t]) continue;
        DPH_CUDA(cudaMalloc((void**)&e->wsplit[t], (size_t)split_layer_floats() * ENC_LAYERS * 4));
        for (int l = 0; l < ENC_LAYERS; l++) {
            const LayerW& L = e->tw[t].L[l];
            const float* src[4] = {L.Wqkv, L.Wo, L.Wi, L.Wo2};
            float* p = e->wsplit[t] + (size_t)l * split_layer_floats();
            for (int m = 0; m < 4; m++) { DPH_TRY(dph_launch_split_tf32(src[m], p, p + kGemmW[m], kGemmW[m], e->stream)); p += 2 * kGemmW[m]; }
        }
    }
    return 0;
}
static int ensure_bf16_weights(dph_encoder* e, const int* towers, int ng) {
    for (int g = 0; g < ng; g++) {
        const int t = towers[g];
        if (e->wbf[t]) continue;
        DPH_CUDA(cudaMalloc((void**)&e->wbf[t], (size_t)split_layer_floats() * ENC_LAYERS * 2));
        for (int l = 0; l < ENC_LAYERS; l++) {
            const LayerW& L = e->tw[t].L[l];
            const float* src[4] = {L.Wqkv, L.Wo, L.Wi, L.Wo2};
            unsigned short* p = e->wbf[t] + (size_t)l * split_layer_floats();
            for (int m = 0; m < 4; m++) { DPH_TRY(dph_launch_split_bf16(src[m], p, p + kGemmW[m], kGemmW[m], e->stream)); p += 2 * kGemmW[m]; }
        }
    }
    return 0;
}
static void bf16_ptrs(const dph_encoder* e, int t, int l, int m, const void** hi, const void** lo) {
    const unsigned short* p = e->wbf[t] + (size_t)l * split_layer_floats();
    for (int i = 0; i < m; i++) p += 2 * kGemmW[i];
    *hi = p; *lo = p + kGemmW[m];
}
static void split_ptrs(const dph_encoder* e, int t, int l, int m, const float** hi, const float** lo) {
    const float* p = e->wsplit[t] + (size_t)l * split_layer_floats();
    for (int i = 0; i < m; i++) p += 2 * kGemmW[i];
    *hi = p; *lo = p + kGemmW[m];
}
DPH_API int64_t dph_encoder_tower_floats(const dph_encoder* e) { return tower_floats(e); }
// blob layout (fp32, all nn.Linear weights as stored by torch: [out_features, in_features]):
//   word_embeddings [V,768] | position_embeddings [P,768] | token_type_embeddings [T,768] | embeddings.LayerNorm weight, bias |
//   per layer: [Wq;Wk;Wv] [2304,768] | [bq;bk;bv] | attention.output.dense W [768,768], b | attention.output.LayerNorm w, b |
//              intermediate.dense W [3072,768], b | output.dense W [768,3072], b | output.LayerNorm w, b
DPH_API int dph_encoder_load_tower(dph_encoder* e, int tower, const float* blob, int mem) {
    DPH_CHECK(tower >= 0 && tower < ENC_TOWERS, "tower must be 0 (query_start_encoder), 1 (query_end_encoder) or 2 (phrase_encoder)");
    DPH_CUDA(cudaSetDevice(e->device));
    const size_t bytes = (size_t)tower_floats(e) * 4;
    if (!e->blob[tower]) DPH_CUDA(cudaMalloc((void**)&e->blob[tower], bytes));
    DPH_CUDA(cudaMemcpy(e->blob[tower], blob, bytes, mem == DPH_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
    carve(e, tower);
    if (e->wsplit[tower]) { cudaFree(e->wsplit[tower]); e->wsplit[tower] = nullptr; }
    if (e->wbf[tower]) { cudaFree(e->wbf[tower]); e->wbf[tower] = nullptr; }
    return 0;
}
// filter_linear (encoder.py:32, 137-141): W [2, 768] as stored by torch (row 0: start logit, row 1: end logit), b [2]
DPH_API int dph_encoder_load_filter(dph_encoder* e, const float* W, const float* b, int mem) {
    DPH_CHECK(e && W && b, "filter: bad arguments");
    DPH_CUDA(cudaSetDevice(e->device));
    if (!e->filt) DPH_CUDA(cudaMalloc((void**)&e->filt, (2 * ENC_H + 2) * 4));
    const cudaMemcpyKind k = mem == DPH_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    DPH_CUDA(cudaMemcpy(e->filt, W, 2 * ENC_H * 4, k));
    DPH_CUDA(cudaMemcpy(e->filt + 2 * ENC_H, b, 2 * 4, k));
    return 0;
}
// free + null + allocate, so that a failed allocation never leaves a dangling pointer behind for dph_encoder_free
static int regrow(void** p, size_t bytes) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    DPH_CUDA(cudaMalloc(p, bytes));
    return 0;
}
// workspace of `nslots` towers for T tokens: 13824 floats (55.3 KB) per token and slot, + 24 bytes of ids / mask / token types
static int ensure_ws(dph_encoder* e, int64_t T, int64_t B, int nslots) {
    for (int t = 0; t < nslots; t++) {
        if (T <= e->cap_slot[t]) continue;
        e->cap_slot[t] = 0;                                  // stays 0 if anything below fails: the next call starts over
        float** ps[] = {&e->x[t], &e->qkv[t], &e->ctx[t], &e->a[t], &e->ffn[t], &e->act_hi[t], &e->act_lo[t]};
        size_t sz[] = {(size_t)T * ENC_H, (size_t)T * 3 * ENC_H, (size_t)T * ENC_H, (size_t)T * ENC_H, (size_t)T * ENC_FF, (size_t)T * ENC_FF,
                       (size_t)T * ENC_FF};
        for (int i = 0; i < 7; i++) DPH_TRY(regrow((void**)ps[i], sz[i] * 4));
        e->cap_slot[t] = T;
    }
    if (T > e->cap_tokens) {
        e->cap_tokens = 0;
        long long** ip[] = {&e->ids, &e->mask, &e->tt};
        for (auto p : ip) DPH_TRY(regrow((void**)p, (size_t)T * 8));
        e->cap_tokens = T;
    }
    if (B > e->cap_b) {
        e->cap_b = 0;
        DPH_TRY(regrow((void**)&e->out_s, (size_t)B * ENC_H * 4));
        DPH_TRY(regrow((void**)&e->out_e, (size_t)B * ENC_H * 4));
        e->cap_b = B;
    }
    return 0;
}

// Start of a forward: workspace, the deferred bad-id flag of an earlier asynchronous call, inputs on the device.
static int begin_forward(dph_encoder* e, const int64_t* ids, const int64_t* mask, const int64_t* tt, int B, int S, int nslots, int mem,
                         const long long** d_ids, const long long** d_mask, const long long** d_tt) {
    DPH_CUDA(cudaSetDevice(e->device));
    cudaStream_t st = e->stream;
    const int64_t T = (int64_t)B * S;
    DPH_TRY(ensure_ws(e, T, B, nslots));
    if (!e->bad_ids) { DPH_CUDA(cudaMalloc((void**)&e->bad_ids, 4)); DPH_CUDA(cudaMemset(e->bad_ids, 0, 4)); }
    if (e->bad_pending) {       // flag of the previous asynchronous forward(s): report it now instead of never
        int h = 0;
        DPH_CUDA(cudaMemcpyAsync(&h, e->bad_ids, 4, cudaMemcpyDeviceToHost, st));
        DPH_CUDA(cudaStreamSynchronize(st));
        e->bad_pending = false;
        if (h) { DPH_CUDA(cudaMemsetAsync(e->bad_ids, 0, 4, st)); dph_set_error("encoder: an earlier forward received input_ids / token_type_ids outside the embedding tables"); return 1; }
    }
    *d_ids = (const long long*)ids; *d_mask = (const long long*)mask; *d_tt = (const long long*)tt;
    if (mem == DPH_MEM_HOST) {
        DPH_CUDA(cudaMemcpyAsync(e->ids, ids, T * 8, cudaMemcpyHostToDevice, st));
        DPH_CUDA(cudaMemcpyAsync(e->mask, mask, T * 8, cudaMemcpyHostToDevice, st));
        DPH_CUDA(cudaMemcpyAsync(e->tt, tt, T * 8, cudaMemcpyHostToDevice, st));
        *d_ids = e->ids; *d_mask = e->mask; *d_tt = e->tt;
    }
    return 0;
}
// End of a forward: host buffers -> wait and report the bad-id flag now (IndexError in torch); device buffers -> at the next call.
static int end_forward(dph_encoder* e, int mem) {
    cudaStream_t st = e->stream;
    if (mem == DPH_MEM_HOST) {
        int h = 0;
        DPH_CUDA(cudaMemcpyAsync(&h, e->bad_ids, 4, cudaMemcpyDeviceToHost, st));
        DPH_CUDA(cudaStreamSynchronize(st));
        if (h) { DPH_CUDA(cudaMemsetAsync(e->bad_ids, 0, 4, st)); dph_set_error("encoder: input_ids / token_type_ids outside the embedding tables (IndexError in torch)"); return 1; }
    } else {
        e->bad_pending = true;
    }
    return 0;
}

// The tower body shared by both forwards: embedding LayerNorm and the 12 layers of `ng` towers (weights towers[g], workspace slot g)
// as one grouped problem.
//   cls_only (query side): the last layer keeps only the [CLS] rows (see below); its result is in ctx[g][:B] (S >= 2) or x[g] (S == 1).
//   else (phrase side): every row; the last layer stops BEFORE its output LayerNorm, leaving LayerNorm's input in x[g] for the fused
//   phrase head.
//   long_attention: 64 < S <= 512 runs on attention_long.cu (the query side keeps the SIMT kernels above S = 64).
static int run_towers(dph_encoder* e, const int* towers, int ng, const long long* d_ids, const long long* d_mask, const long long* d_tt, int B,
                      int S, bool cls_only, bool long_attention) {
    cudaStream_t st = e->stream;
    const int64_t T = (int64_t)B * S;
    // bf16x3 mode: (hi, lo) planes of the three T x 768 GEMM inputs (x, ctx, a) live in act_hi / act_lo; their producers (LayerNorm,
    // attention) write them, so no separate split pass runs.  The T x 3072 FFN intermediate's planes live in ffn[] (see `linear`).
    unsigned short *xh[2] = {}, *xl[2] = {}, *ch[2] = {}, *cl[2] = {}, *ah[2] = {}, *al[2] = {};
    for (int t = 0; t < ng; t++) {
        xh[t] = reinterpret_cast<unsigned short*>(e->act_hi[t]); xl[t] = reinterpret_cast<unsigned short*>(e->act_lo[t]);
        ch[t] = xh[t] + T * ENC_H; cl[t] = xl[t] + T * ENC_H;
        ah[t] = ch[t] + T * ENC_H; al[t] = cl[t] + T * ENC_H;
    }
    const TowerW* W[2] = {&e->tw[towers[0]], &e->tw[towers[ng - 1]]};
    {
        EmbedArgs a = {};
        a.ids = d_ids; a.tt = d_tt; a.S = S;
        for (int t = 0; t < ng; t++) { a.word[t] = W[t]->word; a.pos[t] = W[t]->pos; a.type[t] = W[t]->type; a.g[t] = W[t]->embg; a.b[t] = W[t]->embb; a.out[t] = e->x[t]; }
        a.vocab = e->vocab; a.type_vocab = e->type_vocab; a.bad = e->bad_ids;
        for (int t = 0; t < ng; t++) { a.out_hi[t] = e->precise == 2 ? xh[t] : nullptr; a.out_lo[t] = e->precise == 2 ? xl[t] : nullptr; }
        embed_ln_kernel<<<dim3((unsigned)T, (unsigned)ng), 256, 0, st>>>(a);
        DPH_CUDA(cudaGetLastError());
    }
    if (e->precise == 1) DPH_TRY(ensure_split_weights(e, towers, ng));
    if (e->precise == 2) DPH_TRY(ensure_bf16_weights(e, towers, ng));
    // one grouped linear layer: out = act(in . W^T + b) + residual; m = which weight of the layer (0 qkv, 1 attn out, 2 ffn in, 3 ffn out)
    unsigned short* const PH[3][2] = {{xh[0], xh[1]}, {ch[0], ch[1]}, {ah[0], ah[1]}};
    unsigned short* const PL[3][2] = {{xl[0], xl[1]}, {cl[0], cl[1]}, {al[0], al[1]}};
    // planes_ready (bf16x3 mode): the producer of `in` already wrote its (hi, lo) planes into PH[m] / PL[m]
    auto linear = [&](int l, int m, float* const in[2], const float* const bias[2], float* const resid[2], float* const out[2], int N, int K, int act,
                      long long rows, bool planes_ready) -> int {
        const float* Wfull[2] = {};
        for (int t = 0; t < ng; t++) {
            const LayerW& Lt = W[t]->L[l];
            Wfull[t] = m == 0 ? Lt.Wqkv : m == 1 ? Lt.Wo : m == 2 ? Lt.Wi : Lt.Wo2;
        }
        const float* R[2] = {resid ? resid[0] : nullptr, resid ? resid[1] : nullptr};
        if (!e->precise) {
            const float* A[2] = {in[0], in[1]};
            return dph_launch_gemm_tf32(ng, A, Wfull, bias, resid ? R : nullptr, out, (int)rows, N, K, act, st, nullptr, nullptr);
        }
        if (e->precise == 2) {
            // bf16x3: operands as (hi, lo) bf16 planes.  The FFN intermediate never exists in fp32: the GELU epilogue of GEMM m = 2
            // writes its planes (into the memory of `out`), GEMM m = 3 reads them; the other inputs' planes come from their producers
            // (LayerNorm / embedding / tensor-core attention) or, failing that, from one split pass.
            const void *Whi[2] = {}, *Wlo[2] = {}, *Ahi[2] = {}, *Alo[2] = {};
            void *Ohi[2] = {nullptr, nullptr}, *Olo[2] = {nullptr, nullptr};
            for (int t = 0; t < ng; t++) {
                bf16_ptrs(e, towers[t], l, m, &Whi[t], &Wlo[t]);
                if (m == 3) {                                                     // planes left by GEMM m = 2 in `in`
                    Ahi[t] = in[t]; Alo[t] = reinterpret_cast<const unsigned short*>(in[t]) + rows * (long long)K;
                } else {
                    if (!planes_ready) DPH_TRY(dph_launch_split_bf16(in[t], PH[m][t], PL[m][t], rows * K, st));
                    Ahi[t] = PH[m][t]; Alo[t] = PL[m][t];
                }
                if (m == 2) { Ohi[t] = out[t]; Olo[t] = reinterpret_cast<unsigned short*>(out[t]) + rows * (long long)N; }
            }
            return dph_launch_gemm_bf16x3(ng, Ahi, Alo, Whi, Wlo, bias, resid ? R : nullptr, m == 2 ? nullptr : out, m == 2 ? Ohi : nullptr,
                                          m == 2 ? Olo : nullptr, (int)rows, N, K, act, st);
        }
        const float *Whi[2] = {}, *Wlo[2] = {};
        for (int t = 0; t < ng; t++) {
            split_ptrs(e, towers[t], l, m, &Whi[t], &Wlo[t]);
            DPH_TRY(dph_launch_split_tf32(in[t], e->act_hi[t], e->act_lo[t], rows * K, st));
        }
        const float* Ahi[2] = {e->act_hi[0], e->act_hi[1]}; const float* Alo[2] = {e->act_lo[0], e->act_lo[1]};
        return dph_launch_gemm_tf32(ng, Ahi, Whi, bias, resid ? R : nullptr, out, (int)rows, N, K, act, st, Alo, Wlo);
    };
    for (int l = 0; l < ENC_LAYERS; l++) {
        const LayerW &L0 = W[0]->L[l], &L1 = W[1]->L[l];
        float* X[2] = {e->x[0], e->x[1]};
        float* QKV[2] = {e->qkv[0], e->qkv[1]};
        float* CTX[2] = {e->ctx[0], e->ctx[1]};
        float* A2[2] = {e->a[0], e->a[1]};
        float* FF[2] = {e->ffn[0], e->ffn[1]};
        const float* bqkv[2] = {L0.bqkv, L1.bqkv}; const float* bo[2] = {L0.bo, L1.bo}; const float* bi[2] = {L0.bi, L1.bi}; const float* bo2[2] = {L0.bo2, L1.bo2};
        const bool bx = e->precise == 2;
        DPH_TRY(linear(l, 0, X, bqkv, nullptr, QKV, 3 * ENC_H, ENC_H, 0, T, bx));          // x planes: embedding LayerNorm / previous layer's LayerNorm
        AttnArgs aa; aa.qkv[0] = e->qkv[0]; aa.qkv[1] = e->qkv[1]; aa.ctx[0] = e->ctx[0]; aa.ctx[1] = e->ctx[1]; aa.mask = d_mask; aa.S = S;
        bool ctx_planes = false;
        if (e->attention_tc && S <= 64) {      // tensor cores: TF32 in the 1xTF32 mode, the bf16 (hi, lo) plane kernel (fp32-accurate) in the precise modes
            const float* q2[2] = {e->qkv[0], e->qkv[1]}; float* c2[2] = {e->ctx[0], e->ctx[1]};
            DPH_TRY(dph_launch_attention_tc(q2, c2, d_mask, B, S, T, st, e->precise ? 1 : 0, bx ? ch : nullptr, bx ? cl : nullptr, ng));
            ctx_planes = bx;
        } else if (e->attention_tc && long_attention) {
            for (int t = 0; t < ng; t++)
                DPH_TRY(dph_launch_attention_long(e->qkv[t], e->ctx[t], d_mask, B, S, st, e->precise ? 1 : 0, bx ? ch[t] : nullptr, bx ? cl[t] : nullptr));
            ctx_planes = bx;
        } else {
            DPH_TRY(launch_attention(aa, B, ng, st));
        }
        // Query side: only position 0 of the LAST layer is returned (encoder.py:116-117): after its attention, everything (attention
        // output projection, both LayerNorms, the FFN) runs on the B [CLS] rows instead of all B*S tokens.
        const bool last = cls_only && (l == ENC_LAYERS - 1) && S >= 2;      // (S == 1: the scratch aliasing below needs T >= 2B rows)
        long long rows = T;
        if (last) {
            rows = B;
            const unsigned gb = (unsigned)((B * (ENC_H / 4) + 255) / 256);
            gather_cls_kernel<<<dim3(gb, (unsigned)ng), 256, 0, st>>>(e->ctx[0], e->ctx[1], e->ffn[0], e->ffn[1], S, B);                         // ctx rows  -> ffn[:B]  (scratch)
            gather_cls_kernel<<<dim3(gb, (unsigned)ng), 256, 0, st>>>(e->x[0], e->x[1], e->ffn[0] + (size_t)B * ENC_H, e->ffn[1] + (size_t)B * ENC_H, S, B);   // residual rows
            DPH_CUDA(cudaGetLastError());
            CTX[0] = e->ffn[0]; CTX[1] = e->ffn[1];
            X[0] = e->ffn[0] + (size_t)B * ENC_H; X[1] = e->ffn[1] + (size_t)B * ENC_H;
            FF[0] = e->qkv[0]; FF[1] = e->qkv[1];                                                                                     // qkv is dead after attention: [B, 3072] fits
        }
        DPH_TRY(linear(l, 1, CTX, bo, X, A2, ENC_H, ENC_H, 0, rows, ctx_planes && !last));           // dense + residual (last layer: gathered rows, split here)
        LnArgs ln1 = {}; for (int t = 0; t < ng; t++) { ln1.in[t] = e->a[t]; ln1.out[t] = e->a[t]; ln1.out_hi[t] = bx ? ah[t] : nullptr; ln1.out_lo[t] = bx ? al[t] : nullptr; }
        ln1.g[0] = L0.ln1g; ln1.g[1] = L1.ln1g; ln1.b[0] = L0.ln1b; ln1.b[1] = L1.ln1b;
        ln1.rows = rows; ln1.in_stride = ENC_H; ln1.out_stride = ENC_H;
        layernorm_kernel<<<dim3((unsigned)((rows + 7) / 8), (unsigned)ng), 256, 0, st>>>(ln1);
        DPH_CUDA(cudaGetLastError());
        DPH_TRY(linear(l, 2, A2, bi, nullptr, FF, ENC_FF, ENC_H, 1, rows, bx));                          // intermediate + erf-GELU
        float* XO[2] = {last ? e->ctx[0] : e->x[0], last ? e->ctx[1] : e->x[1]};                         // last layer: dense [B,768] result in ctx
        DPH_TRY(linear(l, 3, FF, bo2, A2, XO, ENC_H, ENC_FF, 0, rows, bx));                              // output dense + residual
        if (!cls_only && l == ENC_LAYERS - 1) break;                                                     // phrase side: fused head LayerNorm
        LnArgs ln2 = {}; for (int t = 0; t < ng; t++) { ln2.in[t] = XO[t]; ln2.out[t] = XO[t]; ln2.out_hi[t] = (bx && !last) ? xh[t] : nullptr; ln2.out_lo[t] = (bx && !last) ? xl[t] : nullptr; }
        ln2.g[0] = L0.ln2g; ln2.g[1] = L1.ln2g; ln2.b[0] = L0.ln2b; ln2.b[1] = L1.ln2b;
        ln2.rows = rows; ln2.in_stride = ENC_H; ln2.out_stride = ENC_H;
        layernorm_kernel<<<dim3((unsigned)((rows + 7) / 8), (unsigned)ng), 256, 0, st>>>(ln2);
        DPH_CUDA(cudaGetLastError());
    }
    return 0;
}

// == Encoder.forward(input_ids_, attention_mask_, token_type_ids_, return_query=True) (encoder.py:146-152):
// ids/mask/tt int64 [B,S]; start_out/end_out fp32 [B,768] (the reference returns [B,1,768]).
DPH_API int dph_encoder_embed_query(dph_encoder* e, const int64_t* ids, const int64_t* mask, const int64_t* tt, int B, int S, float* start_out,
                                    float* end_out, int mem) {
    DPH_CHECK(e && e->blob[0] && e->blob[1], "encoder weights not loaded");
    DPH_CHECK(B >= 1 && S >= 1 && S <= ENC_MAX_S && S <= e->max_pos, "sequence length out of range (1..384)");
    cudaStream_t st = e->stream;
    const long long *d_ids, *d_mask, *d_tt;
    DPH_TRY(begin_forward(e, ids, mask, tt, B, S, 2, mem, &d_ids, &d_mask, &d_tt));
    static const int kQueryTowers[2] = {0, 1};
    DPH_TRY(run_towers(e, kQueryTowers, 2, d_ids, d_mask, d_tt, B, S, true, false));
    // hidden state at position 0 of every sequence ([:, :1, :], encoder.py:116-117)
    float* ds = mem == DPH_MEM_HOST ? e->out_s : start_out;
    float* de = mem == DPH_MEM_HOST ? e->out_e : end_out;
    if (S >= 2) {
        DPH_CUDA(cudaMemcpyAsync(ds, e->ctx[0], (size_t)B * ENC_H * 4, cudaMemcpyDeviceToDevice, st));
        DPH_CUDA(cudaMemcpyAsync(de, e->ctx[1], (size_t)B * ENC_H * 4, cudaMemcpyDeviceToDevice, st));
    } else {
        DPH_CUDA(cudaMemcpyAsync(ds, e->x[0], (size_t)B * ENC_H * 4, cudaMemcpyDeviceToDevice, st));
        DPH_CUDA(cudaMemcpyAsync(de, e->x[1], (size_t)B * ENC_H * 4, cudaMemcpyDeviceToDevice, st));
    }
    if (mem == DPH_MEM_HOST) {
        DPH_CUDA(cudaMemcpyAsync(start_out, ds, (size_t)B * ENC_H * 4, cudaMemcpyDeviceToHost, st));
        DPH_CUDA(cudaMemcpyAsync(end_out, de, (size_t)B * ENC_H * 4, cudaMemcpyDeviceToHost, st));
    }
    return end_forward(e, mem);
}

// ---- phrase head: the last layer's output LayerNorm fused with filter_linear and the int8 dump quantisation ----------------------
// One warp per token row, as layernorm_kernel (same two-pass mean / variance, same arithmetic for the normalised row), then
//   filter_start / filter_end = <row, W[0 / 1]> + b[0 / 1]                                      (encoder.py:137-141)
//   out_q = int8(rint(clamp((row - offset) * scale, -128, 127)))                   (float_to_int8, embed_utils.py:141-145)
// with the subtraction and the product each rounded to fp32 like numpy on fp32 data, and round half to even like np.round.
struct HeadArgs { const float* in; const float* g; const float* b; const float* filt; long long rows;
                  float* out; float* fs; float* fe; signed char* q; float offset, scale; };      // out, q nullable
__global__ void __launch_bounds__(256) phrase_head_kernel(HeadArgs a) {
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= a.rows) return;
    const float4* x = reinterpret_cast<const float4*>(a.in + row * ENC_H);
    float4 v[6];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 6; i++) { v[i] = x[lane + 32 * i]; s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float mean = s * (1.0f / ENC_H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
    const float rstd = rsqrtf(q * (1.0f / ENC_H) + 1e-12f);
    const float4* g = reinterpret_cast<const float4*>(a.g);
    const float4* b = reinterpret_cast<const float4*>(a.b);
    const float4* w0 = reinterpret_cast<const float4*>(a.filt);
    const float4* w1 = reinterpret_cast<const float4*>(a.filt + ENC_H);
    float f0 = 0.f, f1 = 0.f;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const int c = lane + 32 * i;
        const float4 gg = g[c], bb = b[c];
        const float4 r4 = make_float4(v[i].x * rstd * gg.x + bb.x, v[i].y * rstd * gg.y + bb.y, v[i].z * rstd * gg.z + bb.z, v[i].w * rstd * gg.w + bb.w);
        if (a.out) reinterpret_cast<float4*>(a.out + row * ENC_H)[c] = r4;
        const float4 a0 = w0[c], a1 = w1[c];
        f0 = fmaf(r4.x, a0.x, fmaf(r4.y, a0.y, fmaf(r4.z, a0.z, fmaf(r4.w, a0.w, f0))));
        f1 = fmaf(r4.x, a1.x, fmaf(r4.y, a1.y, fmaf(r4.z, a1.z, fmaf(r4.w, a1.w, f1))));
        if (a.q) {
            const float e[4] = {r4.x, r4.y, r4.z, r4.w};
            char4 c4;
            signed char* cp = reinterpret_cast<signed char*>(&c4);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float t = fminf(fmaxf(__fmul_rn(__fsub_rn(e[k], a.offset), a.scale), -128.f), 127.f);
                cp[k] = (signed char)(int)rintf(t);
            }
            reinterpret_cast<char4*>(a.q + row * ENC_H)[c] = c4;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { f0 += __shfl_xor_sync(0xffffffffu, f0, off); f1 += __shfl_xor_sync(0xffffffffu, f1, off); }
    if (lane == 0) { a.fs[row] = f0 + a.filt[2 * ENC_H]; a.fe[row] = f1 + a.filt[2 * ENC_H + 1]; }
}

// == Encoder.forward(input_ids=..., attention_mask=..., token_type_ids=..., return_phrase=True) (encoder.py:130-144) and the
// int8 `start` that write_phrases stores: the phrase tower over every token (one tower, no [CLS] gather), the last LayerNorm fused
// with the filter head and, when out_q is given, float_to_int8(out, dense_offset, dense_scale).
DPH_API int dph_encoder_embed_phrase(dph_encoder* e, const int64_t* ids, const int64_t* mask, const int64_t* tt, int B, int S, float* out,
                                     float* filter_start, float* filter_end, int8_t* out_q, float dense_offset, float dense_scale, int mem) {
    DPH_CHECK(e && e->blob[2] && e->filt, "phrase encoder weights (tower 2 + filter head) not loaded");
    DPH_CHECK(B >= 1 && S >= 1 && S <= ENC_MAX_S_LONG && S <= e->max_pos, "sequence length out of range (1..512)");
    DPH_CHECK(e->attention_tc || S <= ENC_MAX_S, "the SIMT attention kernels handle S <= 384 (set_attention(1) for longer sequences)");
    DPH_CHECK(filter_start && filter_end, "filter_start / filter_end are required");
    cudaStream_t st = e->stream;
    const int64_t T = (int64_t)B * S;
    const long long *d_ids, *d_mask, *d_tt;
    DPH_TRY(begin_forward(e, ids, mask, tt, B, S, 1, mem, &d_ids, &d_mask, &d_tt));
    static const int kPhraseTower[1] = {2};
    DPH_TRY(run_towers(e, kPhraseTower, 1, d_ids, d_mask, d_tt, B, S, false, true));
    // host buffers: results staged in the workspace (out over the head's input rows, which each warp reads before it writes; the
    // logits and codes in qkv, dead after the last attention)
    const bool host = mem == DPH_MEM_HOST;
    HeadArgs h;
    h.in = e->x[0]; h.g = e->tw[2].L[ENC_LAYERS - 1].ln2g; h.b = e->tw[2].L[ENC_LAYERS - 1].ln2b; h.filt = e->filt; h.rows = T;
    h.out = out ? (host ? e->x[0] : out) : nullptr;
    h.fs = host ? e->qkv[0] : filter_start;
    h.fe = host ? e->qkv[0] + T : filter_end;
    h.q = out_q ? (host ? reinterpret_cast<signed char*>(e->qkv[0] + 2 * T) : reinterpret_cast<signed char*>(out_q)) : nullptr;
    h.offset = dense_offset; h.scale = dense_scale;
    phrase_head_kernel<<<(unsigned)((T + 7) / 8), 256, 0, st>>>(h);
    DPH_CUDA(cudaGetLastError());
    if (host) {
        if (out) DPH_CUDA(cudaMemcpyAsync(out, h.out, (size_t)T * ENC_H * 4, cudaMemcpyDeviceToHost, st));
        DPH_CUDA(cudaMemcpyAsync(filter_start, h.fs, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
        DPH_CUDA(cudaMemcpyAsync(filter_end, h.fe, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
        if (out_q) DPH_CUDA(cudaMemcpyAsync(out_q, h.q, (size_t)T * ENC_H, cudaMemcpyDeviceToHost, st));
    }
    return end_forward(e, mem);
}
