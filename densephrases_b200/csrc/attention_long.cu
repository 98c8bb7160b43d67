// attention_long.cu -- BERT self-attention for context-length sequences (64 < S <= 512: max_seq_length 384 by default, 512 in
// the phrase-dump recipe) on the 5th-gen tensor cores.  Same arithmetic as attention_tc.cu and HF BertSelfAttention behind
// Encoder.embed_phrase: softmax(Q K^T / 8 + (1 - mask) * -10000) V per head, fp32 softmax.  Two variants, one template:
//   BX = false: Q, K, P, V^T as TF32 operands, one kind::tf32 MMA per contraction (precision mode 0);
//   BX = true : Q, K, P, V^T as bf16 (hi, lo) planes, every contraction hi.lo + lo.hi + hi.hi in kind::f16 (~2^-17 relative;
//               modes 1 and 2), and the context is also written as bf16 planes for the bf16x3 output projection.
//
// At S = 512 a 128-row fp32 score tile is 512 TMEM columns -- all of TMEM -- so the kernel never holds a whole score row: it walks
// the keys in tiles of 64 with an online softmax (running max m and sum l per row, flash-attention style).
// One CTA (128 threads) handles 128 query rows of one head of one sequence; thread r owns query row r.
//   0. Q (128 x 64) is staged once.  Threads stage every operand themselves (global -> registers -> swizzled shared memory): the
//      bf16 variant has to pass every element through registers to split it anyway, and one staging path serves both variants.
//   per key tile j (64 keys):
//   1. S = Q K_j^T : UMMA 128x64 into TMEM columns 0..63; meanwhile the loads of K_{j+1} are issued into registers;
//   2. thread r: tcgen05.ld of its 64 scores, scale + mask, m_new = max(m, tile max), p = exp(s - m_new), l = l e^(m - m_new) + sum p;
//      the unnormalised P row goes to shared memory in the swizzled K-major layout; K_{j+1} goes to the now idle K tile;
//   3. O_j = P V_j : UMMA 128x64 into TMEM columns 64..127; meanwhile the loads of V_{j+1} are issued; thread r then folds O_j
//      into its 64-float register accumulator, acc = acc e^(m_old - m_new) + O_j, and writes V_{j+1} to the now idle V^T tile.
//   Finally ctx = acc / l for the query rows < S.
// Rows are contiguous over sequences (T = B*S): a tile that crosses position S would hold the next sequence's rows, so keys at
// positions >= S are never loaded (zeros) and get probability exactly 0; padded keys at positions < S get the additive -10000 like
// the reference; query rows >= S are neither loaded nor stored.
// Budget per CTA: 96 KB of operand tiles (Q 32 KB | P 32 KB | K 16 KB | V^T 16 KB, the same in both variants: a TF32 row of 64 is
// 256 bytes = two 128-byte swizzle blocks, a bf16 row is one block per plane) + 1.6 KB tail and alignment slack; 128 TMEM columns.
// -> two CTAs per SM (shared memory bound; 256 of 512 TMEM columns).
#include "umma.cuh"
#include <cuda_bf16.h>

#define AL_H 768
#define AL_DH 64
#define AL_KT 64                        // keys per tile
#define AL_Q 0                          // Q operand  [128 rows x 64]: TF32 2 blocks [128 x 32 floats] | bf16 planes hi, lo
#define AL_P (32 * 1024)                // P operand  [128 rows x 64 keys], same layout as Q
#define AL_K (64 * 1024)                // K tile     [64 keys x 64]: TF32 2 blocks [64 x 32 floats] | bf16 planes hi, lo (8 KB each)
#define AL_V (80 * 1024)                // V^T tile   [64 d x 64 keys], same layout as K
#define AL_TAIL (96 * 1024)             // [2][64] additive key mask (double-buffered) | mbarrier | TMEM slot
#define AL_SMEM_BYTES (AL_TAIL + 2 * AL_KT * 4 + 64 + 1024)

struct AttnLongArgs { const float* qkv; float* ctx; const long long* mask; int S;
                      unsigned short* ctx_hi; unsigned short* ctx_lo; };             // BX only, nullable: bf16 (hi, lo) planes of the context

__device__ __forceinline__ void al_split2(float x0, float x1, unsigned& hi, unsigned& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const unsigned*>(&h);
    lo = *reinterpret_cast<const unsigned*>(&l);
}
__device__ __forceinline__ void al_split8(const float4& a, const float4& b, uint4& h, uint4& l) {
    al_split2(a.x, a.y, h.x, l.x); al_split2(a.z, a.w, h.y, l.y); al_split2(b.x, b.y, h.z, l.z); al_split2(b.z, b.w, h.w, l.w);
}

// one 64-element operand row (fp32 in registers) -> K-major SWIZZLE_128B tile(s), row r; `half` selects elements 32*half .. +31 when
// the caller holds only 8 float4 (v[0..7] = elements 32*half + 4c ..), else (half < 0) v[0..15] is the whole row.
// TF32: block kb = element / 32 at base + kb * blk, 16-byte chunk c at r*128 + ((c ^ (r & 7)) << 4).
// bf16: hi plane at base, lo plane at base + blk, 16-byte chunk q (8 elements) at r*128 + ((q ^ (r & 7)) << 4).
template <bool BX, int N4>
__device__ __forceinline__ void al_store_row(unsigned char* base, unsigned blk, unsigned r, int half, const float4 (&v)[N4]) {
    const int c0 = half < 0 ? 0 : half * 8;
    if constexpr (!BX) {
#pragma unroll
        for (int i = 0; i < N4; i++) {
            const unsigned c = (unsigned)(c0 + i);
            *reinterpret_cast<float4*>(base + (c >> 3) * blk + r * 128 + (((c & 7u) ^ (r & 7u)) << 4)) = v[i];
        }
    } else {
#pragma unroll
        for (int i = 0; i < N4; i += 2) {
            const unsigned q = (unsigned)((c0 + i) >> 1);
            uint4 h, l;
            al_split8(v[i], v[i + 1], h, l);
            const unsigned off = r * 128 + ((q ^ (r & 7u)) << 4);
            *reinterpret_cast<uint4*>(base + off) = h;
            *reinterpret_cast<uint4*>(base + blk + off) = l;
        }
    }
}

template <bool BX>
__global__ void __launch_bounds__(128, 2) attention_long_kernel(const AttnLongArgs a) {
    extern __shared__ __align__(1024) unsigned char alsm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int S = a.S;
    unsigned char* base = (unsigned char*)((((unsigned long long)alsm) + 1023ull) & ~1023ull);   // swizzle atoms: 1024-byte aligned
    const unsigned sbase = smem_u32(base);
    float* mb = reinterpret_cast<float*>(base + AL_TAIL);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(base + AL_TAIL + 2 * AL_KT * 4);
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(base + AL_TAIL + 2 * AL_KT * 4 + 16);
    const unsigned bar_mma = smem_u32(bar);
    const long long row0 = (long long)b * S;
    const float* qkv = a.qkv + h * AL_DH;

    if (tid == 0) {
        mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(128) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // Q row of this thread (query position qt*128 + tid)
    const int qpos = qt * 128 + tid;
    {
        float4 v[16];
        const float4* src = reinterpret_cast<const float4*>(qkv + (row0 + qpos) * (3 * AL_H));
        const bool ok = qpos < S;
#pragma unroll
        for (int c = 0; c < 16; c++) v[c] = ok ? __ldg(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        al_store_row<BX, 16>(base + AL_Q, 16 * 1024, (unsigned)tid, -1, v);
    }
    // K / V staging: thread t holds key kk = t & 63, elements 32*half .. +31 with half = t >> 6
    const int kk = tid & 63, half = tid >> 6;
    float4 kr[8], vr[8];
    float mval = 0.f;
    auto src_row = [&](int j, int op) {          // op 1: K, 2: V; keys of the next sequence (or past the end) are never read
        return reinterpret_cast<const float4*>(qkv + (row0 + j * AL_KT + kk) * (3 * AL_H) + op * AL_H + half * 32);
    };
    auto load_k = [&](int j) {
        const bool ok = j * AL_KT + kk < S;
        const float4* ks = src_row(j, 1);
#pragma unroll
        for (int c = 0; c < 8; c++) kr[c] = ok ? __ldg(ks + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        mval = ok ? (1.0f - (float)a.mask[row0 + j * AL_KT + kk]) * -10000.0f : 0.f;
    };
    auto load_v = [&](int j) {
        const bool ok = j * AL_KT + kk < S;
        const float4* vs = src_row(j, 2);
#pragma unroll
        for (int c = 0; c < 8; c++) vr[c] = ok ? __ldg(vs + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto store_k = [&](int j) {
        al_store_row<BX, 8>(base + AL_K, 8 * 1024, (unsigned)kk, half, kr);
        if (half == 0) mb[(j & 1) * AL_KT + kk] = mval;
    };
    auto store_v = [&]() {
        // V^T: element (d, key).  TF32: block kb = key / 32, at d*128 + (((k >> 2) ^ (d & 7)) << 4) + (k & 3)*4 with k = key % 32;
        // bf16: at d*128 + (((key >> 3) ^ (d & 7)) << 4) + (key & 7)*2.  A warp's 32 lanes (consecutive keys, same d) fill one row.
        const unsigned key = (unsigned)kk;
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const float e[4] = {vr[c].x, vr[c].y, vr[c].z, vr[c].w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const unsigned d = (unsigned)(half * 32 + c * 4 + t);
                if constexpr (!BX) {
                    const unsigned k = key & 31u;
                    *reinterpret_cast<float*>(base + AL_V + (key >> 5) * 8192 + d * 128 + ((((k >> 2) ^ (d & 7u)) << 4) | ((k & 3u) << 2))) = e[t];
                } else {
                    const unsigned off = d * 128 + ((((key >> 3) ^ (d & 7u)) << 4) | ((key & 7u) << 1));
                    const __nv_bfloat16 hb = __float2bfloat16_rn(e[t]);
                    *reinterpret_cast<__nv_bfloat16*>(base + AL_V + off) = hb;
                    *reinterpret_cast<__nv_bfloat16*>(base + AL_V + 8192 + off) = __float2bfloat16_rn(e[t] - __bfloat162float(hb));
                }
            }
        }
    };
    load_k(0); load_v(0);
    store_k(0); store_v();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_base = *tmem_slot;
    const unsigned lane_addr = tmem_base + ((unsigned)(warp * 32) << 16);

    // instruction descriptor: D = F32, A = B = TF32 (2) or BF16 (1), both K-major, N = 64 (>> 3 at bit 17), M = 128 (>> 4 at bit 24)
    constexpr unsigned AB = BX ? 1u : 2u;
    constexpr unsigned IDESC = (1u << 4) | (AB << 7) | (AB << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
    float acc[64];
#pragma unroll
    for (int d = 0; d < 64; d++) acc[d] = 0.f;
    float m = -3.0e38f, l = 0.f;
    const int nt = (S + AL_KT - 1) / AL_KT;
    for (int j = 0; j < nt; j++) {
        // ---- S = Q K_j^T -> TMEM columns 0..63 ----
        if (warp == 0) {
            if (lane == 0) {
                if constexpr (!BX) {
#pragma unroll
                    for (int kb = 0; kb < 2; kb++) {
                        const unsigned long long qd = make_sw128_desc(sbase + AL_Q + kb * 16384), kd = make_sw128_desc(sbase + AL_K + kb * 8192);
#pragma unroll
                        for (int k = 0; k < 4; k++) umma_tf32(tmem_base, qd + (unsigned long long)(k * 2), kd + (unsigned long long)(k * 2), IDESC, (kb | k) ? 1u : 0u);
                    }
                } else {
                    const unsigned long long qh = make_sw128_desc(sbase + AL_Q), ql = make_sw128_desc(sbase + AL_Q + 16384);
                    const unsigned long long kh = make_sw128_desc(sbase + AL_K), kl = make_sw128_desc(sbase + AL_K + 8192);
#pragma unroll
                    for (int k = 0; k < 4; k++) {            // UMMA_K = 16 bf16 = 32 bytes
                        const unsigned long long ko = (unsigned long long)(k * 2);
                        umma_bf16(tmem_base, qh + ko, kl + ko, IDESC, k ? 1u : 0u);
                        umma_bf16(tmem_base, ql + ko, kh + ko, IDESC, 1u);
                        umma_bf16(tmem_base, qh + ko, kh + ko, IDESC, 1u);
                    }
                }
                umma_commit(bar_mma);
            }
            __syncwarp();
        }
        if (j + 1 < nt) load_k(j + 1);          // lands during the softmax
        mbar_wait(bar_mma, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- online softmax of row tid over this tile's keys ----
        // Two passes over the two 32-column halves of the score row (TMEM is re-read rather than holding 64 scores next to the
        // 64-float accumulator): the tile max, then exp / sum / the P row.
        float alpha;
        {
            const float* mbj = mb + (j & 1) * AL_KT;
            const int nvalid = min(AL_KT, S - j * AL_KT);
            float mt = -3.0e38f;
#pragma unroll
            for (int hf = 0; hf < 2; hf++) {
                unsigned sc[32];
                tmem_ld32(lane_addr + (unsigned)(hf * 32), sc);
#pragma unroll
                for (int c = 0; c < 32; c++) if (hf * 32 + c < nvalid) mt = fmaxf(mt, __uint_as_float(sc[c]) * 0.125f + mbj[hf * 32 + c]);
            }
            const float m_new = fmaxf(m, mt);
            alpha = expf(m - m_new);
            float sum = 0.f;
            const unsigned r = (unsigned)tid;
#pragma unroll
            for (int hf = 0; hf < 2; hf++) {
                unsigned sc[32];
                tmem_ld32(lane_addr + (unsigned)(hf * 32), sc);
                float p[32];
#pragma unroll
                for (int c = 0; c < 32; c++) {
                    p[c] = (hf * 32 + c < nvalid) ? expf((__uint_as_float(sc[c]) * 0.125f + mbj[hf * 32 + c]) - m_new) : 0.f;
                    sum += p[c];
                }
                if constexpr (!BX) {         // keys 32 hf .. +31 = TF32 block hf
#pragma unroll
                    for (unsigned c = 0; c < 8; c++)
                        *reinterpret_cast<float4*>(base + AL_P + hf * 16384 + r * 128 + ((c ^ (r & 7u)) << 4)) =
                            make_float4(p[4 * c], p[4 * c + 1], p[4 * c + 2], p[4 * c + 3]);
                } else {                     // = 16-byte chunks 4 hf .. +3 of the bf16 planes
#pragma unroll
                    for (unsigned c = 0; c < 4; c++) {
                        uint4 hh, ll;
                        al_split8(make_float4(p[8 * c], p[8 * c + 1], p[8 * c + 2], p[8 * c + 3]),
                                  make_float4(p[8 * c + 4], p[8 * c + 5], p[8 * c + 6], p[8 * c + 7]), hh, ll);
                        const unsigned off = r * 128 + (((4u * hf + c) ^ (r & 7u)) << 4);
                        *reinterpret_cast<uint4*>(base + AL_P + off) = hh;
                        *reinterpret_cast<uint4*>(base + AL_P + 16384 + off) = ll;
                    }
                }
            }
            l = l * alpha + sum;
            m = m_new;
        }
        if (j + 1 < nt) store_k(j + 1);         // S = Q K_j^T is complete: the K tile (and mask slot j+1 & 1) is free
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- O_j = P V_j -> TMEM columns 64..127 ----
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                const unsigned d_o = tmem_base + 64u;
                if constexpr (!BX) {
#pragma unroll
                    for (int kb = 0; kb < 2; kb++) {
                        const unsigned long long pd = make_sw128_desc(sbase + AL_P + kb * 16384), vd = make_sw128_desc(sbase + AL_V + kb * 8192);
#pragma unroll
                        for (int k = 0; k < 4; k++) umma_tf32(d_o, pd + (unsigned long long)(k * 2), vd + (unsigned long long)(k * 2), IDESC, (kb | k) ? 1u : 0u);
                    }
                } else {
                    const unsigned long long ph = make_sw128_desc(sbase + AL_P), pl = make_sw128_desc(sbase + AL_P + 16384);
                    const unsigned long long vh = make_sw128_desc(sbase + AL_V), vl = make_sw128_desc(sbase + AL_V + 8192);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const unsigned long long ko = (unsigned long long)(k * 2);
                        umma_bf16(d_o, ph + ko, vl + ko, IDESC, k ? 1u : 0u);
                        umma_bf16(d_o, pl + ko, vh + ko, IDESC, 1u);
                        umma_bf16(d_o, ph + ko, vh + ko, IDESC, 1u);
                    }
                }
                umma_commit(bar_mma);
            }
            __syncwarp();
        }
        if (j + 1 < nt) load_v(j + 1);          // lands while P V runs
        mbar_wait(bar_mma, 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
            unsigned o[32];
            tmem_ld32(lane_addr + 64u + (unsigned)(hf * 32), o);
#pragma unroll
            for (int c = 0; c < 32; c++) acc[hf * 32 + c] = acc[hf * 32 + c] * alpha + __uint_as_float(o[c]);
        }
        if (j + 1 < nt) store_v();              // P V_j is complete: the V^T tile is free
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (qpos < S) {
        const float inv = 1.0f / l;
        float* out = a.ctx + (row0 + qpos) * AL_H + h * AL_DH;
#pragma unroll
        for (int c = 0; c < 64; c += 4)
            *reinterpret_cast<float4*>(out + c) = make_float4(acc[c] * inv, acc[c + 1] * inv, acc[c + 2] * inv, acc[c + 3] * inv);
        if constexpr (BX) {
            if (a.ctx_hi) {               // the same row segment as (hi, lo) bf16 planes for the bf16x3 output projection
                unsigned short* gh = a.ctx_hi + (row0 + qpos) * AL_H + h * AL_DH;
                unsigned short* gl = a.ctx_lo + (row0 + qpos) * AL_H + h * AL_DH;
#pragma unroll
                for (int c = 0; c < 64; c += 8) {
                    uint4 hh, ll;
                    al_split8(make_float4(acc[c] * inv, acc[c + 1] * inv, acc[c + 2] * inv, acc[c + 3] * inv),
                              make_float4(acc[c + 4] * inv, acc[c + 5] * inv, acc[c + 6] * inv, acc[c + 7] * inv), hh, ll);
                    *reinterpret_cast<uint4*>(gh + c) = hh;
                    *reinterpret_cast<uint4*>(gl + c) = ll;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(128) : "memory");
}

// qkv: [B*S, 2304] fp32 (Q | K | V, heads contiguous inside each), ctx: [B*S, 768]; mask int64 [B, S]; 64 < S <= 512, 12 heads.
// split = 0: TF32 operands; 1: bf16 (hi, lo) planes (ctx_hi / ctx_lo, nullable, receive the context's planes).
int dph_launch_attention_long(const float* qkv, float* ctx, const long long* mask, int B, int S, cudaStream_t st, int split,
                              unsigned short* ctx_hi, unsigned short* ctx_lo) {
    DPH_CHECK(S > 64 && S <= 512 && B >= 1, "attention_long: S must be 65..512");
    static DphPerDeviceOnce once;
    if (once.first()) {
        DPH_CUDA(cudaFuncSetAttribute(attention_long_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AL_SMEM_BYTES));
        DPH_CUDA(cudaFuncSetAttribute(attention_long_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, AL_SMEM_BYTES));
    }
    AttnLongArgs a;
    a.qkv = qkv; a.ctx = ctx; a.mask = mask; a.S = S; a.ctx_hi = ctx_hi; a.ctx_lo = ctx_lo;
    const dim3 grid((unsigned)((S + 127) / 128), 12, (unsigned)B);
    if (split) attention_long_kernel<true><<<grid, 128, AL_SMEM_BYTES, st>>>(a);
    else attention_long_kernel<false><<<grid, 128, AL_SMEM_BYTES, st>>>(a);
    DPH_CUDA(cudaGetLastError());
    return 0;
}
