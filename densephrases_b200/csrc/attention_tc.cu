// attention_tc.cu -- BERT self-attention for query-length sequences (S <= 64: max_query_length 24 / 32 / 64, options.py:38,
// Makefile:441) on the 5th-gen tensor cores.  Same arithmetic as HF BertSelfAttention behind Encoder.embed_query
// (/root/reference/densephrases/encoder.py:101-118): softmax(Q K^T / 8 + (1 - mask) * -10000) V per head, fp32 softmax; the two
// contractions run as tcgen05.mma kind::tf32 with fp32 accumulation in TMEM (torch 1.9 -- the reference's pin -- also ran the
// attention matmuls in TF32 on Ampere+).
// attention_tc_bx_kernel (further down) is the fp32-accurate variant used by the 3xTF32 / bf16x3 encoder modes: Q, K, P and V^T are
// carried as bf16 (hi, lo) planes and every contraction is hi.lo + lo.hi + hi.hi (three kind::f16 MMAs, ~2^-17 relative).
//
// One CTA (128 threads) handles TWO heads of one sequence of one tower so that every MMA has M = 128:
//   rows 0..63 = tokens of head h0, rows 64..127 = tokens of head h0+1.
//   1. TMA (SWIZZLE_128B boxes of 32 floats x 64 rows out of the [T, 2304] QKV activation) stages Q and K of both heads as two
//      K-major [128 x 64] operands; meanwhile the 128 threads stage V TRANSPOSED ([d][key], the K-major B operand of P V) with
//      the same 128-byte swizzle written by hand, one warp per 32-key block, conflict-free.
//   2. S = Q K^T : 8 x UMMA 128x128x8 into TMEM columns 0..127.  Only the diagonal 64x64 blocks are meaningful (a head's queries
//      against its own keys); the off-diagonal half is wasted tensor work that costs nothing at this size.
//   3. Thread r owns row r: tcgen05.ld of its head's 64 scores, scale + mask + softmax in registers, P row written back to shared
//      memory (over the dead Q tile) in the swizzled K-major layout.
//   4. O = P V : P [128 x 64] against V^T of head h0 -> columns 128..191 and against V^T of head h0+1 -> columns 192..255
//      (2 x 8 UMMA 128x64x8); rows 0..63 read the first result, rows 64..127 the second.
//   5. tcgen05.ld -> 256-byte row segments of the context activation.
// ~97 KB shared memory and 256 TMEM columns per CTA -> two CTAs per SM.
#include "umma.cuh"
#include <cuda_bf16.h>

#define AT_H 768
#define AT_DH 64
#define AT_TILE (128 * 128)            // bytes of one [128 rows x 32 floats] swizzled operand block
#define AT_VT_TILE (64 * 128)          // bytes of one [64 d x 32 keys] block of V^T
#define AT_SMEM_QK 0                   // Q kb0, Q kb1, K kb0, K kb1 (P kb0, kb1 alias Q after S is complete)
#define AT_SMEM_VT (4 * AT_TILE)       // [head][kb] : 4 blocks
#define AT_SMEM_TAIL (AT_SMEM_VT + 4 * AT_VT_TILE)
#define AT_SMEM_BYTES (AT_SMEM_TAIL + 64 * 4 + 64 + 1024)

struct AttnTcMaps { CUtensorMap qkv[2]; };
struct AttnTcArgs { const float* qkv[2]; float* ctx[2]; const long long* mask; int S;
                    unsigned short* ctx_hi[2]; unsigned short* ctx_lo[2]; };       // bx kernel only, nullable: bf16 (hi, lo) planes of the context

__device__ __forceinline__ unsigned short bf16_bits_rn(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }
// x -> (hi, lo) bf16 bit patterns with x = hi + lo up to 2^-18 |x|; two elements per 32-bit word (element 0 in the low half):
// one packed convert for the hi parts, one for the remainders
__device__ __forceinline__ void bx_split2(float x0, float x1, unsigned& hi, unsigned& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const unsigned*>(&h);
    lo = *reinterpret_cast<const unsigned*>(&l);
}

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__global__ void __launch_bounds__(128, 2) attention_tc_kernel(const __grid_constant__ AttnTcMaps maps, const AttnTcArgs a) {
    extern __shared__ __align__(1024) unsigned char atsm[];
    // swizzle atoms need 1024-byte alignment: the window is rounded up here (the launch reserves 1 KB of slack)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int hp = blockIdx.x, b = blockIdx.y, tw = blockIdx.z;
    const int S = a.S, h0 = hp * 2;
    unsigned char* base = (unsigned char*)((((unsigned long long)atsm) + 1023ull) & ~1023ull);
    const unsigned sbase = smem_u32(base);
    float* mb = reinterpret_cast<float*>(base + AT_SMEM_TAIL);                         // [64] additive key mask
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(base + AT_SMEM_TAIL + 256);   // tma, mma
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(base + AT_SMEM_TAIL + 256 + 32);
    const unsigned bar_tma = smem_u32(bars), bar_mma = smem_u32(bars + 1);
    const CUtensorMap* map = &maps.qkv[tw];
    const long long row0 = (long long)b * S;

    if (tid == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
        mbar_init(bar_tma, 1); mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_base = *tmem_slot;

    if (tid == 0) {
        mbar_expect_tx(bar_tma, 4 * AT_TILE);
#pragma unroll
        for (int op = 0; op < 2; op++)              // 0: Q (columns 0..767), 1: K (columns 768..1535)
#pragma unroll
            for (int kb = 0; kb < 2; kb++)
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
                    tma_load_2d(sbase + AT_SMEM_QK + (op * 2 + kb) * AT_TILE + hh * (64 * 128), map, op * AT_H + (h0 + hh) * AT_DH + kb * 32, (int)row0, bar_tma);
    }
    // V^T, hand-swizzled: warp w stages block (head w>>1, keys 32(w&1) .. +31); lane = key, so the 32 lanes of one store fill one
    // 128-byte row (d fixed) -- every bank once.  Element (d, kk) of a block: d*128 + ((kk>>2 ^ d&7) << 4) + (kk&3)*4.
    {
        const int hh = warp >> 1, j = (warp & 1) * 32 + lane;
        const bool ok = j < S;
        const float4* src = reinterpret_cast<const float4*>(a.qkv[tw] + (row0 + j) * (3 * AT_H) + 2 * AT_H + (h0 + hh) * AT_DH);
        unsigned char* blk = base + AT_SMEM_VT + warp * AT_VT_TILE;
        const unsigned kk = (unsigned)lane;
#pragma unroll 4
        for (int d4 = 0; d4 < 16; d4++) {
            const float4 v = ok ? __ldg(src + d4) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const unsigned d = (unsigned)(d4 * 4 + t);
                *reinterpret_cast<float*>(blk + d * 128 + ((((kk >> 2) ^ (d & 7u)) << 4) | ((kk & 3u) << 2))) = e[t];
            }
        }
        if (tid < 64) mb[tid] = (tid < S) ? (1.0f - (float)a.mask[row0 + tid]) * -10000.0f : 0.f;
    }
    fence_proxy_async_smem();                       // generic-proxy stores above -> visible to the tensor core's async-proxy reads
    __syncthreads();

    // instruction descriptor: D = F32, A = B = TF32, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
    constexpr unsigned IDESC_S = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    constexpr unsigned IDESC_O = (1u << 4) | (2u << 7) | (2u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
    if (warp == 0) {
        mbar_wait(bar_tma, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
#pragma unroll
            for (int kb = 0; kb < 2; kb++) {
                const unsigned long long qd = make_sw128_desc(sbase + AT_SMEM_QK + kb * AT_TILE), kd = make_sw128_desc(sbase + AT_SMEM_QK + (2 + kb) * AT_TILE);
#pragma unroll
                for (int k = 0; k < 4; k++) umma_tf32(tmem_base, qd + (unsigned long long)(k * 2), kd + (unsigned long long)(k * 2), IDESC_S, (kb | k) ? 1u : 0u);
            }
            umma_commit(bar_mma);
        }
        __syncwarp();
    }
    mbar_wait(bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- softmax of row r = tid over its head's 64 keys ----
    const int hh = tid >> 6;                                    // which head of the pair (warp-uniform)
    const unsigned lane_addr = tmem_base + ((unsigned)(warp * 32) << 16);
    {
        unsigned s0[32], s1[32];
        tmem_ld32(lane_addr + (unsigned)(hh * 64), s0);
        tmem_ld32(lane_addr + (unsigned)(hh * 64 + 32), s1);
        float p[64];
        float mx = -3.0e38f;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            p[j] = __uint_as_float(s0[j]) * 0.125f + mb[j];
            p[j + 32] = __uint_as_float(s1[j]) * 0.125f + mb[j + 32];
        }
#pragma unroll
        for (int j = 0; j < 64; j++) if (j < S) mx = fmaxf(mx, p[j]);
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < 64; j++) { p[j] = (j < S) ? expf(p[j] - mx) : 0.f; sum += p[j]; }
        const float inv = 1.0f / sum;
        // P row -> blocks kb = 0,1 over the Q tile (S complete => the tensor core is done reading Q and K)
        const unsigned r = (unsigned)tid;
#pragma unroll
        for (int kb = 0; kb < 2; kb++)
#pragma unroll
            for (int c = 0; c < 8; c++) {
                const int j = kb * 32 + c * 4;
                *reinterpret_cast<float4*>(base + AT_SMEM_QK + kb * AT_TILE + r * 128 + ((((unsigned)c) ^ (r & 7u)) << 4)) =
                    make_float4(p[j] * inv, p[j + 1] * inv, p[j + 2] * inv, p[j + 3] * inv);
            }
    }
    fence_proxy_async_smem();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
#pragma unroll
            for (int vh = 0; vh < 2; vh++)
#pragma unroll
                for (int kb = 0; kb < 2; kb++) {
                    const unsigned long long pd = make_sw128_desc(sbase + AT_SMEM_QK + kb * AT_TILE);
                    const unsigned long long vd = make_sw128_desc(sbase + AT_SMEM_VT + (vh * 2 + kb) * AT_VT_TILE);
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        umma_tf32(tmem_base + 128u + (unsigned)(vh * 64), pd + (unsigned long long)(k * 2), vd + (unsigned long long)(k * 2), IDESC_O, (kb | k) ? 1u : 0u);
                }
            umma_commit(bar_mma);
        }
        __syncwarp();
    }
    mbar_wait(bar_mma, 1);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    {
        const int i = tid & 63;
        float* out = a.ctx[tw] + (row0 + i) * AT_H + (h0 + hh) * AT_DH;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            unsigned o[32];
            tmem_ld32(lane_addr + 128u + (unsigned)(hh * 64 + half * 32), o);
            if (i < S) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(out + half * 32 + j) =
                        make_float4(__uint_as_float(o[j]), __uint_as_float(o[j + 1]), __uint_as_float(o[j + 2]), __uint_as_float(o[j + 3]));
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256) : "memory");
}


// =================================================================================================
// fp32-accurate variant: bf16 (hi, lo) planes, three kind::f16 MMAs per contraction.  Same work split as above (two heads per CTA,
// thread r = row r), three 32 KB shared-memory regions that are reused as the data moves on, so that the CTA still needs only
// ~97 KB and TWO CTAs share an SM (one CTA is a serial latency chain: TMA -> convert -> MMA -> softmax -> MMA -> store):
//   R0: Q as fp32 (TMA landing, 2 k-block tiles)        -> K planes  [K_hi 16 KB | K_lo 16 KB]
//   R1: K as fp32 (TMA landing)                         -> V^T planes [h0 hi | h1 hi | h0 lo | h1 lo] (8 KB each)
//   R2: Q planes [Q_hi 16 KB | Q_lo 16 KB]              -> P planes  [P_hi | P_lo]
// A plane tile is [128 rows x 64 bf16] = 128-byte rows, SWIZZLE_128B, K-major: logical 16-byte chunk q of row r sits at
// r*128 + ((q ^ (r & 7)) << 4).  The fp32 -> planes conversion is done by the row's own thread (reads two fp32 chunks of the TMA tile,
// writes one bf16 chunk per plane); a quarter-warp touches 8 different chunk positions -> conflict-free.
// =================================================================================================
#define ATB_R0 0
#define ATB_R1 (32 * 1024)
#define ATB_R2 (64 * 1024)
#define ATB_TAIL (96 * 1024)
#define ATB_SMEM_BYTES (ATB_TAIL + 64 * 4 + 64 + 1024)
#define ATB_PLANE (16 * 1024)

// fp32 TMA tiles (2 k-blocks of [128 x 32 floats]) at `src` -> bf16 planes [128 x 64] at dst_hi / dst_lo, row r = this thread
__device__ __forceinline__ void atb_convert_rows(const unsigned char* src, unsigned char* dst_hi, unsigned char* dst_lo, unsigned r) {
#pragma unroll
    for (unsigned q = 0; q < 8; q++) {
        const unsigned kb = q >> 2, c0 = (q & 3u) * 2u;
        const float4 a = *reinterpret_cast<const float4*>(src + kb * AT_TILE + r * 128 + (((c0) ^ (r & 7u)) << 4));
        const float4 b = *reinterpret_cast<const float4*>(src + kb * AT_TILE + r * 128 + (((c0 + 1u) ^ (r & 7u)) << 4));
        uint4 h, l;
        bx_split2(a.x, a.y, h.x, l.x); bx_split2(a.z, a.w, h.y, l.y); bx_split2(b.x, b.y, h.z, l.z); bx_split2(b.z, b.w, h.w, l.w);
        const unsigned off = r * 128 + ((q ^ (r & 7u)) << 4);
        *reinterpret_cast<uint4*>(dst_hi + off) = h;
        *reinterpret_cast<uint4*>(dst_lo + off) = l;
    }
}
__device__ __forceinline__ void umma_bf16_at(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

__global__ void __launch_bounds__(128, 2) attention_tc_bx_kernel(const __grid_constant__ AttnTcMaps maps, const AttnTcArgs a) {
    extern __shared__ __align__(1024) unsigned char atsm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int hp = blockIdx.x, b = blockIdx.y, tw = blockIdx.z;
    const int S = a.S, h0 = hp * 2;
    unsigned char* base = (unsigned char*)((((unsigned long long)atsm) + 1023ull) & ~1023ull);
    const unsigned sbase = smem_u32(base);
    float* mb = reinterpret_cast<float*>(base + ATB_TAIL);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(base + ATB_TAIL + 256);
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(base + ATB_TAIL + 256 + 32);
    const unsigned bar_tma = smem_u32(bars), bar_mma = smem_u32(bars + 1);
    const CUtensorMap* map = &maps.qkv[tw];
    const long long row0 = (long long)b * S;

    if (tid == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
        mbar_init(bar_tma, 1); mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_base = *tmem_slot;

    if (tid == 0) {
        mbar_expect_tx(bar_tma, 4 * AT_TILE);
#pragma unroll
        for (int op = 0; op < 2; op++)              // 0: Q -> R0, 1: K -> R1
#pragma unroll
            for (int kb = 0; kb < 2; kb++)
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
                    tma_load_2d(sbase + (op ? ATB_R1 : ATB_R0) + kb * AT_TILE + hh * (64 * 128), map, op * AT_H + (h0 + hh) * AT_DH + kb * 32, (int)row0, bar_tma);
    }
    // V of this thread's (head, key) while the TMA is in flight: warp w -> head w>>1, keys 32(w&1) .. +31, lane = key
    const int vhh = warp >> 1, vj = (warp & 1) * 32 + lane;
    float4 vreg[16];
    {
        const bool ok = vj < S;
        const float4* src = reinterpret_cast<const float4*>(a.qkv[tw] + (row0 + vj) * (3 * AT_H) + 2 * AT_H + (h0 + vhh) * AT_DH);
#pragma unroll
        for (int d4 = 0; d4 < 16; d4++) vreg[d4] = ok ? __ldg(src + d4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (tid < 64) mb[tid] = (tid < S) ? (1.0f - (float)a.mask[row0 + tid]) * -10000.0f : 0.f;
    mbar_wait(bar_tma, 0);
    atb_convert_rows(base + ATB_R0, base + ATB_R2, base + ATB_R2 + ATB_PLANE, (unsigned)tid);            // Q: R0 -> R2
    __syncthreads();                                                                                       // every row of R0 has been read
    atb_convert_rows(base + ATB_R1, base + ATB_R0, base + ATB_R0 + ATB_PLANE, (unsigned)tid);            // K: R1 -> R0
    __syncthreads();                                                                                       // every row of R1 has been read
    {   // V^T planes into R1: element (d, key) of head hh at  hh*8K + d*128 + (((key >> 3) ^ (d & 7)) << 4) + (key & 7)*2
        unsigned char* vh = base + ATB_R1 + vhh * (8 * 1024);
        unsigned char* vl = vh + 16 * 1024;
        const unsigned kk = (unsigned)vj;
#pragma unroll
        for (int d4 = 0; d4 < 16; d4++) {
            const float e[4] = {vreg[d4].x, vreg[d4].y, vreg[d4].z, vreg[d4].w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const unsigned d = (unsigned)(d4 * 4 + t);
                const unsigned off = d * 128 + ((((kk >> 3) ^ (d & 7u)) << 4) | ((kk & 7u) << 1));
                const __nv_bfloat16 hb = __float2bfloat16_rn(e[t]);
                *reinterpret_cast<__nv_bfloat16*>(vh + off) = hb;
                *reinterpret_cast<__nv_bfloat16*>(vl + off) = __float2bfloat16_rn(e[t] - __bfloat162float(hb));
            }
        }
    }
    fence_proxy_async_smem();
    __syncthreads();

    // instruction descriptors: D = F32, A = B = BF16, both K-major
    constexpr unsigned IDESC_S = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    constexpr unsigned IDESC_O = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
    if (warp == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
            const unsigned long long qh = make_sw128_desc(sbase + ATB_R2), ql = make_sw128_desc(sbase + ATB_R2 + ATB_PLANE);
            const unsigned long long kh = make_sw128_desc(sbase + ATB_R0), kl = make_sw128_desc(sbase + ATB_R0 + ATB_PLANE);
#pragma unroll
            for (int k = 0; k < 4; k++) {           // UMMA_K = 16 bf16 = 32 bytes
                const unsigned long long ko = (unsigned long long)(k * 2);
                umma_bf16_at(tmem_base, qh + ko, kl + ko, IDESC_S, k ? 1u : 0u);
                umma_bf16_at(tmem_base, ql + ko, kh + ko, IDESC_S, 1u);
                umma_bf16_at(tmem_base, qh + ko, kh + ko, IDESC_S, 1u);
            }
            umma_commit(bar_mma);
        }
        __syncwarp();
    }
    mbar_wait(bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    const int hh = tid >> 6;
    const unsigned lane_addr = tmem_base + ((unsigned)(warp * 32) << 16);
    {
        unsigned s0[32], s1[32];
        tmem_ld32(lane_addr + (unsigned)(hh * 64), s0);
        tmem_ld32(lane_addr + (unsigned)(hh * 64 + 32), s1);
        float p[64];
        float mx = -3.0e38f;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            p[j] = __uint_as_float(s0[j]) * 0.125f + mb[j];
            p[j + 32] = __uint_as_float(s1[j]) * 0.125f + mb[j + 32];
        }
#pragma unroll
        for (int j = 0; j < 64; j++) if (j < S) mx = fmaxf(mx, p[j]);
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < 64; j++) { p[j] = (j < S) ? expf(p[j] - mx) : 0.f; sum += p[j]; }
        const float inv = 1.0f / sum;
        const unsigned r = (unsigned)tid;                  // P planes over the Q planes (S complete => the tensor core is done with Q and K)
#pragma unroll
        for (unsigned q = 0; q < 8; q++) {
            uint4 h, l;
            bx_split2(p[8 * q] * inv, p[8 * q + 1] * inv, h.x, l.x); bx_split2(p[8 * q + 2] * inv, p[8 * q + 3] * inv, h.y, l.y);
            bx_split2(p[8 * q + 4] * inv, p[8 * q + 5] * inv, h.z, l.z); bx_split2(p[8 * q + 6] * inv, p[8 * q + 7] * inv, h.w, l.w);
            const unsigned off = r * 128 + ((q ^ (r & 7u)) << 4);
            *reinterpret_cast<uint4*>(base + ATB_R2 + off) = h;
            *reinterpret_cast<uint4*>(base + ATB_R2 + ATB_PLANE + off) = l;
        }
    }
    fence_proxy_async_smem();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (lane == 0) {
            const unsigned long long ph = make_sw128_desc(sbase + ATB_R2), pl = make_sw128_desc(sbase + ATB_R2 + ATB_PLANE);
#pragma unroll
            for (int vh = 0; vh < 2; vh++) {
                const unsigned long long vhd = make_sw128_desc(sbase + ATB_R1 + vh * (8 * 1024)), vld = make_sw128_desc(sbase + ATB_R1 + 16 * 1024 + vh * (8 * 1024));
                const unsigned d_o = tmem_base + 128u + (unsigned)(vh * 64);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const unsigned long long ko = (unsigned long long)(k * 2);
                    umma_bf16_at(d_o, ph + ko, vld + ko, IDESC_O, k ? 1u : 0u);
                    umma_bf16_at(d_o, pl + ko, vhd + ko, IDESC_O, 1u);
                    umma_bf16_at(d_o, ph + ko, vhd + ko, IDESC_O, 1u);
                }
            }
            umma_commit(bar_mma);
        }
        __syncwarp();
    }
    mbar_wait(bar_mma, 1);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    {
        const int i = tid & 63;
        float* out = a.ctx[tw] + (row0 + i) * AT_H + (h0 + hh) * AT_DH;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            unsigned o[32];
            tmem_ld32(lane_addr + 128u + (unsigned)(hh * 64 + half * 32), o);
            if (i < S) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(out + half * 32 + j) =
                        make_float4(__uint_as_float(o[j]), __uint_as_float(o[j + 1]), __uint_as_float(o[j + 2]), __uint_as_float(o[j + 3]));
                if (a.ctx_hi[tw]) {               // the same row segment as (hi, lo) bf16 planes for the bf16x3 output projection
                    unsigned short* gh = a.ctx_hi[tw] + (row0 + i) * AT_H + (h0 + hh) * AT_DH + half * 32;
                    unsigned short* gl = a.ctx_lo[tw] + (row0 + i) * AT_H + (h0 + hh) * AT_DH + half * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint4 h, l;
                        bx_split2(__uint_as_float(o[j]), __uint_as_float(o[j + 1]), h.x, l.x); bx_split2(__uint_as_float(o[j + 2]), __uint_as_float(o[j + 3]), h.y, l.y);
                        bx_split2(__uint_as_float(o[j + 4]), __uint_as_float(o[j + 5]), h.z, l.z); bx_split2(__uint_as_float(o[j + 6]), __uint_as_float(o[j + 7]), h.w, l.w);
                        *reinterpret_cast<uint4*>(gh + j) = h;
                        *reinterpret_cast<uint4*>(gl + j) = l;
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256) : "memory");
}

// qkv[t]: [T, 2304] fp32 (Q | K | V, heads contiguous inside each), ctx[t]: [T, 768]; mask int64 [B, S]; S <= 64, 12 heads;
// towers t < ntw (blockIdx.z).
int dph_launch_attention_tc(const float* const qkv[2], float* const ctx[2], const long long* mask, int B, int S, long long T, cudaStream_t st, int split,
                            unsigned short* const* ctx_hi, unsigned short* const* ctx_lo, int ntw) {
    DPH_CHECK(S >= 1 && S <= 64 && B >= 1 && T >= (long long)B * S, "attention_tc: S must be 1..64");
    DPH_CHECK(ntw == 1 || ntw == 2, "attention_tc: one or two towers");
    static DphPerDeviceOnce once;
    if (once.first()) {
        DPH_CUDA(cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BYTES));
        DPH_CUDA(cudaFuncSetAttribute(attention_tc_bx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM_BYTES));
    }
    AttnTcMaps maps = {};
    AttnTcArgs a = {};
    for (int t = 0; t < ntw; t++) {
        DPH_TRY(dph_make_map_f32(&maps.qkv[t], qkv[t], T, 3 * AT_H, 3 * AT_H, 64));
        a.qkv[t] = qkv[t]; a.ctx[t] = ctx[t];
        a.ctx_hi[t] = ctx_hi ? ctx_hi[t] : nullptr; a.ctx_lo[t] = ctx_lo ? ctx_lo[t] : nullptr;
    }
    a.mask = mask; a.S = S;
    if (split) attention_tc_bx_kernel<<<dim3(6, (unsigned)B, (unsigned)ntw), 128, ATB_SMEM_BYTES, st>>>(maps, a);
    else attention_tc_kernel<<<dim3(6, (unsigned)B, (unsigned)ntw), 128, AT_SMEM_BYTES, st>>>(maps, a);
    DPH_CUDA(cudaGetLastError());
    return 0;
}
