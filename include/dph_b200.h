/*
 * dph_b200.h -- C ABI of libdph_b200.so: the B200-native replacement for the FAISS calls on the
 * DensePhrases retrieval hot path.  Plain pointers and sizes only (no torch / faiss types).
 *
 * Every entry point names the reference interface it replaces (paths relative to /root/reference):
 *
 *   dph_index_search            <- faiss.IndexPreTransform.search(x, k)      densephrases/index.py:200
 *   dph_index_reconstruct_batch <- faiss IndexIVFPQ.reconstruct(id) per id   densephrases/index.py:31,282-300
 *   dph_index_get_opq           <- faiss.vector_to_array(OPQMatrix.A)        densephrases/index.py:32
 *   dph_index_ntotal/d/nlist    <- index.ntotal / index.d / index_ivf.nlist  densephrases/index.py:33,128-133
 *   dph_index_set_nprobe        <- index_ivf.nprobe = 256                    densephrases/index.py:53,62
 *   dph_index_create/set_*      <- faiss.read_index(...) / IndexPreTransform(OPQMatrix, IndexIVFPQ(...))
 *                                  densephrases/index.py:30 ; build_phrase_index.py:113-116,149-150
 *
 * Conventions: every function returns 0 on success, non-zero on error (dph_last_error() gives the
 * message; the Python layer raises RuntimeError like faiss' SWIG layer does).  `mem` arguments say
 * where caller buffers live.  All device work is issued on the stream passed to dph_index_set_stream
 * (default: the legacy default stream).  Calls with host buffers are synchronous; calls with device
 * buffers are asynchronous on that stream.  Inputs are never modified.
 */
#ifndef DPH_B200_H
#define DPH_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define DPH_MEM_HOST 0
#define DPH_MEM_DEVICE 1

/* scan kernel selection (dph_index_set_scan_mode) */
#define DPH_SCAN_FAST 0   /* default: conflict-free gather filter + proof + exact fp32 re-scoring; picks QUAD / PAIR / SINGLE per batch */
#define DPH_SCAN_EXACT 1  /* canonical-order fp32 ADC for every code (slow; fallback + cross-check) */
#define DPH_SCAN_PAIR 2   /* force: two queries share every gather (int16-packed quantised LUTs), lists grouped by probing queries */
#define DPH_SCAN_SINGLE 3 /* force: one query per gather (fp32 LUT) */
#define DPH_SCAN_QUAD 4   /* force: four queries share every gather (int8-packed quantised LUTs), lists grouped by probing queries */

typedef struct dph_index dph_index;

const char* dph_last_error(void);
int dph_version(void);

/* ---- construction (replaces faiss.read_index / index build; build_phrase_index.py:113-116) ---- */
/* d = M*dsub, nbits must be 8 (ksub 256), M must be 96 (PQ96: code row = 96 bytes). */
int dph_index_create(dph_index** out, int d, int64_t nlist, int M, int nbits, int device);
void dph_index_free(dph_index* ix);
int dph_index_set_stream(dph_index* ix, void* cuda_stream);
/* OPQ matrix A [d,d] row-major (d_out rows), centroids [nlist,d], PQ codebooks [M,256,dsub]; fp32. */
int dph_index_set_opq(dph_index* ix, const float* A, int mem);
int dph_index_set_centroids(dph_index* ix, const float* C, int mem);
int dph_index_set_pq(dph_index* ix, const float* pq, int mem);
/* Synthetic centroids/PQ (bit-identical to oracle ref_gen_centroids / ref_gen_pq), generated on device. */
int dph_index_gen_centroids(dph_index* ix, uint64_t seed, float sigma);
int dph_index_gen_pq(dph_index* ix, uint64_t seed, float sigma);
/* This process holds only inverted lists [list_lo, list_hi) (list-range shard, SURVEY 8e). Call before set_lists. */
int dph_index_set_shard(dph_index* ix, int64_t list_lo, int64_t list_hi);
/* list_len [nlist] (ALL lists, host). codes: [ntotal,96] list-major rows of the lists in the shard only
 * (host), ids likewise [ntotal_shard] or NULL for sequential labels (label = global list-major row,
 * build_phrase_index.py:149-150). */
int dph_index_set_lists(dph_index* ix, const int64_t* list_len, const uint8_t* codes, const int64_t* ids);
/* Same but codes are generated on device from `seed` (bit-identical to oracle ref_gen_codes); ids sequential. */
int dph_index_set_lists_synthetic(dph_index* ix, const int64_t* list_len, uint64_t seed);

/* ---- getters ---- */
int64_t dph_index_ntotal(const dph_index* ix);       /* all shards */
int64_t dph_index_ntotal_local(const dph_index* ix); /* this shard */
int dph_index_d(const dph_index* ix);
int64_t dph_index_nlist(const dph_index* ix);
int dph_index_nprobe(const dph_index* ix);
int dph_index_set_nprobe(dph_index* ix, int nprobe);
int dph_index_set_scan_mode(dph_index* ix, int mode);
/* Coarse quantizer on the tensor cores (3xTF32 candidate pass + exact sequential-FMA re-rank + proof; bit-identical probes).
 * 1 (default): used when the shape allows (lists % 128 == 0, batch >= 32, nprobe + margin <= 1024); 0: always the exact SIMT GEMM. */
int dph_index_set_coarse_tc(dph_index* ix, int on);
int dph_index_get_opq(const dph_index* ix, float* A_out, int mem);
int64_t dph_index_device_bytes(const dph_index* ix);
/* Measurement hook: when on, CUDA events bracket the scan kernel of each search (last chunk); last_scan_ms waits
 * for it and returns the kernel's duration in milliseconds (bench.py roofline). */
int dph_index_set_profile(dph_index* ix, int on);
int dph_index_last_scan_ms(dph_index* ix, float* ms);
/* Durations of the scan kernels of the last (up to 64) searches since profiling was switched on, oldest first;
 * dph_index_profile_count gives how many.  Lets bench.py time the kernel inside a back-to-back step loop. */
int dph_index_profile_scan_ms(dph_index* ix, float* ms_out, int max_out);
int dph_index_profile_count(const dph_index* ix);

/* ---- search (replaces index.search at index.py:200) ----
 * x [n,d] fp32; D [n,k] fp32, I [n,k] int64 labels; sorted by descending score; unfilled slots are
 * (-FLT_MAX, -1) like faiss' CMin heap.  Uses the index's nprobe (default 256, index.py:53,62). */
int dph_index_search(dph_index* ix, const float* x, int64_t n, int k, float* D, int64_t* I, int mem);
/* Sharded search: per-shard partial top-k.  G [n,k] uint32 = canonical scan position (tie-break key,
 * global over all shards).  Buffers on device.  After an all-gather over shards feed dph_merge_shards. */
int dph_index_search_partial(dph_index* ix, const float* x_dev, int64_t n, int k, float* D_dev, int64_t* I_dev,
                             uint32_t* G_dev);
/* Sharded coarse quantizer (scales the IndexFlatIP coarse search with the number of shards): every shard scores only its own
 * lists' centroids and emits its best nprobe as keys (score key << 32 | ~global list id, 0 = empty) [n,nprobe];
 * after an all-gather of the keys [nshards,n,nprobe], search_preassigned merges them into the global top-nprobe (identical to
 * the unsharded selection) and runs the rest of the search on this shard's lists.  n must fit one chunk (<= 4096). */
int dph_index_coarse_local(dph_index* ix, const float* x_dev, int64_t n, uint64_t* keys_dev);
int dph_index_search_preassigned(dph_index* ix, const uint64_t* keys_gathered_dev, int nshards, int64_t n, int k, float* D_dev,
                                 int64_t* I_dev, uint32_t* G_dev);
/* Query-split variant of the same step (large batches): every shard rotates and assigns only ITS SLICE of the batch (n_local queries),
 * but over ALL lists (the coarse quantizer is replicated, index.py:200 runs it once per batch), and emits one record per query:
 * rec [n_local, dph_index_record_floats()] = [768 f32 rotated query | nprobe i32 list numbers | nprobe f32 coarse scores].  After an
 * all-gather of the records, search_assigned (rec [n, ...], all queries in batch order) runs the rest of the search on this shard's
 * lists.  Same probes and scores as the unsharded search; the rotation and the exact re-rank of the tensor-core coarse quantizer are
 * done once per query instead of once per query and shard.  Records and candidate keys are an exchange format between ranks running
 * THIS library on replicas of the same coarse quantizer: list numbers inside them are trusted, not validated (a caller that
 * fabricates them must keep them in [-1, nlist)). */
int dph_index_record_floats(const dph_index* ix);
int dph_index_coarse_split(dph_index* ix, const float* x_dev, int64_t n_local, float* rec_dev);
int dph_index_search_assigned(dph_index* ix, const float* rec_dev, int64_t n, int k, float* D_dev, int64_t* I_dev, uint32_t* G_dev);
/* Dg/Ig/Gg [nshards,n,k] (all-gathered, device) -> D/I [n,k] (device).  Order: score desc, scan position asc. */
int dph_merge_shards(const float* Dg, const int64_t* Ig, const uint32_t* Gg, int nshards, int64_t n, int k, float* D,
                     int64_t* I, void* cuda_stream);
/* Same exchange as ONE buffer: pack (D, I, G) [n,k] into P [n,k,2] int64 = {candidate key (score, scan position), label};
 * all-gather P; merge Pg [nshards,n,k,2] -> D/I [n,k]. */
int dph_pack_topk(const float* D, const int64_t* I, const uint32_t* G, int64_t n, int k, int64_t* P, void* cuda_stream);
int dph_merge_shards_packed(const int64_t* Pg, int nshards, int64_t n, int k, float* D, int64_t* I, void* cuda_stream);
/* Per-query flags of the last search (device pointer, int32 [n]): bit0 = fast filter could not prove
 * exactness and the query was re-run through the exact kernel. */
const int32_t* dph_index_last_flags(const dph_index* ix);
/* Intermediate results of the last search, for tests (device pointers): probed lists [n,nprobe] int32,
 * coarse scores [n,nprobe] fp32, rotated queries [n,d]. */
const int32_t* dph_index_last_probes(const dph_index* ix);
const float* dph_index_last_coarse(const dph_index* ix);
const float* dph_index_last_xr(const dph_index* ix);
int dph_index_last_used_pair_mode(const dph_index* ix);   /* 1 when the last search shared gathers between queries (pair or quad) */
int dph_index_last_group_size(const dph_index* ix);       /* queries per gather of the last search: 1, 2 or 4 */
/* Copy one of them to the host (synchronises): which = 0 flags, 1 probes, 2 coarse scores, 3 rotated queries. */
int dph_index_copy_last(dph_index* ix, int which, void* dst_host, int64_t bytes);

/* ---- reconstruct (replaces reconst_fn loop, index.py:282-300) ----
 * out [m,d] fp32 in ROTATED space (caller un-rotates with R = OPQ matrix, index.py:340,365);
 * found [m] u8: 0 -> label not in this shard / not in the index, row is zeros (index.py:287-288). */
int dph_index_reconstruct_batch(dph_index* ix, const int64_t* ids, int64_t m, float* out, uint8_t* found, int mem);

/* ---- phrase re-scoring (replaces index.py:323-371: end.matmul(R); (q*end).sum; argmax with mask) ----
 * For each of m hits: window of L consecutive labels starting at first_id[i]; score[i,l] =
 * <q[i], R^T-unrotated reconstruct(first_id[i]+l)> computed as <A q[i] , reconstruct> (A orthonormal);
 * out_scores [m,L] fp32 (missing label -> 0, like the zero vector at index.py:287-288). */
int dph_index_window_scores(dph_index* ix, const float* q /*[m,d]*/, const int64_t* first_id /*[m]*/, int64_t m, int L,
                            float* out_scores, int mem);

/* ---- encoder (replaces Encoder.forward(return_query=True) -> embed_query, densephrases/encoder.py:146-152,101-118, and
 * Encoder.forward(input_ids=..., return_phrase=True) -> embed_phrase + filter_linear, encoder.py:92-99,130-144) ----
 * BERT-base towers (12 layers, 768 hidden, 12 heads, 3072 FFN; SpanBERT-base-cased geometry, options.py:23).  tower 0 =
 * query_start_encoder.*, tower 1 = query_end_encoder.*, tower 2 = phrase_encoder.* (encoder.py:50-52); each is allocated only when
 * loaded.  Weight blob layout: encoder.cu. */
typedef struct dph_encoder dph_encoder;
int dph_encoder_create(dph_encoder** out, int device, int vocab_size, int max_position_embeddings, int type_vocab_size);
void dph_encoder_free(dph_encoder* e);
int dph_encoder_set_stream(dph_encoder* e, void* cuda_stream);
int64_t dph_encoder_tower_floats(const dph_encoder* e);
int dph_encoder_load_tower(dph_encoder* e, int tower, const float* blob, int mem);
/* filter_linear (encoder.py:32): W fp32 [2,768] (row 0: start logit, row 1: end logit), b fp32 [2]. */
int dph_encoder_load_filter(dph_encoder* e, const float* W, const float* b, int mem);
/* 0 (default): GEMMs as one TF32 MMA per product -- what torch 1.9 (the reference's pin) does for fp32 matmuls on Ampere+;
 * 1: 3xTF32 split GEMMs, fp32-accurate (matches the reference's CPU/fp32 path to ~1e-5);
 * 2: bf16x3 split GEMMs (operands as (hi, lo) bf16 planes, three kind::f16 MMAs per product, ~2^-17 relative): meets the 1e-3
 *    tolerance on the query vectors at the speed of mode 0. */
int dph_encoder_set_precision(dph_encoder* e, int precise);
/* 1 (default): self-attention of sequences with S <= 64 (and, in the phrase forward, 64 < S <= 512) on the tensor cores -- TF32
 * operands in precision mode 0, bf16 (hi, lo) planes with three MMAs per contraction (fp32-accurate) in modes 1 and 2; fp32
 * accumulation and softmax.  0: always the fp32 SIMT attention kernels (S <= 384). */
int dph_encoder_set_attention(dph_encoder* e, int tensor_core);
/* One BERT-base self-attention (12 heads x 64; HF BertSelfAttention as used by encoder.py:101-118) on device buffers:
 * qkv fp32 [B*S, 2304] = (Q | K | V), mask int64 [B,S] -> ctx fp32 [B*S, 768].  tensor_core: 0 SIMT fp32 (S <= 384),
 * 1 tcgen05 TF32, 2 tcgen05 on bf16 (hi, lo) operand planes, three MMAs per contraction (fp32-accurate); 1 and 2: S <= 512 (S > 64
 * runs the long-sequence kernel with an online softmax over key tiles). */
int dph_attention_bert(const float* qkv, const int64_t* attention_mask, int B, int S, float* ctx, int tensor_core, void* cuda_stream);
/* input_ids / attention_mask / token_type_ids int64 [B,S] (S <= 384); start_out / end_out fp32 [B,768] = hidden state at
 * position 0 of each tower (the reference returns them as [B,1,768]). */
int dph_encoder_embed_query(dph_encoder* e, const int64_t* input_ids, const int64_t* attention_mask, const int64_t* token_type_ids,
                            int B, int S, float* start_out, float* end_out, int mem);
/* Phrase tower over every token: input_ids / attention_mask / token_type_ids int64 [B,S], 1 <= S <= min(512, max_position_embeddings).
 * out fp32 [B,S,768] (nullable) = the last hidden state (start == end in the reference); filter_start / filter_end fp32 [B,S] =
 * filter_linear logits; out_q int8 [B,S,768] (nullable) = float_to_int8(out, dense_offset, dense_scale) (embed_utils.py:141-145:
 * fp32 (x - offset) * scale, clamped to [-128, 127], rounded half to even).  Needs tower 2 and the filter head.  Buffers and the
 * out-of-range id flag follow dph_encoder_embed_query. */
int dph_encoder_embed_phrase(dph_encoder* e, const int64_t* input_ids, const int64_t* attention_mask, const int64_t* token_type_ids,
                             int B, int S, float* out, float* filter_start, float* filter_end, int8_t* out_q, float dense_offset,
                             float dense_scale, int mem);

/* ---- exact sequential-k fp32 GEMM (the inner-product definition shared with the oracle): out [n,m] = X [n,K] . W [m,K]^T,
 * acc = fmaf(x[t], w[t], acc) for t ascending; device pointers; K % 32 == 0.  Used for the OPQ rotation and the coarse quantizer. */
int dph_sgemm_nt_seq(const float* X, int64_t n, const float* W, int64_t m, int64_t K, float* out, void* cuda_stream);

/* ---- dense fp32 GEMM on the tcgen05 tensor cores (kind::tf32), the encoder's building block ----
 * out [M,N] = act(A [M,K] . W [N,K]^T + bias [N]) + residual [M,N]; act: 0 none, 1 erf-GELU; device pointers;
 * N % 128 == 0, K % 32 == 0.  == torch.nn.functional.linear (HF BertSelfAttention/BertOutput/BertIntermediate). */
int dph_gemm_tf32_nt(const float* A, const float* W, const float* bias, const float* residual, float* out, int64_t M, int64_t N,
                     int64_t K, int act, int precise /* 0: 1xTF32, 1: 3xTF32 split (fp32-accurate), 2: bf16x3 split (N % 256 == 0) */,
                     void* cuda_stream);
/* Scheduling of the 1xTF32 GEMMs (process-wide; every mode issues the same MMAs in the same order -> bit-identical results):
 * 0: one 128x128 tile per CTA, two CTAs per SM;  1: the same as 2-CTA thread-block clusters sharing the A tile through TMA
 * multicast (N/128 even);  2 (default): persistent CTAs walking 128x256 tiles with double-buffered TMEM accumulators and twelve
 * epilogue warps (N % 256 == 0, else mode 0). */
int dph_gemm_tf32_set_mode(int mode);
/* Measurement hook (process-wide): choose between kernel variants that compute bit-identical results, for A/B timing on hardware
 * (tools/bench_variants.py).  knob 0: additions of the quad scan issued on the FMA pipe (0 none .. 3 all; default 1);
 * knob 1: tile shape of the sequential-k SGEMM (0 auto, 1: 128x128, 2: 64x64, 3: 32x64, 4: 16x64);
 * knob 2: shape of the PQ-table kernel (default: 4 queries x 32 sub-quantizers per CTA; 2: 8 x 16). */
int dph_set_tuning(int knob, int value);

#ifdef __cplusplus
}
#endif
#endif
