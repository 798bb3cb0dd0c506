/* chatts_b200 -- C-ABI of the B200 (sm_100a) hot path of ChatTS.
 *
 * The reference (NetManAIOps/ChatTS @ 09fae34) has NO native boundary for this path: it is Python on
 * top of torch / vLLM / transformers.  This header is the boundary a maintainer binds from Python with
 * ctypes (see INTEGRATION.md); each entry point names the reference code it replaces (file:line relative
 * to the reference repo, or the third-party file the reference calls).
 *
 * Conventions
 *   - every function returns int: 0 = CTS_OK, negative = error; cts_last_error(ctx) holds the message.
 *   - the caller owns ALL device memory (plain device pointers + explicit sizes); the library owns nothing
 *     but the ctx.  No hidden allocation, no hidden synchronisation, every launch takes a cudaStream_t
 *     (passed as void*).  Launches are CUDA-graph capturable.
 *   - one host thread per ctx; distinct ctxs are independent.
 *   - `dtype` is the model dtype of activations and weights: CTS_BF16 or CTS_F16 (fp32 accumulate).
 *   - there is NO CPU implementation behind any of these symbols.
 */
#ifndef CHATTS_B200_H
#define CHATTS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define CTS_OK 0
#define CTS_ERR_BAD_ARG (-1)
#define CTS_ERR_UNSUPPORTED (-2)
#define CTS_ERR_CUDA (-3)
#define CTS_ERR_NCCL (-4)

#define CTS_BF16 0
#define CTS_F16 1

typedef struct cts_ctx cts_ctx;

/* library identity: cts_arch() must say "sm_100a". */
int cts_version(void);
const char* cts_arch(void);

int cts_ctx_create(int device, cts_ctx** out);
void cts_ctx_destroy(cts_ctx* ctx);
const char* cts_last_error(const cts_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * A3  mask -> valid length -> patch count            chatts/vllm/chatts_vllm.py:94-100 and :198-207
 *   x            [n_series, row_len] model dtype; row_len = num_features * Lmax, interleaved
 *                (value, mask) pairs as produced by sp_encoding (encoding_utils.py:35), zero padded
 *                (chatts_vllm.py:517-529).
 *   valid_len    int32[n_series]   = sum(long(mask))
 *   patch_cnt    int32[n_series]   = ceil(valid_len / patch_size)
 *   row_offset   int32[n_series+1] = exclusive prefix sum of patch_cnt (row order of :187)
 *   max_valid    int32[1]          = max(valid_len)   (needed by use_position_idx, :146)
 */
int cts_ts_patch_count(cts_ctx* ctx, const void* x, int dtype, int n_series, int row_len, int num_features,
                       int patch_size, int* valid_len, int* patch_cnt, int* row_offset, int* max_valid,
                       void* stream);

/* A4+A5  patchify + last-value pad + position features   chatts/vllm/chatts_vllm.py:107-183
 *   mode: 0 = values only (:157), 1 = use_position_embedding (:135-142,161-183), 2 = use_position_idx (:143-154)
 *   pos_table    [max_seq_len+1, emb_dim] model dtype (mode 1), padding id = max_seq_len (:76,128)
 *   rows_out     [total_rows, in0] model dtype, in0 = patch (mode 0) | patch*(1+emb_dim) (1) | 2*patch (2)
 *   max_patches  grid bound: ceil(Lmax / patch_size)
 */
int cts_ts_patchify(cts_ctx* ctx, const void* x, int dtype, int n_series, int row_len, int num_features,
                    int patch_size, int mode, const void* pos_table, int emb_dim, int max_seq_len,
                    const int* valid_len, const int* row_offset, const int* max_valid, int max_patches,
                    void* rows_out, int in0, void* stream);

/* ------------------------------------------------------------------------------------------------
 * tcgen05 GEMM  Y[T, N] = X[T, K] * W[N, K]^T  (+ fused epilogue)
 *   replaces nn.Linear in  TimeSeriesEmbedding.mlp (chatts_vllm.py:83-91,188) and every projection of the
 *   decoder (transformers qwen2/modeling_qwen2.py:44-48,217-219,245; vllm qwen2.py:93-116,159-174;
 *   lm_head chatts_vllm.py:607-610).
 *   Weights stream through TMA as the 128-row MMA operand, tokens are the MMA N dimension ("swap-AB"), so
 *   decode batches of 1..32 tokens still issue full-width tcgen05.mma and the kernel is HBM-bound on W.
 */
#define CTS_EPI_NONE 0        /* out = dtype(acc + bias)                                      */
#define CTS_EPI_GELU 1        /* out = dtype(gelu_erf(dtype(acc + bias)))      chatts_vllm.py:86-87 */
#define CTS_EPI_SWIGLU 2      /* out = dtype(silu(dtype(acc_w)) * dtype(acc_w2))  modeling_qwen2.py:47 */
#define CTS_EPI_PARTIAL_F32 3 /* out_f32[split][t][n] = acc   (split-K; reduced by a cts_reduce_* call) */
#define CTS_EPI_RESIDUAL 4    /* out = dtype(residual + dtype(acc + bias))     modeling_qwen2.py:302,308 */
#define CTS_EPI_SWIGLU_IL 6   /* gate_up weights INTERLEAVED per 128-row tile (64 gate rows, then the 64 matching up rows):
                                 out[t][i] = dtype(silu(dtype(gate_i)) * dtype(up_i)), out has n/2 columns; t > 128 only */
#define CTS_EPI_SPLITK_F32 5  /* out_f32[t][n] = acc summed over the splits INSIDE the kernel: each split writes its partial to
                                 splitk_ws, the last split of a tile to arrive (tile_counters) adds them in split order */

typedef struct {
  const void* w;        /* [n, k] row-major, leading dimension w_ld elements */
  const void* w2;       /* second weight (up_proj) for CTS_EPI_SWIGLU, same shape/ld, else NULL */
  const void* x;        /* [t, k] row-major, leading dimension x_ld */
  const void* bias;     /* [n] model dtype or NULL */
  const void* residual; /* [t, n] (leading dimension out_ld) for CTS_EPI_RESIDUAL; may alias out */
  void* out;            /* [t, n] model dtype, or fp32 [split_k, t, n] for CTS_EPI_PARTIAL_F32 */
  const int* row_map;   /* optional: output row of token i is row_map[i] (<0: dropped) -- the sp-mask scatter
                           of patch rows into the embedding sequence (chatts_vllm.py:569-573) */
  long long n, k, t;
  long long w_ld, x_ld, out_ld;
  int dtype;
  int epilogue;
  int split_k;          /* >=1; >1 only with CTS_EPI_PARTIAL_F32 / CTS_EPI_SPLITK_F32 */
  int reserved;
  void* splitk_ws;      /* CTS_EPI_SPLITK_F32, split_k > 1: fp32 [split_k, t, n] scratch */
  int* tile_counters;   /* CTS_EPI_SPLITK_F32, split_k > 1: int32 [ceil(n/128) * ceil(t/BN)] zero-filled once (self-resetting) */
  /* Optional hint (decode-sized t only): the weight the NEXT weight-streaming GEMM of the chain will read.  A CTA whose own last
   * weight tile has been requested prefetches a share of that matrix into L2 (the first K blocks of every (128-row tile, K split)
   * unit of the next launch, next_prefetch_bytes in total), so HBM keeps streaming through this kernel's drain, the kernel
   * boundary and the small dependent kernel in between instead of idling (csrc/trace.cuh timeline).  NULL / 0 = no hint. */
  const void* next_w;   /* [next_n, next_k] row-major, leading dimension next_ld, same dtype */
  long long next_n, next_k, next_ld;
  int next_split;       /* split_k of the next launch (its K ranges decide which blocks it reads first) */
  int next_reserved;
  long long next_prefetch_bytes;
} cts_gemm_args;

int cts_gemm(cts_ctx* ctx, const cts_gemm_args* args, void* stream);
/* heuristic used by the host code: split-K factor that fills the SMs for a weight-streaming GEMM */
int cts_gemm_suggest_split(cts_ctx* ctx, long long n, long long k, long long t, int dual);

/* split-K reduction fused with the op that follows the projection ------------------------------- */

/* out[row_map?][n] = act(dtype(sum_s partial[s][t][n] + bias[n]))   act: CTS_EPI_NONE | CTS_EPI_GELU
 * (TS-encoder MLP layers, chatts_vllm.py:83-91; last layer scatters through row_map, :569-573) */
int cts_reduce_bias_act(cts_ctx* ctx, const float* partial, int split_k, long long t, long long n,
                        const void* bias, int act, void* out, long long out_ld, const int* row_map, int dtype,
                        void* stream);

/* h = resid_in + dtype(sum_s partial[s]) ; resid_out = h ; norm_out = w * dtype(h * rsqrt(mean(h^2)+eps))
 * (modeling_qwen2.py:258-263 RMSNorm, :302/:308 residual adds).  partial may be NULL (split_k = 0): plain
 * RMSNorm of resid_in.  norm_w may be NULL: only the residual update.  resid_out may alias resid_in. */
int cts_reduce_residual_rmsnorm(cts_ctx* ctx, const float* partial, int split_k, const void* resid_in,
                                void* resid_out, const void* norm_w, float eps, void* norm_out, long long t,
                                long long h, int dtype, void* stream);

/* out[t][i] = dtype(silu(dtype(sum_s p[s][t][g(i)])) * dtype(sum_s p[s][t][u(i)]))   (modeling_qwen2.py:47)
 * stacked layout: g(i) = i, u(i) = inter + i;  interleaved (CTS_EPI_SWIGLU_IL weights): g(i) = (i/64)*128 + i%64, u = g + 64 */
int cts_reduce_swiglu(cts_ctx* ctx, const float* partial, int split_k, long long t, long long inter, void* out,
                      int interleaved, int dtype, void* stream);

/* q/k/v = dtype(sum_s partial + bias); RoPE(q,k) with the fp32-computed cos/sin tables cast to dtype
 * (modeling_qwen2.py:107-146,217-222); q -> q_out [t, nh*d]; k,v -> paged KV cache slot slot_map[t]
 * (vllm Attention KV write, qwen2.py:233-235) and, when k_out/v_out != NULL, contiguous [t, nkv*d] copies
 * for the prefill attention.
 *   src: fp32 [split_k, t, (nh+2nkv)*d] when src_is_partial, else model-dtype [t, (nh+2nkv)*d] (bias already in)
 *   cos/sin: [max_pos, d/2] model dtype;  positions int32[t];  slot_map int32[t] (<0: no cache write)
 *   cache layout: [num_pages, nkv, page_size, d]
 *   q_norm_w / k_norm_w [d] (or NULL): Qwen3 / ChatTS-8B per-head RMSNorm of q and k before RoPE
 *   (chatts_vllm.py:633-668 selects Qwen3ForCausalLM; transformers qwen3/modeling_qwen3.py), eps = norm_eps
 */
int cts_qkv_rope_cache(cts_ctx* ctx, const void* src, int src_is_partial, int split_k, const void* bias,
                       const int* positions, const void* cos_tab, const void* sin_tab, const int* slot_map,
                       void* q_out, void* k_cache, void* v_cache, void* k_out, void* v_out, long long t, int nh,
                       int nkv, int head_dim, int page_size, const void* q_norm_w, const void* k_norm_w, float norm_eps,
                       int dtype, void* stream);

/* K4  embedding lookup: out[i] = table[ids[i]] for ids[i] >= 0 (rows with id < 0 are left untouched:
 * they are the patch rows the TS encoder scatters)            chatts_vllm.py:569 */
int cts_embed_gather(cts_ctx* ctx, const void* table, const int* ids, void* out, long long t, long long h,
                     long long vocab, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K8 attention                       modeling_qwen2.py:161-184 ; vllm qwen2.py:188-197,234
 * prefill: causal GQA over the tokens of this call, variable length, cu_seqlens int32[batch+1]
 *   q [t, nh, d], k/v [t, nkv, d] (RoPE applied), out [t, nh*d]; total_tokens = t (rows of q/k/v; bounds the TMA maps)
 *   head_dim 128: tcgen05 kernel (TMA-staged Q/K/V, S and O accumulators in TMEM); head_dim 64: HMMA (wmma) kernel
 */
int cts_attn_prefill(cts_ctx* ctx, const void* q, const void* k, const void* v, const int* cu_seqlens, int batch,
                     int max_seqlen, long long total_tokens, int nh, int nkv, int head_dim, float scale, void* out,
                     int dtype, void* stream);

/* decode: one query token per sequence against the paged cache (flash-decoding split over KV tiles of 64 tokens;
 * pages are staged by TMA with the 128-byte swizzle, QK^T and PV run on mma.sync, the last split to finish merges).
 *   q [batch, nh, d]; k_cache/v_cache [num_pages, nkv, page_size, d]; page_table int32[batch, max_pages];
 *   seq_lens int32[batch] (tokens incl. the current one); out [batch, nh*d]
 *   workspace: fp32, cts_attn_decode_workspace_floats(...) elements, ZERO-FILLED ONCE by the caller (it holds the
 *   self-resetting arrival counters after the partials)
 * Preconditions:
 *   - the kernel this one follows on the stream (its programmatic-dependent-launch predecessor) may write only q and row
 *     seq_len - 1 of each sequence's K and V: the KV tiles before the one holding that row are loaded ahead of the dependency
 *     wait, and seq_lens / page_table are read there too, so they must not change inside the step either;
 *   - every cache row past seq_len that a sequence's last 64-token tile covers (the rest of its last page and the pages the
 *     table lists after it) must hold finite values: masked keys get probability 0, and 0 times a non-finite value is NaN.
 */
long long cts_attn_decode_workspace_floats(int batch, int nh, int head_dim, int num_splits);
int cts_attn_decode(cts_ctx* ctx, const void* q, const void* k_cache, const void* v_cache, int num_pages,
                    const int* page_table, int max_pages, const int* seq_lens, int batch, int nh, int nkv, int head_dim,
                    int page_size, float scale, int num_splits, float* workspace, void* out, int dtype, void* stream);

/* K13 greedy sampling + device-side bookkeeping of the decode loop, so that a whole step
 * (embed -> 48 layers -> lm_head -> argmax -> advance) replays as one CUDA graph with no host round trip
 * (HF GenerationMixin greedy loop, README.md:102; vLLM sampler).
 *   logits [batch, vocab] model dtype -> next id (first max, like torch.argmax)
 *   out_tokens int32[batch, out_ld] column `*step_ptr` receives the id; cur_ids int32[batch] = id;
 *   positions[b] += 1; seq_lens[b] += 1; slot_map[b] = slot of the NEW position in the paged cache;
 *   step_ptr int32[2] = {step, arrival counter}: step += 1 once every sequence has been processed (device counter).
 */
int cts_greedy_advance(cts_ctx* ctx, const void* logits, long long vocab, int batch, int* out_tokens, int out_ld,
                       int* step_ptr, int* cur_ids, int* positions, int* seq_lens, int* slot_map,
                       const int* page_table, int max_pages, int page_size, int dtype, void* stream);

/* K13, sampled variant: temperature -> top-k -> top-p -> multinomial (transformers TemperatureLogitsWarper / TopKLogitsWarper /
 * TopPLogitsWarper + torch.multinomial; vLLM Sampler -- chatts/utils/inference_tsmllm_deepspeed.py:95-100 decodes with
 * temperature 0.2, chatts/utils/llm_utils.py:166-170 passes temperature / top_p) fused with the same device-side advance as
 * cts_greedy_advance, so a sampled decode step needs no host round trip either.
 *   kept set = {i : z_i >= tau}, z = logits / temperature; tau by bisection over the 16-bit ordered key of the logit (no sort):
 *   top_k > 0: the k largest (ties at the k-th value kept); 0 < top_p < 1: the smallest threshold set whose probability reaches
 *   top_p of the top-k mass.  The token is drawn by inverse CDF in index order with the counter-based uniform
 *   u = splitmix64(seed ^ splitmix64(step << 32 | sequence)) >> 40 / 2^24: (seed, step, sequence) fixes the draw.
 *   temperature > 0 (greedy is cts_greedy_advance); vocab <= 2^24; state pointers as in cts_greedy_advance. */
int cts_sample_advance(cts_ctx* ctx, const void* logits, long long vocab, int batch, float temperature, int top_k, float top_p,
                       unsigned long long seed, int* out_tokens, int out_ld, int* step_ptr, int* cur_ids, int* positions,
                       int* seq_lens, int* slot_map, const int* page_table, int max_pages, int page_size, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Tensor parallelism over NVLink peer memory (SURVEY.md §5, §8e; replaces RowParallelLinear's NCCL all-reduce +
 * residual add + RMSNorm, vllm qwen2.py:100-116,168-174,299-311, for decode-sized messages).
 * cts_ipc_*: symmetric buffers -- cudaMalloc + cudaIpc handle on the owner, cudaIpcOpenMemHandle on the peers
 *   (handle = 64 opaque bytes the host exchanges through torch.distributed).
 * cts_peer_allreduce_residual_rmsnorm: ONE kernel = reduction of this rank's split-K partials + per-token cross-GPU flag
 *   barrier + peer pull of every rank's reduced fp32 row (rank order, bit-identical on all ranks) + residual add + RMSNorm.
 *   local_partial: fp32 [split_k, t, h] in local memory (output of cts_gemm with CTS_EPI_PARTIAL_F32)
 *   peer_rows:  device array float*[world] (entry r = rank r's symmetric buffer fp32 [world, max_tokens, h]: every rank
 *               PUSHES its reduced rows into slot [its rank] of every peer, then each rank sums its local slots)
 *   peer_flags: device array int*[world]   (entry r = rank r's flag table int[world][max_tokens][8], zero-initialised;
 *               one flag per (token, column chunk): the kernel runs a cluster of up to 8 CTAs per token)
 *   state:      local int[2] {epoch, done-counter}, zero-initialised, owned by the kernel
 *   Consecutive calls must alternate between two (rows, flags) sets: the barrier of call n+1 is what licenses
 *   overwriting the rows of call n.
 */
int cts_ipc_alloc(cts_ctx* ctx, long long bytes, void** dptr, unsigned char* handle64);
int cts_ipc_open(cts_ctx* ctx, const unsigned char* handle64, void** dptr);
int cts_ipc_close(cts_ctx* ctx, void* dptr);
int cts_ipc_free(cts_ctx* ctx, void* dptr);
int cts_peer_allreduce_residual_rmsnorm(cts_ctx* ctx, const float* local_partial, int split_k, const void* peer_rows,
                                        const void* peer_flags, int* state, int rank, int world, int max_tokens,
                                        const void* resid_in, void* resid_out, const void* norm_w, float eps, void* norm_out,
                                        long long t, long long h, int dtype, void* stream);

/* Low-latency variant of cts_peer_allreduce_residual_rmsnorm (same result contract: h = resid + dtype(sum over ranks, rank order),
 * norm_out = RMSNorm(h) * w, bit-identical on every rank; replaces the same RowParallelLinear -> all-reduce -> add -> RMSNorm,
 * vllm qwen2.py:100-116,168-174): a two-shot all-reduce -- reduce-scatter of the fp32 partials to per-column-chunk owners, then
 * an all-gather of the owners' rounded h chunks and sums of squares -- whose validity flags travel inside the data (16-byte units
 * {d0, epoch, d1, epoch}), so there is no fence, no flag store and no round trip: two one-way NVLink hops per call and
 * T*h*12 bytes of egress instead of (world-1)*T*h*4.  world in {2, 4, 8}; h % (4*world) == 0.
 *   peer_regions: device array void*[world]; entry r = rank r's region of THIS buffer set (zero-initialised, >= region_bytes,
 *                 cts_peer_ll_region_bytes(world, max_tokens, h)); two sets must alternate between consecutive calls
 *   state:        local int[2], zero-initialised (epoch, arrivals)
 */
long long cts_peer_ll_region_bytes(int world, int max_tokens, long long h);
int cts_peer_allreduce_ll(cts_ctx* ctx, const float* local_partial, int split_k, const void* peer_regions, long long region_bytes,
                          int* state, int rank, int world, int max_tokens, const void* resid_in, void* resid_out, const void* norm_w,
                          float eps, void* norm_out, long long t, long long h, int dtype, void* stream);

/* vocab-parallel greedy sampling + decode-state advance over peer memory (no NCCL): local argmax of this rank's logits
 * shard [batch, vocab_shard], candidates pushed to every peer, global winner chosen identically on all ranks
 * (replaces ParallelLMHead's logits all-gather + sampler, chatts_vllm.py:607-610, for greedy decoding).
 *   peer_cand:  device array float2*[world] (entry r = rank r's candidate table float2[world][max_batch])
 *   peer_flags: device array int*[world]    (entry r = rank r's flag table int[world][max_batch], zero-initialised)
 *   state:      local int[2], zero-initialised;  step_ptr int[2] as in cts_greedy_advance
 */
int cts_peer_greedy_advance(cts_ctx* ctx, const void* logits, long long vocab_shard, int batch, int rank, int world,
                            const void* peer_cand, const void* peer_flags, int* state, int max_batch, int* out_tokens, int out_ld,
                            int* step_ptr, int* cur_ids, int* positions, int* seq_lens, int* slot_map, const int* page_table,
                            int max_pages, int page_size, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decode "chain": everything between two attention calls of a decode step (t <= 32 tokens) in ONE persistent,
 * cooperatively launched kernel (modeling_qwen2.py:269-310 minus the attention):
 *   phase 0 o_proj GEMM | 1 residual+RMSNorm(ln_post) | 2 gate_up GEMM | 3 SwiGLU | 4 down GEMM |
 *   phase 5 residual+RMSNorm(ln_next) | 6 QKV GEMM of the next layer | 7 bias+(q/k norm)+RoPE+paged KV write
 * Phases [phase_begin, phase_end) run, separated by grid barriers; the TMA producer pre-loads the weight tiles of the
 * next GEMM phase before each barrier so the HBM stream never stops.  Same arithmetic / rounding points as cts_gemm +
 * the cts_reduce_* / cts_qkv_rope_cache kernels it replaces on the decode path.
 *   split[4]: split-K factors of {o_proj, gate_up, down, qkv}; tiles*split of every phase must fit one co-resident wave.
 *   ws: fp32 >= max(split*t*n) floats; ssq: fp32 [t*8]; sync: int32[2], zero-filled once (self-resetting).
 *   wgu is the INTERLEAVED gate/up weight (see CTS_EPI_SWIGLU_IL).  norm5_has_partial = 0: phase 5 is a plain RMSNorm of h
 *   (the "head" chain embed -> norm -> QKV -> RoPE of layer 0).
 */
typedef struct {
  int t, hidden, inter, nh, nkv, head_dim;
  int phase_begin, phase_end, norm5_has_partial, dtype;
  int split[4];
  const void* wo; const void* wgu; const void* wd; const void* wqkv;     /* weights of the phases that run (else NULL) */
  const void* ao;                                                         /* [t, nh*head_dim] attention output      */
  void* h; void* xn; void* act;                                           /* [t,hidden] residual, [t,hidden], [t,inter] */
  const void* ln_post; const void* ln_next; float eps;
  const void* bqkv; const void* q_norm_w; const void* k_norm_w;
  const int* positions; const void* cos_tab; const void* sin_tab; const int* slot_map;
  void* q_out; void* k_cache; void* v_cache; int page_size;
  float* ws; float* ssq; int* sync;
} cts_chain_args;

int cts_decode_chain(cts_ctx* ctx, const cts_chain_args* args, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Decode GEMM with the split-K reduction and the projection's tail fused in (csrc/gemm_decode_fused.cu): the K splits of one
 * 128-feature tile form one thread-block cluster (grid.z = cluster.z = split_k <= 8), park their fp32 accumulator tiles in
 * shared memory and reduce disjoint tokens over distributed shared memory in split order -- bit-identical to
 * cts_gemm(CTS_EPI_PARTIAL_F32) + the matching cts_reduce_* / cts_qkv_rope_cache call, without the second launch and without
 * the fp32 round trip through L2.  t <= 32 tokens.
 *   CTS_FUSED_RESIDUAL : h[t][f] = dtype(h[t][f] + dtype(acc))                     o_proj / down_proj  (modeling_qwen2.py:302,308)
 *   CTS_FUSED_SWIGLU   : act[t][i] = dtype(silu(dtype(gate_i)) * dtype(up_i)), interleaved gate/up weight, act [t, n/2]      (:47)
 *   CTS_FUSED_QKV_ROPE : bias + Qwen3 q/k norm + RoPE + q_out / paged KV write, arguments as cts_qkv_rope_cache  (:116-146,217-222)
 */
#define CTS_FUSED_RESIDUAL 0
#define CTS_FUSED_SWIGLU 1
#define CTS_FUSED_QKV_ROPE 2
typedef struct {
  const void* w; const void* x;          /* w [n, k] row-major (ld = k), x [t, k] (ld = k) */
  long long n, k, t;
  int dtype, mode, split_k, reserved;
  const void* bias;                      /* [n] or NULL (QKV_ROPE) */
  void* h;                               /* RESIDUAL: [t, n], updated in place */
  void* act;                             /* SWIGLU: [t, n/2] */
  const int* positions; const void* cos_tab; const void* sin_tab; const int* slot_map;
  void* q_out; void* k_cache; void* v_cache; const void* q_norm; const void* k_norm;
  float eps; int nh, nkv, head_dim, page_size;
  /* optional RMSNorm fusion on both sides (5 stages per layer instead of 7):
   *   norm_h != NULL: the token operand is norm_w * dtype(norm_h * rsqrt(sum_j ssq_in[t][j] / k + norm_eps)) (modeling_qwen2.py:258-263),
   *     written by the kernel straight into its B tiles -- x is ignored; ssq_in fp32 [t][ssq_tiles] = per-tile sums of squares of norm_h
   *   ssq_out != NULL (CTS_FUSED_RESIDUAL): fp32 [t][ceil(n/128)] = sum of squares of the updated h over each 128-feature tile */
  const void* norm_h; const void* norm_w; const float* ssq_in; int ssq_tiles; float norm_eps;
  float* ssq_out;
  /* optional tensor-parallel tail (CTS_FUSED_RESIDUAL of a ROW-parallel projection; world in 2..8, n % (128 * world) == 0): the
   * kernel is GEMM + all-reduce + residual in ONE launch -- every (tile, token) partial is scattered to the rank that owns the
   * tile's columns, the owner adds the contributions in rank order + residual and broadcasts the rounded h and the tile's sum of
   * squares, every rank writes h / ssq_out from the broadcast (bit-identical on all ranks).  Same wire format, regions, epoch
   * state and safety argument as cts_peer_allreduce_ll (units with the epoch inside); the two may alternate on the same regions.
   *   peer_regions: device array void*[world] for this buffer set; peer_region_bytes >= t_max * n * 12 + t_max * ceil(n/128) * 8 */
  const void* peer_regions; int* peer_state; int peer_rank, peer_world, peer_max_tokens, peer_reserved; long long peer_region_bytes;
} cts_fused_gemm_args;
int cts_gemm_decode_fused(cts_ctx* ctx, const cts_fused_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Whole decode step from C, and the two aliases of SURVEY.md 8(b)'s symbol list.  Host-side executors only: they enqueue the
 * kernels above on `stream` (capturable into a CUDA graph), nothing new runs on the device.
 *   cts_rmsnorm : out = w * dtype(x * rsqrt(mean(x^2) + eps))                      modeling_qwen2.py:258-263
 *   cts_lm_head : logits[t, vocab] = hidden[t, h] @ w[vocab, h]^T                  chatts_vllm.py:607-610
 *   cts_decoder_step : one decode step of the whole batch (modeling_qwen2.py:269-310 x n_layers; chatts_vllm.py:595-610):
 *     embed(cur_ids) -> layers -> final norm -> lm_head -> (sample != 0) greedy advance of the device-side loop state.
 *     Same launches and rounding points as the Python orchestration (chatts_b200/model.py:_decode_body, tp = 1).
 */
int cts_rmsnorm(cts_ctx* ctx, const void* x, const void* w, float eps, void* out, long long t, long long h, int dtype, void* stream);
int cts_lm_head(cts_ctx* ctx, const void* hidden, const void* w, void* logits, long long t, long long h, long long vocab, int dtype,
                void* stream);

/* A3..A7 of the TS encoder from one C call (SURVEY.md 8(b) `cts_ts_encode`): cts_ts_patch_count -> cts_ts_patchify ->
 * num_layers x cts_gemm (+ cts_reduce_bias_act when the library splits K), bias + exact-erf GELU between layers, the last layer
 * scattering row i to out[row_map[i]] (chatts_vllm.py:93-193, :569-573).  total_rows = sum of the patch counts, known to the
 * HOST (it sizes the merged sequence); act_ws: two [total_rows, hidden] ping-pong buffers; rows_ws [total_rows, in0];
 * splitk_ws: fp32, >= 16 * total_rows * hidden floats covers every split the library may choose. */
typedef struct {
  const void* x; int dtype, n_series, row_len, num_features, patch_size, mode;
  const void* pos_table; int emb_dim, max_seq_len;
  int num_layers, hidden, in0;
  const void* const* weights;        /* HOST array [num_layers] of device pointers: W_0 [hidden, in0], W_i [hidden, hidden] */
  const void* const* biases;         /* HOST array [num_layers] of device pointers: [hidden] */
  int* valid_len; int* patch_cnt; int* row_offset; int* max_valid;      /* device outputs of the count stage (n_series [+1]) */
  long long total_rows;
  void* rows_ws; void* act_ws[2]; float* splitk_ws; long long splitk_floats;
  void* out; long long out_ld; const int* row_map;                     /* row_map NULL: rows land at out[0..total_rows) */
} cts_ts_encode_args;
int cts_ts_encode(cts_ctx* ctx, const cts_ts_encode_args* args, void* stream);

/* The same encoder as ONE launch (csrc/ts_encoder_fused.cu) for prompts of up to 256 patch rows -- the BASELINE.json metric prompt is
 * 8 series x 256 points = 128 rows: patchify + last-value pad + position-embedding gather (chatts_vllm.py:107-183), every MLP layer
 * (tcgen05, the K splits of a 128-feature tile reduced over distributed shared memory inside a thread-block cluster, bias + exact-erf
 * GELU, chatts_vllm.py:83-91,186-188) and the row scatter into inputs_embeds (chatts_vllm.py:569-573), grid barriers between the
 * layers, the next layer's weight tiles requested while a CTA waits.  HBM-bound on the weight stream (212 MB at the 14B shape).
 * valid_len / row_offset / max_valid are INPUTS (cts_ts_patch_count ran: the host sizes the merged sequence from the counts);
 * splitk_ws is unused.  cts_ts_encode_fused_ok: 1 when the shape is in range (cts_ts_encode then takes this path by itself). */
int cts_ts_encode_fused_ok(const cts_ts_encode_args* args);
int cts_ts_encode_fused(cts_ctx* ctx, const cts_ts_encode_args* args, void* stream);

typedef struct {
  const void* wqkv;   /* [(nh+2nkv)*d, hidden]                                       */
  const void* bqkv;   /* [(nh+2nkv)*d] or NULL (Qwen3)                               */
  const void* q_norm; /* [d] or NULL                                                 */
  const void* k_norm; /* [d] or NULL                                                 */
  const void* wo;     /* [hidden, nh*d]                                              */
  const void* wgu;    /* [2*inter, hidden], gate/up INTERLEAVED (CTS_EPI_SWIGLU_IL)  */
  const void* wd;     /* [hidden, inter]                                             */
  const void* ln1;    /* input_layernorm [hidden]                                    */
  const void* ln2;    /* post_attention_layernorm [hidden]                           */
  void* k_cache;      /* [num_pages, nkv, page_size, d] of THIS layer                */
  void* v_cache;
} cts_layer_weights;

typedef struct {
  int n_layers, hidden, inter, nh, nkv, head_dim, vocab, vocab_rows;   /* vocab_rows: rows of the embedding table (0 = vocab) */
  int page_size, num_pages, max_pages, dtype, batch, sample;
  float eps;
  int split_qkv, split_o, split_gu, split_d;   /* split-K factors (>= 1; cts_gemm_suggest_split gives the library's choice) */
  int attn_splits;
  const cts_layer_weights* layers;              /* HOST array [n_layers] */
  const void* embed; const void* final_norm; const void* lm_head; const void* cos_tab; const void* sin_tab;
  int* cur_ids; int* positions; int* seq_lens; int* slot_map; const int* page_table;     /* decode state, as cts_greedy_advance */
  int* out_tokens; int out_ld; int* step_ptr;
  void* h; void* xn; void* q; void* ao; void* act; void* logits;                         /* [batch, ...] activations */
  float* ws; long long ws_floats;               /* split-K partials, >= cts_decoder_step_ws_floats(args) */
  float* attn_ws;                               /* cts_attn_decode workspace (zero-filled once) */
} cts_decoder_step_args;

long long cts_decoder_step_ws_floats(const cts_decoder_step_args* args);
int cts_decoder_step(cts_ctx* ctx, const cts_decoder_step_args* args, void* stream);

/* ================================================================================================
 * A9  LoRA fine-tune step (SURVEY.md 8(a) row A9, BASELINE config 5: ChatTS-8B, forward + backward, data parallel).
 * The reference repo holds no training code (README.md:216-218 -> external ChatTS-Training; demo/demo_lora.ipynb cells
 * 3-4 only LOAD a peft adapter): these entry points implement the published algorithms that recipe is made of -- peft
 * lora.Linear (y = W x + (alpha/r) B A x, base frozen), transformers ForCausalLMLoss (label shift, ignore_index -100,
 * fp32 cross entropy), torch.optim.AdamW, torch clip_grad_norm_ -- and are checked against oracle/lora.py (autograd).
 *
 * Every matrix product of the step runs on cts_gemm: the forward projections, the LoRA down/up products (small-N /
 * small-K GEMMs with CTS_EPI_RESIDUAL), and the input gradients dX = dY W through TRANSPOSED copies of the frozen
 * weights kept resident in HBM ([K, N] row-major, so dX is again a K-major "TN" GEMM).  What is new here is everything
 * else: the softmax statistics of the forward attention, the attention backward, the backward of RMSNorm / SwiGLU /
 * RoPE(+q,k-norm), the fused cross-entropy forward+backward, the skinny LoRA weight gradients (HBM-bound: 2r flop per
 * 2-byte element streamed), AdamW and the global-norm clip on flat fp32 arenas, and the packing of the fp32 master
 * adapters into the bf16 fused operands the GEMMs read.
 * ================================================================================================ */

/* cts_attn_prefill that also returns the softmax statistics the backward needs:
 *   lse fp32 [t, nh] = log(sum_j exp(scale * q_i.k_j))  (natural log, causal, per token and q head).
 * Same kernels as cts_attn_prefill (a template flag adds the one store per row). */
int cts_attn_prefill_lse(cts_ctx* ctx, const void* q, const void* k, const void* v, const int* cu_seqlens, int batch,
                         int max_seqlen, long long total_tokens, int nh, int nkv, int head_dim, float scale, void* out,
                         float* lse, int dtype, void* stream);

/* Backward of the causal GQA attention (modeling_qwen2.py:161-184 under autograd; FlashAttention-2 recomputation:
 * P = exp(scale S - lse), dV = P^T dO, dP = dO V^T, dS = P o (dP - delta), dQ = scale dS K, dK = scale dS^T Q).
 *   q [t, nh*d], k/v [t, nkv*d] (RoPE applied, as given to the forward), out/dout [t, nh*d], lse fp32 [t, nh]
 *   delta_ws fp32 [t, nh] scratch (rowsum(dO o O), written by the first of the three launches)
 *   dq [t, nh*d], dk/dv [t, nkv*d] model dtype (dk/dv summed over the q heads of the group inside the kernel: no atomics)
 */
int cts_attn_bwd(cts_ctx* ctx, const void* q, const void* k, const void* v, const void* out, const void* dout,
                 const float* lse, const int* cu_seqlens, int batch, int max_seqlen, long long total_tokens, int nh, int nkv,
                 int head_dim, float scale, float* delta_ws, void* dq, void* dk, void* dv, int dtype, void* stream);

/* SwiGLU from a model-dtype gate/up tensor (the LoRA update lands on gate and up BEFORE the activation, so the training
 * forward cannot use the fused CTS_EPI_SWIGLU_IL epilogue):  out[t][i] = dtype(dtype(silu(g_i)) * u_i)   (modeling_qwen2.py:47)
 *   gu [t, 2*inter]: stacked (g_i at i, u_i at inter+i) or interleaved per 128-column tile (see CTS_EPI_SWIGLU_IL)
 * backward: dgu[g_i] = dact_i * u_i * silu'(g_i), dgu[u_i] = dact_i * silu(g_i), same layout as gu. */
int cts_swiglu(cts_ctx* ctx, const void* gu, long long t, long long inter, int interleaved, void* out, int dtype, void* stream);
int cts_swiglu_bwd(cts_ctx* ctx, const void* gu, const void* dact, long long t, long long inter, int interleaved, void* dgu,
                   int dtype, void* stream);

/* Backward of y = w * dtype(x * rsqrt(mean(x^2) + eps)) (modeling_qwen2.py:258-263) w.r.t. x, weight frozen, fused with the
 * residual-stream add:  dx_out = (dres_in ? dres_in : 0) + rstd * (g - xhat * mean(g o xhat)),  g = dy o w, xhat = x * rstd.
 * dx_out may alias dres_in or dy. */
int cts_rmsnorm_bwd(cts_ctx* ctx, const void* dy, const void* x, const void* w, float eps, const void* dres_in, void* dx_out,
                    long long t, long long h, int dtype, void* stream);

/* Backward of cts_qkv_rope_cache (non-partial input): un-rotate dq/dk (RoPE is orthogonal per pair), then the per-head
 * RMSNorm backward when q_norm_w / k_norm_w are given (Qwen3), dv passes through.
 *   dq [t, nh*d], dk/dv [t, nkv*d]; qkv [t, (nh+2nkv)*d] = the projection output the forward consumed (pre-norm, pre-RoPE)
 *   dqkv [t, (nh+2nkv)*d] */
int cts_qkv_rope_bwd(cts_ctx* ctx, const void* dq, const void* dk, const void* dv, const void* qkv, const int* positions,
                     const void* cos_tab, const void* sin_tab, const void* q_norm_w, const void* k_norm_w, float norm_eps,
                     void* dqkv, long long t, int nh, int nkv, int head_dim, int dtype, void* stream);

/* Fused cross entropy forward + backward over the selected rows (transformers ForCausalLMLoss: fp32 upcast, the caller
 * has already shifted: targets[i] is the label of row i):
 *   row_loss[i] = logsumexp(logits[i]) - logits[i][targets[i]];  logits[i][:] <- (softmax(logits[i]) - onehot) * grad_scale
 *   (in place, model dtype);  loss_out[0] = (accumulate ? loss_out[0] : 0) + grad_scale * sum_i row_loss[i]
 *   grad_scale = 1 / (number of counted label positions of the optimisation step); vocab % 8 == 0. */
int cts_ce_loss_grad(cts_ctx* ctx, void* logits, long long ld, const int* targets, long long n_rows, long long vocab,
                     float grad_scale, float* row_loss, float* loss_out, int accumulate, int dtype, void* stream);

/* dst[i][:] = idx[i] >= 0 ? src[idx[i]][:] : 0   (select the label rows before lm_head; scatter their gradient back) */
int cts_gather_rows(cts_ctx* ctx, const void* src, const int* idx, long long n_out, long long h, void* dst, int dtype,
                    void* stream);

/* Skinny LoRA weight gradient, HBM-bound:  out[m*so_m + j*so_r] += scale * sum_t P[t][col(m)] * Q[t][q_col0 + j]
 *   P [t, p_ld] model dtype; col(m) = p_col0 + m (p_il = 0), or the gate (p_il = 1) / up (p_il = 2) column of feature m
 *   in the interleaved gate_up layout;  Q [t, q_ld] model dtype;  m < M (even), j < r (<= 64);  out fp32, ALWAYS accumulated
 *   (the caller zero-fills the gradient arena once per optimisation step; the token range is split over CTAs and
 *   combined with fp32 atomics).
 *   dB[out, r] = s * dY^T U : P = dY, Q = U, so_m = r, so_r = 1;    dA[r, in] = dU^T X : P = X, Q = dU, so_m = 1, so_r = in */
int cts_lora_wgrad(cts_ctx* ctx, const void* p, long long p_ld, long long p_col0, int p_il, long long m, const void* q,
                   long long q_ld, long long q_col0, int r, long long t, float scale, float* out, long long so_m,
                   long long so_r, int dtype, void* stream);

/* torch.optim.AdamW on a flat fp32 arena (decoupled weight decay, bias correction; `step` counts from 1).
 * grad_scale: optional DEVICE pointer to a float the gradient is multiplied with first (the clip coefficient of
 * cts_grad_norm_clip: no host round trip between backward and update). */
int cts_adamw(cts_ctx* ctx, float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
              float eps, float weight_decay, int step, const float* grad_scale, void* stream);

/* torch.nn.utils.clip_grad_norm_ on a flat arena: out[0] = ||g||_2, out[1] = min(1, max_norm / (out[0] + 1e-6))
 * (max_norm <= 0: out[1] = 1).  ws: fp32 [cts_grad_norm_ws_floats()] scratch.  Fixed summation order. */
long long cts_grad_norm_ws_floats(void);
int cts_grad_norm_clip(cts_ctx* ctx, const float* g, long long n, float max_norm, float* ws, float* out, void* stream);

/* Pack the fp32 master adapters into the model-dtype fused operands the GEMMs read (run once after every AdamW step).
 * desc: DEVICE int64 [n_desc][CTS_PACK_DESC_LONGS], one per adapter matrix `src` [rows, cols] at master + src_off:
 *   {src_off, rows, cols, dst_off, dst_ld, row0, il_mode, col0, dstT_off, dstT_ld, scale_bits (fp32 bit pattern), 0}
 *   work[dst_off  + rowmap(i) * dst_ld  + col0 + j]   = dtype(scale * src[i][j])
 *   work[dstT_off + (col0 + j) * dstT_ld + rowmap(i)] = dtype(scale * src[i][j])            (transposed copy)
 *   rowmap(i) = row0 + i (il_mode 0) | gate (1) / up (2) row of feature i in the interleaved gate_up layout
 * max_elems = max over the descriptors of rows * cols (grid bound). */
#define CTS_PACK_DESC_LONGS 12
int cts_lora_pack(cts_ctx* ctx, const float* master, const long long* desc, int n_desc, long long max_elems, void* work,
                  int dtype, void* stream);

/* W4A16 decode GEMM for GPTQ-Int4 checkpoints (README.md:52,262-263): partial[s][t][n] = sum over split s of x[t][k] * W[n][k] with
 * W[n][k] = scales[n][k / g] * (q[n][k] - zeros[n][k / g]) dequantised inside the TMA -> shared memory -> tcgen05 operand path
 * (csrc/gemm_w4.cu), so a decode step streams the 4-bit codes -- a quarter of the bf16 bytes.  1 <= t <= 32; out = fp32 split-K
 * partials [split_k, t, n] exactly as cts_gemm(CTS_EPI_PARTIAL_F32) writes them (the cts_reduce_* / cts_qkv_rope_cache tails finish
 * the projection); results are bit-identical to cts_gemm on the dequantised weight.
 *   qw     uint8 [n, k/2]  4-bit codes, 8 consecutive k per 32-bit word in the order chatts_b200/weights.py:repack_gptq_w4 writes
 *   scales [n, k/group_size] model dtype;  zeros uint8 [n, k/group_size] integer zero points (checkpoint offset included) */
typedef struct {
  const void* qw; const void* scales; const void* zeros; const void* x; float* out;
  long long n, k, t, x_ld;
  int group_size, split_k, dtype, reserved;
} cts_gemm_w4_args;
int cts_gemm_w4(cts_ctx* ctx, const cts_gemm_w4_args* args, void* stream);
int cts_gemm_w4_suggest_split(cts_ctx* ctx, long long n, long long k);

/* The same projection with the weight operand dequantised in REGISTERS (csrc/gemm_w4_mma.cu: mma.sync, persistent CTAs, the 4-bit
 * stream by cp.async.bulk) -- the decode path's default for Int4 checkpoints since the shared-memory round trip of cts_gemm_w4 caps it at
 * the speed of the 16-bit GEMM.  Same outputs up to the fp32 summation order (the 16-bit operand values are identical).
 *   qw   uint8, ceil(n / 256) * (k / 64) chunks of 8192 bytes: chunk (tile, kb) holds features [256 tile, 256 tile + 256) x K [64 kb, 64 kb + 64) as
 *        mma.m16n8k16 A fragments -- byte ((m * 32 + lane) * 16 + 4 ks) is the word of m-tile m (16 features), lane (g = lane / 4, t = lane % 4), k16 step ks,
 *        nibble i < 4 / i + 4 = the codes at k = 16 ks + 2t + 8 (i / 2) + {0 / 1} of feature row g + 8 (i % 2)   (chatts_b200/weights.py:repack_w4_mma)
 *   szp  uint32 [ceil(n / 256), k / group_size, 256]: scale bits (model dtype) | (magic + zero point) << 16, magic = 0x4300 (bf16) / 0x6400 (fp16);
 *        features beyond n: 0
 * k must be a multiple of 128, group_size 64 or a multiple of 128; split_k <= k / 128 (the K ranges of the partials are cut at multiples of 128). */
typedef struct {
  const void* qw; const void* szp; const void* x; float* out;
  long long n, k, t, x_ld;
  int group_size, split_k, dtype, reserved;
} cts_gemm_w4f_args;
int cts_gemm_w4_mma(cts_ctx* ctx, const cts_gemm_w4f_args* args, void* stream);
int cts_gemm_w4_mma_suggest_split(cts_ctx* ctx, long long n, long long k, long long t);

/* The W4A16 projection for prefill-sized steps (any t; the model uses it for t > 32) of GPTQ-Int4 checkpoints (README.md:52,262-263):
 * a persistent tcgen05 GEMM (csrc/gemm_w4_persistent.cu) that dequantises the SAME fragment-major copy cts_gemm_w4_mma streams (qw, szp
 * exactly as in cts_gemm_w4f_args) into the shared-memory A operand, so a model needs no dense copy of its projections.  Epilogues with
 * cts_gemm's semantics, and results BIT-IDENTICAL to cts_gemm on the dequantised weight (weights.py:dequantize_w4):
 *   CTS_EPI_NONE         out[t][n] = dtype(acc + bias)                                 (bias optional, [n] model dtype)
 *   CTS_EPI_RESIDUAL     out[t][n] = dtype(dtype(acc + bias) + residual[t][n])         (residual may alias out; row stride out_ld)
 *   CTS_EPI_SWIGLU_IL    out[t][j] = dtype(dtype(silu(dtype(gate))) * dtype(up)) over a gate/up weight interleaved per 64 rows
 *                        (n % 128 == 0, t > 128; out [t, n / 2])
 *   CTS_EPI_PARTIAL_F32  out = fp32 [split_k, t, n]; split s sums the 64-wide K blocks [kb * s / split_k, kb * (s + 1) / split_k),
 *                        kb = k / 64 -- cts_gemm's partition, so the cts_reduce_* / cts_qkv_rope_cache tails take either
 * k % 128 == 0; group_size 64 or a multiple of 128 dividing k; 1 <= split_k <= k / 64 (> 1 only with CTS_EPI_PARTIAL_F32); x rows
 * 16-byte aligned (x_ld >= k, x_ld % 8 == 0); qw / szp 16-byte aligned.  A failed check returns CTS_ERR_BAD_ARG and launches nothing. */
typedef struct {
  const void* qw; const void* szp; const void* x; const void* bias; const void* residual; void* out;
  long long n, k, t, x_ld, out_ld;
  int group_size, split_k, dtype, epilogue;
} cts_gemm_w4p_args;
int cts_gemm_w4_prefill(cts_ctx* ctx, const cts_gemm_w4p_args* args, void* stream);

/* Repetition penalty (transformers RepetitionPenaltyLogitsProcessor; generation_config.json of a checkpoint may set it): the set of
 * token ids that occur in a row's sequence is a bit mask seen[batch][words_per_row] (words_per_row >= ceil(vocab / 32), zeroed by the
 * caller).  _mark sets the bits of n (row, token) pairs (rows NULL: pair i belongs to row i -- the new token of every sequence after
 * a step); _apply rewrites logit = logit / penalty (logit > 0) or logit * penalty for every marked token, once per token. */
int cts_rep_penalty_mark(cts_ctx* ctx, const int* tokens, const int* rows, int n, unsigned* seen, int words_per_row, long long vocab,
                         void* stream);
int cts_rep_penalty_apply(cts_ctx* ctx, void* logits, long long vocab, long long ld, int batch, const unsigned* seen, int words_per_row,
                          float penalty, int dtype, void* stream);

/* Debug / profiling aid (csrc/trace.cuh): instrumented kernels append {tag, %globaltimer} records to `buf` (unsigned long long
 * [2 + 2*capacity]: [0] cursor, [1] capacity, then the records) -- the overlapped timeline of a CUDA-graph replay that ncu, which
 * serialises kernels, cannot show (tools/trace_decode_step.py).  buf = NULL switches it off (the default). */
int cts_trace_enable(cts_ctx* ctx, unsigned long long* buf);

#ifdef __cplusplus
}
#endif
#endif /* CHATTS_B200_H */
