/*
 * pli_attention.h — C ABI of the B200-native attention hot path.
 *
 * This is the drop-in boundary for the one data-parallel path of
 * Infatoshi/physics-llm-inference that this repository rebuilds (SURVEY.md §8):
 * chapter 6's tiled FlashAttention forward, with chapter 1's causal mask and GQA head map,
 * and the decode-time read of the chapter 2 contiguous KV cache / chapter 7 paged KV blocks.
 *
 * The reference has no FFI of its own (SURVEY.md §8(b)): its boundary is the Python function
 * `flash_attention_forward(q, k, v, scale=None, config=None)`.  Each entry point below names
 * the reference code (path:line under /root/reference) whose arithmetic it replaces.  The Python
 * host side (`physics_llm_inference_b200/`) binds these symbols with ctypes and keeps the
 * reference's call signature; INTEGRATION.md shows the stub a maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *   - strides are in ELEMENTS; the innermost (head_dim) stride is always 1;
 *   - the caller owns every buffer (outputs, workspace); nothing is allocated or freed here;
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous, no host sync, safe
 *     under CUDA-graph capture;
 *   - return value 0 = success, negative = error (`pli_last_error()` gives the text; errors are
 *     thread-local).  Nothing throws across the ABI.  There is no CPU fallback.
 */
#ifndef PLI_ATTENTION_H_
#define PLI_ATTENTION_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLI_ABI_VERSION 1

/* element types of q/k/v/o and of the KV storage */
#define PLI_BF16 0
#define PLI_F16 1
#define PLI_F32 2

/* error codes */
#define PLI_OK 0
#define PLI_ERR_INVALID (-1)      /* bad shape / dtype / alignment / argument            */
#define PLI_ERR_UNSUPPORTED (-2)  /* valid request this build has no kernel for          */
#define PLI_ERR_CUDA (-3)         /* a CUDA runtime / driver call failed                 */
#define PLI_ERR_DEVICE (-4)       /* current device is not sm_100 (B200)                 */

/* which kernel family served a request (reported by pli_*_kernel_kind) */
#define PLI_KIND_NONE 0
#define PLI_KIND_TCGEN05 1 /* TMA + tcgen05.mma + TMEM, bf16/f16, head_dim 64/128       */
#define PLI_KIND_SIMT 2    /* CUDA-core fp32-accumulate kernel: f32 inputs, odd head_dim */
#define PLI_KIND_MMA_TMA 3 /* decode: TMA page loads + mma.sync, bf16/f16                */

int pli_abi_version(void);
const char* pli_last_error(void);

/* Make `device` current for this library's CUDA runtime (the host side calls it next to
 * torch.cuda.device(...), so both runtimes agree).  Also checks that the device is sm_100. */
int pli_set_device(int device);

/* Number of kernels this library has launched on the calling thread since load (or since the
 * last pli_reset_launch_count).  bench.py reports it as `gpu_launches`. */
uint64_t pli_launch_count(void);
void pli_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Prefill / full attention forward.
 *
 * Replaces ch06/flash_attention.py:14-74 (`flash_attention_forward`: S = QK^T*scale :55,
 * online-softmax rescale :57-62, O update :64-65), with
 *   - GQA head map of ch01/gqa.py:14,30-31: q-head h reads kv-head h / (Hq/Hkv);
 *   - causal rule of ch01/gqa.py:33-34 and ch02/cached_generation.py:85-91: key j is visible to
 *     query i iff j <= i + (Nk - Nq) (bottom-right aligned; requires Nq <= Nk);
 *   - log-sum-exp per row (the reference computes row_max/row_sum at :71-72 and drops them).
 *
 *   q  (B,Hq,Nq,D)   k,v (B,Hkv,Nk,D)   o (B,Hq,Nq,D) same dtype as q   lse (B,Hq,Nq) f32 or NULL
 *   *_strides[3] = {batch, head, token} element strides; head_dim stride is 1.
 *   bf16/f16 with D in {64,128}: tcgen05 kernel (needs 16-byte aligned pointers and non-zero strides that
 *   are multiples of 8 elements; a broadcast / zero stride cannot be described by a TMA tensor map).
 *   Anything else with D <= 256: SIMT kernel, which indexes with the strides exactly as given.
 * ------------------------------------------------------------------------------------------- */
int pli_prefill_fwd(const void* q, const void* k, const void* v, void* o, float* lse,
                    int B, int Hq, int Hkv, int Nq, int Nk, int D,
                    const int64_t q_strides[3], const int64_t k_strides[3],
                    const int64_t v_strides[3], const int64_t o_strides[3],
                    float scale, int causal, int dtype, void* stream);

/* Chunked prefill over PAGED K/V (SURVEY.md §8(f) F1): Nq new query tokens per sequence attend to that sequence's
 * cached keys, read in place from the ch07 pools (ch07/paged_memory.py:38-48) through the block table — what
 * `ChunkedPrefillScheduler` (ch08/chunked_prefill.py:32-51,79-113) emits once the chunk's own K/V have been
 * appended (pli_kv_append).  Maths: ch02/cached_generation.py:72-94 with the offset causal mask :85-91,
 * per sequence: query i sees key j iff j <= i + (seq_lens[b] - Nq); requires seq_lens[b] >= Nq.
 *   q, o (B,Hq,Nq,D) strides {batch, head, token};  pools / block_table / kv_strides / layer as for decode;
 *   seq_lens (B,) int32 device: cached length of each sequence INCLUDING the Nq new tokens;
 *   max_seq_len: host upper bound;  bf16/f16, D in {64,128}, block_size in {16,32,64,128}.
 * Storage past seq_lens[b] (the rest of a sequence's last page, unused pages) may hold anything, NaN/Inf included:
 * the reference's allocator recycles pages without clearing them (ch07/paged_memory.py:100-110).  Scores of those
 * keys are replaced by select and their V rows are zeroed in shared memory before any MMA reads them. */
int pli_prefill_paged_fwd(const void* q, const void* k_pool, const void* v_pool,
                          const int32_t* block_table, const int32_t* seq_lens, void* o, float* lse,
                          int B, int Hq, int Hkv, int Nq, int D, int max_seq_len,
                          int block_size, int table_stride, int layer, int64_t num_pages,
                          const int64_t q_strides[3], const int64_t kv_strides[4], const int64_t o_strides[3],
                          float scale, int dtype, void* stream);

/* The same over RAGGED query lengths: one launch serves a batch whose sequences bring different numbers of new
 * tokens, the attention step of the mixed prefill/decode batches `MixedBatchScheduler.schedule`
 * (ch08/mixed_batch.py:63-104) and `ChunkedPrefillScheduler` (ch08/chunked_prefill.py:79-113) emit.
 *   q, o (total_q, Hq, D) packed over sequences, strides {token, head}; rows [cu_seqlens_q[b], cu_seqlens_q[b+1])
 *   are the newest tokens of sequence b (cu_seqlens_q: (B+1,) int32 device, non-decreasing, [0] = 0, [B] = total_q);
 *   query i of sequence b sees key j iff j <= i + (seq_lens[b] - q_len[b]);  seq_lens[b] >= max(q_len[b], 1);
 *   max_q_len: host upper bound of the q_len[b];  lse (Hq, total_q) or NULL.  Other arguments as above. */
int pli_prefill_varlen_paged_fwd(const void* q, const void* k_pool, const void* v_pool,
                                 const int32_t* block_table, const int32_t* seq_lens, const int32_t* cu_seqlens_q,
                                 void* o, float* lse, int B, int Hq, int Hkv, int64_t total_q, int max_q_len, int D,
                                 int max_seq_len, int block_size, int table_stride, int layer, int64_t num_pages,
                                 const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                                 float scale, int dtype, void* stream);

/* Which kernel pli_prefill_fwd would use for this problem (PLI_KIND_*), without launching. */
int pli_prefill_kernel_kind(int D, int dtype, const int64_t q_strides[3], const int64_t k_strides[3],
                            const int64_t v_strides[3], const int64_t o_strides[3],
                            const void* q, const void* k, const void* v, const void* o);

/* ---------------------------------------------------------------------------------------------
 * Decode: one query token per sequence over a KV cache, split-KV + log-sum-exp combine.
 *
 * Replaces the attention block of ch02/cached_generation.py:72-94 (`CachedGQA.forward`; same
 * maths at ch02/kv_cache.py:81-98) for seq_len == 1 (no mask, :85), reading either
 *   - the contiguous cache of ch02/kv_cache.py:25-34 / ch02/cached_generation.py:23
 *       (B, max_seq_len, Hkv, D), block_table == NULL; or
 *   - the paged pools of ch07/paged_memory.py:38-48 (num_blocks, num_layers, block_size, Hkv, D)
 *     through a block table (ch07/paged_memory.py:7-13): logical token t of sequence b lives in
 *     page block_table[b*table_stride + t / block_size], slot t % block_size (ceil-div rule of
 *     ch07/paged_memory.py:54,84-86).  Tokens >= seq_lens[b] are never read as values.
 *
 *   q (B,Hq,D) with strides {batch, head};  o (B,Hq,D) same dtype;  lse (B,Hq) f32 or NULL.
 *   kv_strides[4] = element strides of the K/V storage:
 *       paged:       {page, layer, slot, head}      contiguous: {batch, 0, token, head}
 *   kv_extent = number of pages in the pool (paged) or B (contiguous): bounds for TMA descriptors.
 *   max_seq_len = upper bound of seq_lens (host value; no device sync is done to find it).
 *   num_splits  = KV splits per (b, kv head), 1..64; pass 0 to let the library pick
 *                 (pli_decode_num_splits); workspace must hold pli_decode_workspace_bytes() and
 *                 needs NO initialisation (it carries the partials and, behind them, one arrival
 *                 counter pair per (b, kv head) that tolerates any previous contents); 16-byte
 *                 aligned; launches that share one must be ordered (e.g. issued on one stream).
 *
 * pli_decode_fwd is ONE launch on the TMA path (bf16 / f16, head_dim 64 / 128): with several splits the
 * CTA of a (b, kv head) that finishes last merges that unit's partials itself.  pli_decode_splitkv
 * (partials into workspace) + pli_decode_combine is the same computation as two launches, and what
 * pli_decode_fwd does on the SIMT path.
 * ------------------------------------------------------------------------------------------- */
int pli_decode_num_splits(int B, int Hkv, int max_seq_len);
size_t pli_decode_workspace_bytes(int B, int Hq, int D, int num_splits);

int pli_decode_splitkv(const void* q, const void* k_store, const void* v_store,
                       const int32_t* block_table, const int32_t* seq_lens,
                       int B, int Hq, int Hkv, int D, int max_seq_len,
                       int block_size, int table_stride, int layer, int64_t kv_extent,
                       const int64_t q_strides[2], const int64_t kv_strides[4],
                       float scale, int dtype, int num_splits,
                       void* workspace, size_t workspace_bytes, void* stream);

int pli_decode_combine(const void* workspace, void* o, float* lse,
                       int B, int Hq, int D, int num_splits,
                       const int64_t o_strides[2], int dtype, void* stream);

int pli_decode_fwd(const void* q, const void* k_store, const void* v_store,
                   const int32_t* block_table, const int32_t* seq_lens,
                   void* o, float* lse,
                   int B, int Hq, int Hkv, int D, int max_seq_len,
                   int block_size, int table_stride, int layer, int64_t kv_extent,
                   const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                   float scale, int dtype, int num_splits,
                   void* workspace, size_t workspace_bytes, void* stream);

int pli_decode_kernel_kind(int D, int dtype, int block_size, const int64_t kv_strides[4],
                           const void* k_store, const void* v_store);

/* Decode with q_len (1..16) new query tokens per sequence in ONE split-KV launch: the verify step of speculative
 * decoding, multi-token-prediction heads, short chunk tails.  Maths: ch02/cached_generation.py:72-94 for seq_len = q_len
 * > 1, with the offset causal mask :85-91: query i of sequence b sees key j iff j <= i + seq_lens[b] - q_len.
 *   q (B,Hq,q_len,D) with strides {batch, head, token}, any (e.g. the (B,q_len,Hq,D).transpose(1,2) view of a projection);
 *   o (B,Hq,q_len,D) with strides {batch, head, token}: its head stride must be q_len * its token stride (a tensor
 *   contiguous in its last three dimensions; PLI_ERR_INVALID otherwise);  lse (B,Hq,q_len) f32 contiguous or NULL;
 *   seq_lens (B,) int32 device: cached length INCLUDING the q_len new tokens (their K/V already appended, as for
 *   pli_prefill_paged_fwd); requires seq_lens[b] >= q_len (not checked on the device).
 *   Other arguments as for pli_decode_fwd.  The q_len rows of a q head are served as extra rows of its KV group (G*q_len
 *   rows per KV head, in 16-row chunks), so each K/V byte is still read once per chunk;
 *   workspace: pli_decode_workspace_bytes(B, Hq*q_len, D, num_splits);
 *   num_splits = 0 picks pli_decode_num_splits_multi(B, Hq, Hkv, q_len, max_seq_len).
 * q_len > 16: PLI_ERR_UNSUPPORTED (use pli_prefill_paged_fwd / pli_prefill_fwd).  The peer-output entries above take one
 * token per sequence.  With q_len = 1 this computes what pli_decode_fwd computes, with the same automatic split count. */
int pli_decode_fwd_multi(const void* q, const void* k_store, const void* v_store,
                         const int32_t* block_table, const int32_t* seq_lens,
                         void* o, float* lse,
                         int B, int Hq, int Hkv, int q_len, int D, int max_seq_len,
                         int block_size, int table_stride, int layer, int64_t kv_extent,
                         const int64_t q_strides[3], const int64_t kv_strides[4], const int64_t o_strides[3],
                         float scale, int dtype, int num_splits,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The split count pli_decode_fwd_multi picks for num_splits = 0: its grid's units are (b, kv head, 16-row chunk of the
 * G*q_len rows of a KV head), i.e. pli_decode_num_splits(B, Hkv*ceil(G*q_len/16), max_seq_len); for q_len = 1 exactly
 * pli_decode_num_splits(B, Hkv, max_seq_len). */
int pli_decode_num_splits_multi(int B, int Hq, int Hkv, int q_len, int max_seq_len);

/* Decode fused with the all-gather of its output over NVLink / NVSwitch peer memory.  The reference has no
 * collective (ch09/nccl_primitives.py:45-67 only models all-gather cost); a tensor-parallel caller that shards KV
 * heads over ranks (one process per GPU) needs every rank's heads on every rank after the attention block.  Here
 * every rank owns the FULL output (B, Hq_total, D) in peer-mapped memory (symmetric memory / CUDA IPC set up by the
 * host), and a rank's decode kernel stores its slice straight into all of them.  pli_peer_publish_wait, launched
 * behind it on the same stream, publishes the step number at peer_flags[r][rank] for every r (release, system
 * scope), makes the stream wait until peer_flags[rank][r] has reached it for all r (every rank's slice has landed
 * HERE) and then advances *epoch.
 *   B, Hq, Hkv and q / kv / workspace describe the LOCAL shard exactly as for pli_decode_fwd;
 *   peer_o[r]: output buffer 0 of rank r, buffer 1 follows buffer_stride elements later; o_strides {batch, head}:
 *   element strides inside one buffer; slice_offset: element offset of this rank's first (batch row, head);
 *   lse (B, Hq) local or NULL;  peer_flags[r]: rank r's array of n_peers zero-initialised words;
 *   epoch: LOCAL zero-initialised device word = steps completed.  The step in flight is *epoch + 1 and writes
 *   buffer (*epoch + 1) & 1; both are read on the device, so the two launches can be captured in a CUDA graph.
 * Double-buffering by step parity is sufficient: a rank only passes the wait of step e+1 after every peer has
 * finished, on its stream, the kernels that read the output of step e. */
#define PLI_MAX_PEERS 8
typedef struct pli_peer_scatter {
    int32_t n_peers, rank;
    void* peer_o[PLI_MAX_PEERS];
    uint32_t* peer_flags[PLI_MAX_PEERS];
    uint32_t* epoch;
    int64_t buffer_stride;
    int64_t slice_offset;
    /* pli_decode_fwd_gather only (may be NULL for the calls above): */
    uint32_t* peer_ready[PLI_MAX_PEERS];   /* rank r's array of n_peers zero-initialised "ready to receive" words */
    uint32_t* cta_counter;                 /* LOCAL zero-initialised device word; only read by builds that publish from the
                                              decode grid's last CTA (-DPLI_PUBLISH_FROM_LAST_CTA=1), may be NULL otherwise */
} pli_peer_scatter;
int pli_decode_fwd_scatter(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                           const int32_t* seq_lens, float* lse, int B, int Hq, int Hkv, int D, int max_seq_len,
                           int block_size, int table_stride, int layer, int64_t kv_extent,
                           const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                           float scale, int dtype, int num_splits, void* workspace, size_t workspace_bytes,
                           const pli_peer_scatter* ps, void* stream);
int pli_peer_publish_wait(const pli_peer_scatter* ps, void* stream);

/* The same gather as ONE call and ONE output buffer per rank (buffer_stride must be 0; the output address never changes,
 * so the step captures into a CUDA graph next to its consumers without a copy).  The publish / wait kernel is launched by
 * this call, programmatically behind the decode grid (no launch latency).  Two credits replace the second buffer:
 *   peer_ready[r][rank] = e  is raised by this rank's kernel of step e when it STARTS (stream order: everything that read
 *                            this rank's buffer of step e-1 is complete), and a CTA stores into rank r's buffer only after
 *                            it has seen peer_ready[rank][r] >= e;
 *   peer_flags[r][rank] = e  is published once the decode grid is complete (the whole slice has been stored); the stream
 *                            then waits for peer_flags[rank][r] >= e for all r and *epoch advances.
 * Same arguments as pli_decode_fwd_scatter; served by the TMA kernel only (bf16 / f16, head_dim 64 / 128, page size a power
 * of two): PLI_ERR_UNSUPPORTED otherwise, before anything is launched.  Stream contract: the kernels that read the output of
 * step e are enqueued before step e+1 on the same stream (or ordered before it by an event).  A peer that does not show up
 * within pli_set_peer_timeout_ms is reported through pli_device_status, not trapped.
 * (ch09/nccl_primitives.py:45-67 is the reference's cost model of the all-gather this replaces.) */
int pli_decode_fwd_gather(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                          const int32_t* seq_lens, float* lse, int B, int Hq, int Hkv, int D, int max_seq_len,
                          int block_size, int table_stride, int layer, int64_t kv_extent,
                          const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                          float scale, int dtype, int num_splits, void* workspace, size_t workspace_bytes,
                          const pli_peer_scatter* ps, void* stream);

/* Copy the output buffer written by the step that has just completed on this stream (its parity is read from the device
 * step counter) into a FIXED destination of `nbytes` bytes (elements of `elem_size` bytes).  Needed under CUDA-graph
 * capture: the buffer a replay writes alternates with the step parity, so a consumer captured in the same graph (the output
 * projection, the next layer) must read from an address that does not.  Launch it after pli_peer_publish_wait. */
int pli_peer_select_copy(const pli_peer_scatter* ps, void* dst, int64_t nbytes, int elem_size, void* stream);

/* How long pli_peer_publish_wait waits for a peer rank's slice before it gives up (milliseconds of wall time; default
 * 60 000; 0 = forever).  Giving up does NOT trap: the kernel records the event (below) and the stream continues. */
int pli_set_peer_timeout_ms(int64_t ms);

/* Host-visible fault record (eight words in host-mapped pinned memory, readable even after a kernel trapped):
 *   out[0] code: 0 none, 1 an intra-kernel mbarrier wait exceeded its wall-time bound (protocol bug; that kernel trapped),
 *                2 a peer rank's slice did not arrive within the peer timeout (no trap; the step's output is incomplete);
 *   out[1] code 1: block << 32 | thread;  code 2: waiting rank << 32 | missing rank;
 *   out[2] code 1: barrier shared-memory address | parity << 32;  code 2: step number;   out[3] %globaltimer (ns).
 * clear != 0 resets the record after reading it. */
int pli_device_status(uint64_t out[8], int clear);

/* Prefill with the same fused all-gather: the epilogue's TMA store of every finished O tile goes to all ranks'
 * full outputs (B_total, Hq_total, Nq, D), so the transfer overlaps the MMAs of the following tiles; follow it with
 * pli_peer_publish_wait.  q/k/v/lse and B, Hq, Hkv describe the LOCAL shard as for pli_prefill_fwd; o_strides
 * {batch, head, token} are those of the full output; the shard's first batch row / q head inside it are
 * batch_offset / head_offset (ps->slice_offset is not used).  bf16/f16, head_dim 64/128 only. */
int pli_prefill_fwd_scatter(const void* q, const void* k, const void* v, float* lse, int B, int Hq, int Hkv,
                            int Nq, int Nk, int D, const int64_t q_strides[3], const int64_t k_strides[3],
                            const int64_t v_strides[3], const int64_t o_strides[3], float scale, int causal,
                            int dtype, int B_total, int Hq_total, int batch_offset, int head_offset,
                            const pli_peer_scatter* ps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * KV-cache write path (SURVEY.md §8(f) F1): append n new tokens per sequence.
 *
 * Replaces the slice-assign of ch02/kv_cache.py:45-46 / ch02/cached_generation.py:30-31
 * (`cache[:, seq_len:seq_len+n] = new`) and, for pages, the write that
 * ch07/paged_memory.py:76-98 (`extend_blocks`) makes room for.
 *
 *   k_new,v_new (B, n, Hkv, D) with new_strides {batch, token, head};
 *   start_pos (B,) int32: position of the first new token per sequence (device);
 *   storage / block_table / kv_strides as for decode.
 * ------------------------------------------------------------------------------------------- */
int pli_kv_append(const void* k_new, const void* v_new, void* k_store, void* v_store,
                  const int32_t* block_table, const int32_t* start_pos,
                  int B, int n_new, int Hkv, int D,
                  int block_size, int table_stride, int layer,
                  const int64_t new_strides[3], const int64_t kv_strides[4],
                  int dtype, void* stream);

/* Debug / parity aid: gather one layer of paged K (or V) into a contiguous (B, max_len, Hkv, D)
 * buffer with the kernel-side address rule, so tests can assert page indexing bit-exactly. */
int pli_paged_gather(const void* store, void* out, const int32_t* block_table, const int32_t* seq_lens,
                     int B, int max_len, int Hkv, int D, int block_size, int table_stride, int layer,
                     const int64_t kv_strides[4], int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The scalar online-softmax recurrence on its own (ch06/online_softmax.py).
 *
 * pli_online_softmax replaces `online_softmax(x)` (:13-25): softmax over the last dimension through the running
 * (max, sum) update  m' = max(m, x_i),  d' = d*exp(m - m') + exp(x_i - m').
 * pli_online_softmax_with_output replaces `online_softmax_with_output(x, v)` (:28-53): the same with the running
 * weighted sum  o' = (o*d*exp(m - m') + v_i*exp(x_i - m')) / d';  writes o (rows, dv) and d (rows,) = sum_i exp(x_i - max).
 *   x (rows, n), out (rows, n), v (rows, n, dv), o (rows, dv): leading dimensions flattened to `rows`;
 *   *_row_stride = elements between consecutive rows, v_elem_stride = elements between consecutive i; innermost
 *   strides are 1.  f32 / bf16 / f16; fp32 arithmetic.  dv <= 256.
 * ------------------------------------------------------------------------------------------- */
int pli_online_softmax(const void* x, void* out, int64_t rows, int n, int64_t x_row_stride, int64_t out_row_stride,
                       int dtype, void* stream);
int pli_online_softmax_with_output(const void* x, const void* v, void* o, float* d, int64_t rows, int n, int dv,
                                   int64_t x_row_stride, int64_t v_row_stride, int64_t v_elem_stride,
                                   int64_t o_row_stride, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PLI_ATTENTION_H_ */
