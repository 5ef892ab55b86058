// decode.cu — split-KV decode attention over the ch02 contiguous cache / ch07 paged pools, the merge of the splits,
// the KV append (write path), the page-gather parity aid and the NVLink gather of the output.
//
// Maths: ch02/cached_generation.py:72-94 for seq_len == 1 (no mask, :85) with the GQA map of
// :77-78, and for 2-16 new tokens per sequence (pli_decode_fwd_multi) with the offset causal mask of :85-91, the tokens
// of a q head served as extra rows of its KV group.  Addressing: ch07/paged_memory.py:38-48 pool layout, token t ->
// page table[t / bs], slot t % bs (ceil-div rule, :54,:84-86).  HBM-bound: each K/V byte is read exactly once and all
// q heads of a KV group are served from that one read.
//
//   decode_tma_kernel   bf16/f16, head_dim 64/128, page size 2^k in [8,256] (or contiguous): two producer warps stream
//                       64-token K / V stages into a 128B-swizzled smem ring with TMA (one box per page, page ids from the
//                       block table), four consumer warps run QK^T and PV on mma.sync m16n8k16 via ldmatrix, fp32 softmax
//                       state.  ONE launch per decode call: a single split writes the output; 2 / 4 / 8 splits of a unit
//                       form a thread-block cluster and merge through distributed shared memory; more splits leave
//                       partials (of clusters of eight) in the workspace and the CTA that arrives last on the unit's
//                       counter merges them (DESIGN.md 3.3).  With a peer table the final stores go to every rank's copy
//                       of the output over NVLink (pli_decode_fwd_gather, DESIGN.md 4).
//   decode_simt_kernel  everything else (f32 storage, odd head_dim / page size): CUDA cores, partials only.
//   decode_combine_kernel  the two-launch form's merge of the partials (pli_decode_splitkv + pli_decode_combine; SIMT path).
#include <atomic>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace pli {
namespace {

// Tokens [t0, t1) of sequence length L handled by split s of S (multiples of 64; may be empty).
__host__ __device__ __forceinline__ void split_range(int L, int S, int s, int& t0, int& t1) {
    int chunk = (((L + S - 1) / S) + 63) & ~63;
    t0 = min(L, s * chunk);
    t1 = min(L, t0 + chunk);
}

// the same with the division by S done as multiply-high + shift (S is a launch constant)
__device__ __forceinline__ void split_range_fast(int L, int S, const FastDiv& fd, int s, int& t0, int& t1) {
    const int chunk = ((int)fd.div((uint32_t)(L + S - 1)) + 63) & ~63;
    t0 = min(L, s * chunk);
    t1 = min(L, t0 + chunk);
}

__device__ __forceinline__ int64_t token_offset(const int32_t* __restrict__ table, int b, int t, int bs,
                                                int table_stride, int layer, int hk, int64_t s_page,
                                                int64_t s_layer, int64_t s_slot, int64_t s_head) {
    if (table != nullptr) {
        const int page = table[(int64_t)b * table_stride + t / bs];
        return page * s_page + layer * s_layer + (int64_t)(t % bs) * s_slot + hk * s_head;
    }
    return b * s_page + (int64_t)t * s_slot + hk * s_head;
}

// ------------------------------------------------------------------------------------------------
// SIMT split-KV kernel (generic)
// ------------------------------------------------------------------------------------------------
template <typename T, int kDC>
__global__ void __launch_bounds__(128) decode_simt_kernel(
    const T* __restrict__ q, const T* __restrict__ ks, const T* __restrict__ vs,
    const int32_t* __restrict__ table, const int32_t* __restrict__ seq_lens, int Hq, int Hkv, int D, int bs,
    int table_stride, int layer, int64_t qsb, int64_t qsh, int64_t s_page, int64_t s_layer, int64_t s_slot,
    int64_t s_head, float scale, int S, float* __restrict__ o_part, float* __restrict__ lse_part, int q_len, int64_t qst) {
    __shared__ float sm_m[4], sm_d[4];
    extern __shared__ float sm_acc[];  // [4][D]
    const int s = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int hk = h / (Hq / Hkv);
    int t0, t1;
    const int L = seq_lens[b];
    split_range(L, S, s, t0, t1);
    // q_len > 1: h is a virtual head (q head * q_len + token index i), and token i sees keys j < L - (q_len - 1 - i)
    // (ch02/cached_generation.py:85-91); a row left without keys in this split ends with m = -inf, den = 0
    t1 = min(t1, L - (q_len - 1 - h % q_len));

    float qv[kDC], acc[kDC];
#pragma unroll
    for (int c = 0; c < kDC; ++c) {
        const int d = lane + 32 * c;
        qv[c] = d < D ? to_f32<T>(q[b * qsb + (h / q_len) * qsh + (h % q_len) * qst + d]) : 0.f;
        acc[c] = 0.f;
    }
    float m = -INFINITY, dsum = 0.f;
    for (int t = t0 + warp; t < t1; t += 4) {
        const int64_t off = token_offset(table, b, t, bs, table_stride, layer, hk, s_page, s_layer, s_slot, s_head);
        float kv[kDC], vv[kDC];
#pragma unroll
        for (int c = 0; c < kDC; ++c) {
            const int d = lane + 32 * c;
            kv[c] = d < D ? to_f32<T>(ks[off + d]) : 0.f;
            vv[c] = d < D ? to_f32<T>(vs[off + d]) : 0.f;
        }
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < kDC; ++c) dot = fmaf(qv[c], kv[c], dot);
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o2);
        const float sv = dot * scale;
        const float m_new = fmaxf(m, sv);
        const float alpha = (m == -INFINITY) ? 0.f : expf(m - m_new);
        const float p = expf(sv - m_new);
        dsum = dsum * alpha + p;
#pragma unroll
        for (int c = 0; c < kDC; ++c) acc[c] = fmaf(p, vv[c], acc[c] * alpha);
        m = m_new;
    }
    if (lane == 0) {
        sm_m[warp] = m;
        sm_d[warp] = dsum;
    }
#pragma unroll
    for (int c = 0; c < kDC; ++c)
        if (lane + 32 * c < D) sm_acc[warp * D + lane + 32 * c] = acc[c];
    __syncthreads();
    float M = fmaxf(fmaxf(sm_m[0], sm_m[1]), fmaxf(sm_m[2], sm_m[3]));
    float w[4], den = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        w[i] = (sm_m[i] == -INFINITY) ? 0.f : expf(sm_m[i] - M);
        den += w[i] * sm_d[i];
    }
    const int64_t row = ((int64_t)b * Hq + h) * S + s;
    const float inv = den > 0.f ? 1.f / den : 0.f;
    for (int d = threadIdx.x; d < D; d += 128) {
        float o = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) o += w[i] * sm_acc[i * D + d];
        o_part[row * D + d] = o * inv;
    }
    if (threadIdx.x == 0) lse_part[row] = den > 0.f ? M + logf(den) : -INFINITY;
}

// ------------------------------------------------------------------------------------------------
// TMA + mma.sync split-KV kernel
// ------------------------------------------------------------------------------------------------
// Option (off): launch the split-KV kernel programmatically behind its predecessor on the stream (launch_tma_t; its first
// statement is griddepcontrol.wait, so only launch latency is hidden).  Eager steps gain ~2 us (C5 share 25.5 -> 23.6 us,
// batch 8 x 8k 46.5 -> 44.3), graph replays nothing, and the clustered many-split case loses 6 us (one 32k sequence: 27.6
// -> 33.5 us graph, 29.8 -> 37.0 eager): the early-resident dependent grid gets in the way of the running grid's clusters.
#ifndef PLI_DECODE_PDL
#define PLI_DECODE_PDL 0
#endif
constexpr bool kDecodePdl = PLI_DECODE_PDL != 0;
constexpr int kStageTokens = 64;   // tokens per pipeline stage (16 per consumer warp)
#ifndef PLI_DECODE_STAGES
#define PLI_DECODE_STAGES 3
#endif
// smem ring depth: 3 x 32 KB at D = 128 -> 2 CTAs per SM.  (6 stages and ONE CTA per SM -- the same bytes in flight, half
// the partials -- measured 15-25 % slower everywhere: C5 share at 8k context 5757 against 6687 GB/s, one 32k sequence 31.3
// against 27.6 us; four consumer warps and one producer pair per SM do not keep up.)
constexpr int kDecodeStages = PLI_DECODE_STAGES;
constexpr int kConsumerWarps = 4;
constexpr int kProducerWarps = 2;  // warp 4 loads the K tiles, warp 5 the V tiles: issuing a TMA from lanes with different
                                   // operands costs ~70 cycles each (an elect / R2UR loop), 16 of them per 16-token-page stage
constexpr int kDecodeThreads = (kConsumerWarps + kProducerWarps) * 32;

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
template <bool kBf16>
__device__ __forceinline__ void mma16816(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    if constexpr (kBf16) {
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
            "{%0,%1,%2,%3};\n"
            : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
            : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    } else {
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
            "{%0,%1,%2,%3};\n"
            : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
            : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
}

// byte offset of (row, 16-byte chunk) inside a [rows][64 el] 128B-swizzled sub-tile
__device__ __forceinline__ uint32_t sw128(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }

// Fused all-gather of the decode output over NVLink peer memory (pli_decode_fwd_scatter): every rank holds the
// FULL (B, Hq_total, D) output in peer-mapped memory and a rank's kernel stores its slice into all of them (plain
// stores, no fence on the hot path).  The kernel boundary completes them; the one-warp peer_publish_wait_kernel
// that follows on the stream publishes `epoch` in every rank's flag word for this rank (release, system scope) and
// then waits for every rank's flag here.
// The step number lives in device memory (*epoch = steps completed; the step in flight is *epoch + 1 and writes
// output buffer (*epoch + 1) & 1), so a captured CUDA graph replays correctly.
struct PeerScatter {
    void* o[PLI_MAX_PEERS];           // buffer 0 of every rank
    int n;
    const uint32_t* epoch;
    int64_t buffer_stride;            // elements from buffer 0 to buffer 1
    int64_t slice_offset;             // element offset of this rank's (batch, head) slice inside the full tensor
    __device__ __forceinline__ int64_t base() const { return slice_offset + (int64_t)((*epoch + 1u) & 1u) * buffer_stride; }
};
struct PeerFlags {
    uint32_t* flags[PLI_MAX_PEERS];
    int n, rank;
    uint32_t* epoch;
    unsigned long long timeout_ns;    // 0: wait forever
    unsigned long long* status;       // host-visible fault record (common.cuh), or NULL
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}

#if defined(PLI_TUNING) && PLI_TUNING
#define PLI_DECODE_TRACE(slot)                                                                                       \
    do {                                                                                                             \
        if (p.trace != nullptr) {                                                                                    \
            const int cta_ = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;                         \
            if (cta_ < p.trace_cap) {                                                                                \
                if ((slot) == 0) p.trace[cta_ * 16 + 7] = global_timer_ns();                                         \
                p.trace[cta_ * 16 + (slot)] = (unsigned long long)clock64();                                         \
            }                                                                                                        \
        }                                                                                                            \
    } while (0)
#else
#define PLI_DECODE_TRACE(slot) do { } while (0)
#endif

// Spin (acquire, system scope) until *w has reached e.  A peer that is merely late is waited for: the bound is WALL time
// (pli_set_peer_timeout_ms; 0 = forever); false when it expired.
__device__ __forceinline__ bool wait_flag_reaches(const uint32_t* w, uint32_t e, unsigned long long timeout_ns) {
    uint64_t t0 = 0;
    for (uint32_t spin = 1; (int32_t)(ld_acquire_sys(w) - e) < 0; ++spin) {
        __nanosleep(32);
        if ((spin & 0x3FFu) == 0 && timeout_ns != 0) {
            const uint64_t now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > timeout_ns) return false;
        }
    }
    return true;
}
// A peer did not show up in time: no trap -- (this rank, the missing rank, the step) go into the host-visible fault
// record, which pli_device_status / PeerOutput turn into an error on the host, and the stream continues.
__device__ __forceinline__ void record_peer_timeout(unsigned long long* status, int rank, int missing, uint32_t e) {
    if (status == nullptr) return;
    status[1] = ((unsigned long long)rank << 32) | (unsigned)missing;
    status[2] = e;
    status[3] = global_timer_ns();
    __threadfence_system();
    status[0] = PLI_FAULT_PEER_TIMEOUT;
    __threadfence_system();
}

// Single-launch gather (pli_decode_fwd_gather): ONE output buffer per rank and a credit in each direction.
//   ready[r][me] = e   written by me into rank r's memory when my kernel of step e STARTS: everything on my stream that read
//                      my buffer's step e-1 contents is complete, rank r may overwrite its slice of it;
//   done[r][me]  = e   written by me into rank r's memory when all of my slice of step e has landed there.
// A CTA stores into rank r's buffer only after it has seen ready[me][r] >= e (polled by a producer warp while the K/V
// stream runs, handed to the consumers through an mbarrier); the last CTA of the grid to finish publishes done, waits for
// every peer's done and advances *epoch.  No rank ever waits for something that depends on its own progress in step e,
// so this cannot deadlock as long as every rank launches step e.
struct PeerGather {
    uint32_t* done[PLI_MAX_PEERS];
    uint32_t* ready[PLI_MAX_PEERS];
    uint32_t* epoch;                  // LOCAL: steps completed
    uint32_t* cta_counter;            // LOCAL: CTAs of the running grid that have finished (zero between launches)
    int n, rank;                      // n == 0: not a single-launch gather
    unsigned long long timeout_ns;
    unsigned long long* status;
};

struct DecodeTmaParams {
    unsigned long long* trace;   // tuning builds: 16 timestamps per CTA (pli_debug_decode_trace), else NULL
    int trace_cap;
    const void* q;
    const int32_t* table;
    const int32_t* seq_lens;
    float* o_part;
    float* lse_part;
    void* o_direct;       // S == 1 only: final output (q's dtype), written instead of the partials
    float* lse_direct;
    int64_t osb, osh;
    int64_t qsb, qsh;
    int64_t qst;                      // kMulti: token stride of q (row v of the problem is q head v / q_len, token v % q_len)
    int Hq, Hkv, G, bs, table_stride, layer, S, box_tokens, max_len;
    int q_len;                        // kMulti: query tokens per sequence; Hq / G count virtual heads (q head * q_len + i)
    int bs_shift, box_shift;          // log2 of bs / box_tokens (both powers of two on this path)
    FastDiv fd_splits;                // division by S
    float scale_log2;
    PeerScatter peer;     // peer.n > 0: the final output (direct or combined in this kernel) goes to every rank
    // S > 1, fused combine: the CTA that arrives LAST on its unit's counter merges the unit's S partials and writes the
    // final output, so no second kernel follows.  counters == NULL: partials only (pli_decode_splitkv).
    unsigned long long* counters;   // two 64-bit words per (b, kv head, 16-row chunk), see unit_arrive
    uint32_t launch_id;
    void* o_final;                  // with osb / osh; unused when peer.n > 0
    float* lse_final;               // or NULL
    PeerGather gather;
    int cluster;                    // 2, 4, 8: `cluster` consecutive splits of a unit form a thread-block cluster and are
                                    // merged through distributed shared memory; else 1
    int parts;                      // partials per unit that go through global memory: S / cluster (1: none, no counters)
    int peer_vec;                   // the peers' slices can be written with 16-byte stores (alignment checked on the host)
};

// Arrival of one split's CTA on its unit's counter pair; returns the number of arrivals before this one.
//   c[0] = kCtrTag | arrivals   the fast path: ONE fetch-add per CTA.  The last arriver stores kCtrTag back (zero arrivals),
//                               so the next launch -- or the next replay of a CUDA graph -- starts from zero.
//   c[1] = launch id << 32 | arrivals   only while c[0] does not carry the tag, i.e. the first launch on a workspace that
//                               was never used (the caller's workspace needs NO initialisation): a compare-and-swap loop
//                               that treats a word left by anything but this launch as zero.  37 CTAs contending on one
//                               CAS cost ~25 us, which is why this is not the steady-state protocol.
// (Never-used memory passes for a tagged word with probability 2^-40 per counter; a launch that died half-way leaves the
// context unusable anyway.  Launches that share a workspace must be ordered, e.g. on one stream.)
// Both atomics are acq_rel at device scope: they release this CTA's partials (ordered before them by the CTA barrier) and
// acquire those of the splits that arrived earlier.
constexpr unsigned long long kCtrTag = 0xA5C3D2E1F0ull << 24;       // upper 40 bits; arrivals in the lower 24
__device__ __forceinline__ uint32_t unit_arrive(unsigned long long* c, uint32_t id, bool& tagged) {
    unsigned long long old;
    asm volatile("atom.acq_rel.gpu.global.add.u64 %0, [%1], 1;\n" : "=l"(old) : "l"(c) : "memory");
    tagged = (old >> 24) == (kCtrTag >> 24);
    if (tagged) return (uint32_t)(old & 0xFFFFFFull);
    unsigned long long seen, assumed;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];\n" : "=l"(seen) : "l"(c + 1) : "memory");
    uint32_t cnt;
    do {
        assumed = seen;
        cnt = (uint32_t)(assumed >> 32) == id ? (uint32_t)assumed : 0u;
        asm volatile("atom.acq_rel.gpu.global.cas.b64 %0, [%1], %2, %3;\n"
                     : "=l"(seen)
                     : "l"(c + 1), "l"(assumed), "l"(((unsigned long long)id << 32) | (cnt + 1u))
                     : "memory");
    } while (seen != assumed);
    return cnt;
}
// The last arriver, after the merge: zero arrivals for the next launch (nobody else touches the pair any more).
__device__ __forceinline__ void unit_reset(unsigned long long* c, uint32_t id, bool tagged) {
    if (!tagged) c[1] = (unsigned long long)id << 32;
    c[0] = kCtrTag;
}

// Merge of the S partials of one unit (rows_here q heads of one sequence) by the 128 consumer threads of the CTA that
// arrived last.  What this costs is the latency chain of the CTA that finishes last.  The unit's partial outputs are ONE
// contiguous block of the workspace ([row][split][kD] f32: 76 KiB for 4 heads x 37 splits), so thread 0 pulls it into
// the (idle) K/V ring with bulk copies -- one request instead of two to three rounds of twenty 16-byte loads per thread,
// which is what the merge cost when it read the partials from L2 directly -- while every thread fetches the row's LSEs
// and works out the weights; then a thread owns four output columns of one row and walks all splits in shared memory.
// Units whose partials do not fit the ring are merged in groups of rows.  No other barrier, no shared-memory reduction.
// (First version: weights per row in one warp, (row, split) pairs spread over the threads, sum through shared memory:
// three barriers and three dependent L2 round trips, 6100 cycles for S = 4 and 8700 for S = 37 against ~1700 for the
// arrival atomic itself.)
// Thread 0 of the last arriver: bulk-copy rows [r0, r0 + nr) of the unit's partial outputs into shared memory.
template <int kD>
__device__ __forceinline__ void combine_fetch(const DecodeTmaParams& p, uint8_t* smem, uint64_t* bar, int b, int h_base, int r0,
                                              int nr) {
    // the partials were written through the generic proxy (by other CTAs, acquired by this thread's arrival); the bulk
    // copy reads them, and overwrites shared memory this CTA has just read, through the async proxy
    fence_proxy_async_all();
    const uint32_t total = (uint32_t)(nr * p.parts * kD * 4);
    mbar_arrive_expect_tx(bar, total);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(p.o_part + ((int64_t)b * p.Hq + h_base + r0) * p.parts * kD);
    for (uint32_t off = 0; off < total; off += 32768u) bulk_load(smem + off, src + off, min(32768u, total - off), bar);
}
__device__ __forceinline__ int combine_rows_per_group(const DecodeTmaParams& p, int kD, int ring_bytes, int rows_here) {
    return max(1, min(rows_here, ring_bytes / (p.parts * kD * 4)));
}

template <int kD, typename elem_t>
__device__ __forceinline__ void combine_unit(const DecodeTmaParams& p, uint8_t* smem, uint64_t* bar, int ring_bytes, int b,
                                             int h_base, int rows_here, int tid) {
    const int S = p.parts;
    constexpr int kVec = kD / 4;                                  // lanes per row: 32 (D 128) or 16 (D 64), 16 bytes each
    constexpr int kPerLane = 64 / kVec;                           // LSEs per lane (S <= 64)
    const int lane_in_row = tid % kVec;
    const int rows_per_group = combine_rows_per_group(p, kD, ring_bytes, rows_here);
    float* stage = reinterpret_cast<float*>(smem);                // [rows of the group][S][kD]
    uint32_t parity = 0;
    for (int r0 = 0; r0 < rows_here; r0 += rows_per_group) {
        const int nr = min(rows_per_group, rows_here - r0);
        if (r0 > 0) named_bar_sync(1, kConsumerWarps * 32);       // the previous group has been read
        if (tid == 0 && r0 > 0) combine_fetch<kD>(p, smem, bar, b, h_base, r0, nr);    // (group 0: requested by the caller)
        const int n_items = nr * kVec;
        for (int base = (tid / 32) * 32; base < n_items; base += kConsumerWarps * 32) {      // warp-uniform trip count
            const int item = base + (tid % 32);
            const bool live = item < n_items;
            const int row = r0 + min(item, n_items - 1) / kVec, dv = lane_in_row * 4;
            const float* lp = p.lse_part + ((int64_t)b * p.Hq + h_base + row) * S;
            // the row's weights, spread over its kVec lanes
            float l[kPerLane], w[kPerLane];
            float M = -INFINITY;
#pragma unroll
            for (int k = 0; k < kPerLane; ++k) {
                const int si = lane_in_row + k * kVec;
                l[k] = si < S ? __ldcg(lp + si) : -INFINITY;
                M = fmaxf(M, l[k]);
            }
#pragma unroll
            for (int o2 = kVec / 2; o2 > 0; o2 >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o2));
            float den = 0.f;
#pragma unroll
            for (int k = 0; k < kPerLane; ++k) {
                w[k] = l[k] == -INFINITY ? 0.f : __expf(l[k] - M);
                den += w[k];
            }
#pragma unroll
            for (int o2 = kVec / 2; o2 > 0; o2 >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o2);
            const float inv = den > 0.f ? 1.f / den : 0.f;
            mbar_wait(bar, parity);                               // the group's partial outputs are in shared memory
            const float* sp = stage + (size_t)(row - r0) * S * kD + dv;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < kPerLane; ++k) {
                if (k * kVec >= S) break;                         // warp-uniform
                const int nj = min(kVec, S - k * kVec);
#pragma unroll 4
                for (int j = 0; j < nj; ++j) {
                    const float wj = __shfl_sync(0xffffffffu, w[k], j, kVec);
                    const float4 v = *reinterpret_cast<const float4*>(sp + (size_t)(k * kVec + j) * kD);
                    acc.x = fmaf(wj, v.x, acc.x); acc.y = fmaf(wj, v.y, acc.y);
                    acc.z = fmaf(wj, v.z, acc.z); acc.w = fmaf(wj, v.w, acc.w);
                }
            }
            if (!live) continue;
            const float ov[4] = {acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv};
            const int64_t off = b * p.osb + (h_base + row) * p.osh + dv;
            if (p.peer.n > 0) {
                const int64_t poff = p.peer.base() + off;
                __align__(8) elem_t pk[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) pk[e] = from_f32<elem_t>(ov[e]);
                for (int r = 0; r < p.peer.n; ++r) {
                    elem_t* dst = reinterpret_cast<elem_t*>(p.peer.o[r]) + poff;
                    if (p.peer_vec) {
                        *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(pk);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) dst[e] = pk[e];
                    }
                }
            } else {
                elem_t* dst = reinterpret_cast<elem_t*>(p.o_final) + off;
#pragma unroll
                for (int e = 0; e < 4; ++e) dst[e] = from_f32<elem_t>(ov[e]);
            }
            if (dv == 0 && p.lse_final != nullptr)
                p.lse_final[(int64_t)b * p.Hq + h_base + row] = den > 0.f ? M + logf(den) : -INFINITY;
        }
        parity ^= 1u;
    }
}

// kMulti: p.q_len query tokens per sequence (pli_decode_fwd_multi).  Row r of a unit is virtual head h_base + r, i.e.
// token i = (h_base + r) % q_len of its q head, and sees keys j < seq_len - (q_len - 1 - i) (ch02/cached_generation.py:
// 85-91).  Only the last q_len - 1 keys of a sequence differ between rows: that mask sits behind a warp-uniform test, so
// interior stages run the one-token code.  A row can then see no key of a whole warp step or split (m = -inf): its
// softmax update subtracts 0 instead of -inf, and the merges already weight a -inf state by 0.
template <int kD, bool kBf16, bool kRows16, bool kMulti>
__global__ void __launch_bounds__(kDecodeThreads) decode_tma_kernel(const __grid_constant__ CUtensorMap map_k,
                                                                    const __grid_constant__ CUtensorMap map_v,
                                                                    const __grid_constant__ DecodeTmaParams p) {
    constexpr int kHalves = kD / 64;
    constexpr int kSubTile = kStageTokens * 128;              // bytes of one [64 tok][64 el] sub-tile
    constexpr int kTileBytes = kHalves * kSubTile;            // K (or V) bytes per stage
    constexpr int kNT = kD / 8;                               // PV n-tiles
    constexpr int kRowSlots = kRows16 ? 2 : 1;
    // regions of the (then idle) K/V ring reused after the last stage: cross-warp merge area, bf16 staging of the peer
    // stores, cluster exchange area -- all inside the ring for both head dims (D 64: 27.9 of 48 KiB)
    constexpr int kMergeBytes = (128 + 64 * (kD + 8)) * 4;
    constexpr int kStageOOffset = (kMergeBytes + 1023) & ~1023;
    constexpr int kXchgOffset = kStageOOffset + 4096;
    static_assert(kXchgOffset + 16 * kD * 4 + 64 <= 2 * kDecodeStages * kTileBytes, "epilogue regions must fit the K/V ring");
    using elem_t = typename std::conditional<kBf16, __nv_bfloat16, __half>::type;

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // (an offset added to the __shared__ array, not a pointer rebuilt from an integer: the compiler keeps the address
    // space, so the merge code below compiles to LDS / STS instead of generic loads)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* k_tiles = smem;                                  // [stages][kTileBytes]
    uint8_t* v_tiles = smem + kDecodeStages * kTileBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(v_tiles + kDecodeStages * kTileBytes);
    uint64_t* empty_bar = full_bar + kDecodeStages;
    uint64_t* peer_ok = empty_bar + kDecodeStages + 1;        // (empty_bar[kDecodeStages] is the is_last word)
    uint64_t* merge_bar = peer_ok + 1;                        // the last arriver's bulk copy of the unit's partials

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x, b = blockIdx.z;
    const int hk = blockIdx.y % p.Hkv, hchunk = blockIdx.y / p.Hkv;   // hchunk: 16-row groups when G > 16
    pdl_wait();                                                       // (see launch_tma_t) no-op for a plain launch
    if (threadIdx.x == 0) PLI_DECODE_TRACE(0);                        // CTA start
    // The parameter block spans several 64-byte lines of the constant bank; one lane per warp touches a line each, so
    // that first-use misses later in the kernel (~600 cycles each) are all in flight together here.
    {
        constexpr int kLines = (int)((sizeof(DecodeTmaParams) + 63) / 64);
        const uint32_t* words = reinterpret_cast<const uint32_t*>(&p);
        if (lane == 0) {
            for (int l = warp; l < kLines; l += kConsumerWarps + kProducerWarps) {
                const uint32_t v = words[l * 16];
                asm volatile("" ::"r"(v));
            }
        }
    }
    // Start-up is a chain of dependent misses (sequence length -> block-table entries -> first TMA): shorten it.  A
    // producer lane fetches the tensor maps first; the consumer threads, idle until the first stage lands, pull the
    // part of this sequence's block-table row the CTA can touch towards L2 while the length is still in flight ...
    if (threadIdx.x == kConsumerWarps * 32) {
        prefetch_tensormap(&map_k);
        prefetch_tensormap(&map_v);
    }
    if (p.table != nullptr && threadIdx.x < kConsumerWarps * 32) {
        const int line = threadIdx.x * 32;                            // 32 entries = 128 bytes
        if (line < p.table_stride) prefetch_l2(p.table + (int64_t)b * p.table_stride + line);
    }
    // single-launch gather: this rank's kernel of step e has started, so its output buffer may be overwritten
    uint32_t step = 0;
    if (!kMulti && p.gather.n > 0) {                                  // (no peer output with q_len > 1)
        step = *p.gather.epoch + 1u;
        if (blockIdx.x + blockIdx.y + blockIdx.z == 0 && warp == kConsumerWarps && lane < p.gather.n)
            st_release_sys(p.gather.ready[lane] + p.gather.rank, step);
    }
    const int seq_len = p.seq_lens[b];                                // in flight; first used below
    // ... and the producers read the block-table entries of their first stage for the split range the sequence would have
    // at the host's max_seq_len (always right for a single split, right for every full-length sequence otherwise) without
    // waiting for the length; a shorter sequence re-reads them once the length is known.
    int t0_guess, t1_guess, page_guess = 0;
    split_range_fast(p.max_len, p.S, p.fd_splits, s, t0_guess, t1_guess);
    if (warp >= kConsumerWarps && p.table != nullptr) {
        const int idx = (t0_guess + (lane << p.box_shift)) >> p.bs_shift;
        if (lane < (kStageTokens >> p.box_shift) && idx < p.table_stride) page_guess = p.table[(int64_t)b * p.table_stride + idx];
    }
    int t0, t1;
    split_range_fast(seq_len, p.S, p.fd_splits, s, t0, t1);
    const int n_stages = (t1 - t0 + kStageTokens - 1) / kStageTokens;
    const int rows_here = min(p.G - hchunk * 16, kRows16 ? 16 : 8);
    const int h_base = hk * p.G + hchunk * 16;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kDecodeStages; ++i) {
            mbar_init(&full_bar[i], kProducerWarps);
            mbar_init(&empty_bar[i], kConsumerWarps);
        }
        mbar_init(peer_ok, 1);
        mbar_init(merge_bar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) PLI_DECODE_TRACE(12);
    // programmatic dependent launch: the combine pass (launched with programmatic stream serialisation) may be
    // scheduled as soon as every CTA of this grid is running; it still waits for this grid's completion and memory
    // flush in its own griddepcontrol.wait, so only its launch latency is hidden.  No-op without a dependent.
    pdl_launch_dependents();

    // ---- fused combine (consumer warps): this CTA's partial (or its cluster's) is in global memory; arrive on the unit's
    // counter, and if this was the last of the unit's p.parts partials, merge them all into the final output ----
    // (the partial stores of the 128 threads -- or, through the cluster barrier, of the whole cluster -- happen before
    // thread 0's release; the merge reads the partial outputs through thread 0's bulk copy, issued behind its acquire and a
    // proxy fence, and the partial LSEs with ld.global.cg, i.e. from L2, after the barrier that follows the acquire)
    auto arrive_and_merge = [&]() {
        const int tid = threadIdx.x;
        int* is_last = reinterpret_cast<int*>(empty_bar + kDecodeStages);
        named_bar_sync(1, kConsumerWarps * 32);
        unsigned long long* ctr = p.counters + 2 * ((int64_t)b * gridDim.y + blockIdx.y);
        bool tagged = false;
        if (tid == 0) {
            const bool last = unit_arrive(ctr, p.launch_id, tagged) == (uint32_t)p.parts - 1u;
            *is_last = last;
            // (every consumer thread is past its last read of the merge area: the barrier above) the first group of the
            // unit's partials is requested before the other threads even learn that this CTA merges
            if (last)
                combine_fetch<kD>(p, smem, merge_bar, b, h_base, 0,
                                  min(rows_here, combine_rows_per_group(p, kD, 2 * kDecodeStages * kTileBytes, rows_here)));
        }
        named_bar_sync(1, kConsumerWarps * 32);
        if (*is_last) {
            if (p.gather.n > 0) mbar_wait(peer_ok, 0);
            combine_unit<kD, elem_t>(p, smem, merge_bar, 2 * kDecodeStages * kTileBytes, b, h_base, rows_here, tid);
            if (tid == 0) unit_reset(ctr, p.launch_id, tagged);
            if (threadIdx.x == 0) PLI_DECODE_TRACE(5);       // combined output written
        }
    };

    if (warp >= kConsumerWarps) {
        // ===================== producer warps: TMA page loads (warp 4: K tiles, warp 5: V tiles) =====================
        if (n_stages > 0) {
            const bool is_v = warp != kConsumerWarps;
            const CUtensorMap* map = is_v ? &map_v : &map_k;
            uint8_t* tiles = is_v ? v_tiles : k_tiles;
            const int boxes = kStageTokens >> p.box_shift;     // boxes (pages or sub-pages) per stage
            const bool paged = p.table != nullptr;
            // lane i < boxes owns box i of every stage; its page id is fetched one stage ahead
            auto page_of = [&](int it) -> int {
                const int t = t0 + it * kStageTokens + (lane << p.box_shift);
                if (!paged || lane >= boxes || t >= t1) return 0;
                return p.table[(int64_t)b * p.table_stride + (t >> p.bs_shift)];
            };
            int page_next = (t0 == t0_guess) ? page_guess : page_of(0);
#if defined(PLI_TUNING) && PLI_TUNING
            if (threadIdx.x == kConsumerWarps * 32 && page_next >= -0x7fffffff) PLI_DECODE_TRACE(13);   // (the compare makes the stamp wait for the load)
#endif
            for (int it = 0; it < n_stages; ++it) {
                const int slot = it % kDecodeStages;
                const uint32_t parity = ((it / kDecodeStages) & 1) ^ 1;
                const int page = page_next;
                if (it + 1 < n_stages) page_next = page_of(it + 1);
                mbar_wait(&empty_bar[slot], parity);
                // boxes that start at or beyond t1 are not loaded; consumers never read their smem as values
                const int remaining = t1 - (t0 + it * kStageTokens);
                const int live_boxes = min(boxes, (remaining + p.box_tokens - 1) >> p.box_shift);
                if (lane == 0)
                    mbar_arrive_expect_tx(&full_bar[slot], (kHalves * live_boxes * 128) << p.box_shift);
                __syncwarp();
                if (it == 0 && threadIdx.x == kConsumerWarps * 32) PLI_DECODE_TRACE(6);        // about to issue the first loads
                if (lane < live_boxes) {
                    const int t = t0 + it * kStageTokens + (lane << p.box_shift);
                    // coordinates (d, head, slot, X, Y): paged (.., t % bs, layer, page); contiguous (.., t, 0, b)
                    const int c2 = paged ? (t & (p.bs - 1)) : t;
                    const int c3 = paged ? p.layer : 0;
                    const int c4 = paged ? page : b;
#pragma unroll
                    for (int hf = 0; hf < kHalves; ++hf) {
                        const int dst = slot * kTileBytes + hf * kSubTile + ((lane * 128) << p.box_shift);
                        // K/V bytes are read once: evict-first, so that the block tables, lengths, queries and partials
                        // every launch re-reads stay in L2 behind the stream
                        tma_load_5d_hint(tiles + dst, map, &full_bar[slot], hf * 64, hk, c2, c3, c4, kL2EvictFirst);
                    }
                }
                if (it == 0 && threadIdx.x == kConsumerWarps * 32) PLI_DECODE_TRACE(1);        // first stage's loads issued
            }
        }
        if (!kMulti && p.gather.n > 0 && warp == kConsumerWarps) {
            // every peer ready to receive step e?  (normally long true: they raised it when their kernels started)
            if (lane < p.gather.n &&
                !wait_flag_reaches(p.gather.ready[p.gather.rank] + lane, step, p.gather.timeout_ns))
                record_peer_timeout(p.gather.status, p.gather.rank, lane, step);
            __syncwarp();
            if (lane == 0) mbar_arrive(peer_ok);
        }
    } else {
        // ===================== consumer warps =====================
        const int g0 = lane >> 2;            // row (q head within the group) of c0,c1 / a0,a1,a4,a5
        const int qd = (lane & 3) * 2;       // column pair inside an 8-wide tile
        // Q A-fragments for every k-step; rows >= rows_here are zero
        uint32_t qa[kD / 16][4];
        {
            const elem_t* qp = reinterpret_cast<const elem_t*>(p.q) + b * p.qsb;
            // kMulti: row v of the unit is q head v / q_len, token v % q_len (two rows per thread: g0, g0 + 8)
            int64_t q_row[2] = {0, 0};
            if (kMulti) {
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                    const int v = h_base + g0 + 8 * rr;
                    q_row[rr] = (int64_t)(v / p.q_len) * p.qsh + (int64_t)(v % p.q_len) * p.qst;
                }
            }
#pragma unroll
            for (int ks = 0; ks < kD / 16; ++ks) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int row = g0 + ((j & 1) ? 8 : 0);
                    const int col = ks * 16 + qd + ((j & 2) ? 8 : 0);
                    uint32_t val = 0;
                    if (row < rows_here && (kRows16 || !(j & 1)))
                        val = *reinterpret_cast<const uint32_t*>(qp + (kMulti ? q_row[j & 1] : (h_base + row) * p.qsh) + col);
                    qa[ks][j] = val;
                }
            }
        }
        float m_run[kRowSlots], d_run[kRowSlots];
        float acc[kNT][4];
#pragma unroll
        for (int r = 0; r < kRowSlots; ++r) {
            m_run[r] = -INFINITY;
            d_run[r] = 0.f;
        }
#pragma unroll
        for (int n = 0; n < kNT; ++n) acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
        // kMulti: keys >= mask_from are hidden from some rows; row_cut[r] is the first key hidden from row g0 (+8)
        const int mask_from = kMulti ? seq_len - p.q_len + 1 : 0;
        int row_cut[kRowSlots];
#pragma unroll
        for (int r = 0; r < kRowSlots; ++r) row_cut[r] = kMulti ? mask_from + (hchunk * 16 + g0 + 8 * r) % p.q_len : 0;

        const uint32_t k_base = smem_u32(k_tiles), v_base = smem_u32(v_tiles);
        // ldmatrix lane roles: matrix id = lane / 8, row inside the matrix = lane % 8
        const int lm = lane >> 3, lr = lane & 7;
        const int k_row = warp * 16 + ((lm & 2) ? 8 : 0) + lr;   // K: matrices {0,1} tokens 0-7, {2,3} tokens 8-15
        const int k_chk = (lm & 1);                              //    matrices {0,2} chunk kc, {1,3} chunk kc+1
        const int v_row = warp * 16 + ((lm & 1) ? 8 : 0) + lr;   // V: matrices {0,2} tokens 0-7, {1,3} tokens 8-15
        const int v_chk = (lm >> 1);                             //    matrices {0,1} chunk nc, {2,3} chunk nc+1

        for (int it = 0; it < n_stages; ++it) {
            const int slot = it % kDecodeStages;
            mbar_wait(&full_bar[slot], (it / kDecodeStages) & 1);
            if (it == 0 && threadIdx.x == 0) PLI_DECODE_TRACE(2);    // first stage landed
            const int tok_base = t0 + it * kStageTokens + warp * 16;
            const int n_valid = t1 - tok_base;                   // valid tokens in this warp's 16
            if (n_valid > 0) {
                // ---- S = Q K^T : 16 rows x 16 tokens ----
                float sacc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
                for (int ks = 0; ks < kD / 16; ++ks) {
                    const int hf = ks / 4, chunk = (ks % 4) * 2 + k_chk;
                    uint32_t b0, b1, b2, b3;
                    ldsm_x4(k_base + slot * kTileBytes + hf * kSubTile + sw128(k_row, chunk), b0, b1, b2, b3);
                    mma16816<kBf16>(sacc[0], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b0, b1);
                    mma16816<kBf16>(sacc[1], qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3], b2, b3);
                }
                // ---- online softmax (log2 domain), rows g0 (+8) ----
                uint32_t pa[4];
#pragma unroll
                for (int r = 0; r < kRowSlots; ++r) {
                    float sv[4] = {sacc[0][2 * r], sacc[0][2 * r + 1], sacc[1][2 * r], sacc[1][2 * r + 1]};
                    if (n_valid < 16) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int tk = (j >> 1) * 8 + qd + (j & 1);
                            if (tk >= n_valid) sv[j] = -INFINITY;
                        }
                    }
                    if (kMulti && tok_base + 16 > mask_from) {           // warp-uniform: the last q_len - 1 keys
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int tk = (j >> 1) * 8 + qd + (j & 1);
                            if (tok_base + tk >= row_cut[r]) sv[j] = -INFINITY;
                        }
                    }
                    float mx = fmaxf(fmaxf(sv[0], sv[1]), fmaxf(sv[2], sv[3]));
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                    const float m_new = fmaxf(m_run[r], mx);
                    // (kMulti: a row with no key so far keeps m = -inf; subtracting 0 keeps alpha and p at 0, not NaN)
                    const float ms = (kMulti && m_new == -INFINITY) ? 0.f : __fmul_rn(m_new, p.scale_log2);
                    // both products rounded (__fmul_rn is never fused): an FMA would keep the rounding residual of
                    // m * scale_log2, making alpha != 1 while the maximum stands still, and the LSE drift by that
                    // residual at every warp step (~3e-3 nats over 4096 keys with logits near 1000 nats)
                    const float alpha = ex2_approx(__fmul_rn(m_run[r], p.scale_log2) - ms);   // m_run = -inf -> 0
                    float pv[4], psum = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        pv[j] = ex2_approx(fmaf(sv[j], p.scale_log2, -ms));
                        psum += pv[j];
                    }
                    psum += __shfl_xor_sync(0xffffffffu, psum, 1);
                    psum += __shfl_xor_sync(0xffffffffu, psum, 2);
                    d_run[r] = d_run[r] * alpha + psum;
                    m_run[r] = m_new;
                    if (alpha != 1.f) {
#pragma unroll
                        for (int n = 0; n < kNT; ++n) {
                            acc[n][2 * r] *= alpha;
                            acc[n][2 * r + 1] *= alpha;
                        }
                    }
                    pa[r] = pack2<kBf16>(pv[0], pv[1]);          // a0a1 (r=0) / a2a3 (r=1): tokens 0-7
                    pa[2 + r] = pack2<kBf16>(pv[2], pv[3]);      // a4a5 / a6a7: tokens 8-15
                }
                if (!kRows16) pa[1] = pa[3] = 0u;
                // ---- O += P V : 16 rows x kD ----
#pragma unroll
                for (int nt = 0; nt < kNT; nt += 2) {
                    const int hf = nt / 8, chunk = (nt % 8) + v_chk;
                    uint32_t b0, b1, b2, b3;
                    ldsm_x4_t(v_base + slot * kTileBytes + hf * kSubTile + sw128(v_row, chunk), b0, b1, b2, b3);
                    if (n_valid < 16) {  // never multiply by storage beyond seq_len (it may hold anything)
                        auto keep = [&](uint32_t x, int tk) -> uint32_t {
                            return tk >= n_valid ? 0u : (tk + 1 >= n_valid ? (x & 0xFFFFu) : x);
                        };
                        b0 = keep(b0, qd);
                        b1 = keep(b1, qd + 8);
                        b2 = keep(b2, qd);
                        b3 = keep(b3, qd + 8);
                    }
                    mma16816<kBf16>(acc[nt], pa[0], pa[1], pa[2], pa[3], b0, b1);
                    mma16816<kBf16>(acc[nt + 1], pa[0], pa[1], pa[2], pa[3], b2, b3);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[slot]);
        }

        // ---- merge the four warps' partial softmax states through smem ----
        if (threadIdx.x == 0) PLI_DECODE_TRACE(3);               // this warp's last stage consumed
        if (lane == 0) PLI_DECODE_TRACE(8 + warp);
        named_bar_sync(1, kConsumerWarps * 32);                  // every stage consumed: ring is reusable
        if (threadIdx.x == 0) PLI_DECODE_TRACE(14);
        float* mg_m = reinterpret_cast<float*>(smem);            // [4 warps][16 rows]
        float* mg_d = mg_m + 64;
        float* mg_o = mg_d + 64;                                 // [4 warps][16 rows][kD + 8]: rows 8 banks apart, so the
        constexpr int kMgStride = kD + 8;                        // float2 stores of a warp (8 rows x 4 column pairs) do not collide
        if ((lane & 3) == 0) {
#pragma unroll
            for (int r = 0; r < kRowSlots; ++r) {
                mg_m[warp * 16 + g0 + 8 * r] = m_run[r] * p.scale_log2;
                mg_d[warp * 16 + g0 + 8 * r] = d_run[r];
            }
        }
#pragma unroll
        for (int n = 0; n < kNT; ++n) {
#pragma unroll
            for (int r = 0; r < kRowSlots; ++r) {
                float2 val = make_float2(acc[n][2 * r], acc[n][2 * r + 1]);
                *reinterpret_cast<float2*>(&mg_o[(warp * 16 + g0 + 8 * r) * kMgStride + n * 8 + qd]) = val;
            }
        }
        named_bar_sync(1, kConsumerWarps * 32);
        if (threadIdx.x == 0) PLI_DECODE_TRACE(15);
        const int tid = threadIdx.x;                             // 0..127
        // four elements per thread and pass, written as four independent chains (shared-memory reads, exp2, reciprocal,
        // store): one element at a time was ~600 dependent cycles per element and warp, 2400 of a short kernel's tail
        if (p.gather.n > 0 && p.o_direct != nullptr) mbar_wait(peer_ok, 0);      // the peers' buffers may be written
        elem_t* stage_o = reinterpret_cast<elem_t*>(smem + kStageOOffset);       // [rows][kD], behind the merge area
        float* xo = reinterpret_cast<float*>(smem + kXchgOffset);                // cluster exchange: [16 rows][kD] + [16] LSEs
        float* xl = xo + 16 * kD;
        constexpr int kIlp = 4;
        for (int base = tid; base < rows_here * kD; base += kIlp * kConsumerWarps * 32) {
            float o_val[kIlp], lse_val[kIlp];
#pragma unroll
            for (int u = 0; u < kIlp; ++u) {
                const int idx = min(base + u * kConsumerWarps * 32, rows_here * kD - 1);   // clamped: the store is guarded
                const int row = idx / kD, d = idx - row * kD;
                float M = -INFINITY;
#pragma unroll
                for (int w = 0; w < 4; ++w) M = fmaxf(M, mg_m[w * 16 + row]);
                float den = 0.f, o = 0.f;
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const float mw = mg_m[w * 16 + row];
                    const float wt = (mw == -INFINITY) ? 0.f : ex2_approx(mw - M);
                    den += wt * mg_d[w * 16 + row];
                    o += wt * mg_o[(w * 16 + row) * kMgStride + d];
                }
                // (approximate division / logarithm: no slow-path call, so the four chains really interleave; both are
                // far inside the output's bf16 / the LSE's 1e-3 tolerance)
                o_val[u] = den > 0.f ? __fdividef(o, den) : 0.f;
                lse_val[u] = den > 0.f ? (M + __log2f(den)) * kLn2 : -INFINITY;
            }
#pragma unroll
            for (int u = 0; u < kIlp; ++u) {
                const int idx = base + u * kConsumerWarps * 32;
                if (idx >= rows_here * kD) break;
                const int row = idx / kD, d = idx - row * kD;
                if (p.o_direct != nullptr && p.peer.n > 0) {
                    const elem_t val = from_f32<elem_t>(o_val[u]);
                    if (p.peer_vec) {
                        stage_o[idx] = val;                      // stored to the peers below, 16 bytes per thread
                    } else {
                        const int64_t off = p.peer.base() + b * p.osb + (h_base + row) * p.osh + d;
                        for (int r = 0; r < p.peer.n; ++r) reinterpret_cast<elem_t*>(p.peer.o[r])[off] = val;
                    }
                    if (d == 0 && p.lse_direct != nullptr) p.lse_direct[(int64_t)b * p.Hq + h_base + row] = lse_val[u];
                } else if (p.o_direct != nullptr) {
                    // single split: this CTA owns the whole sequence, so the combine pass is skipped
                    reinterpret_cast<elem_t*>(p.o_direct)[b * p.osb + (h_base + row) * p.osh + d] = from_f32<elem_t>(o_val[u]);
                    if (d == 0 && p.lse_direct != nullptr) p.lse_direct[(int64_t)b * p.Hq + h_base + row] = lse_val[u];
                } else if (p.cluster > 1) {
                    xo[idx] = o_val[u];                          // read by the CTAs of this unit's cluster (below)
                    if (d == 0) xl[row] = lse_val[u];
                } else {
                    const int64_t prow = ((int64_t)b * p.Hq + h_base + row) * p.parts + s;
                    p.o_part[prow * kD + d] = o_val[u];
                    if (d == 0) p.lse_part[prow] = lse_val[u];
                }
            }
        }
        if (p.o_direct != nullptr && p.peer.n > 0 && p.peer_vec) {
            // the slice goes to every rank over NVLink as 16-byte stores (512 contiguous bytes per warp instruction): a
            // 2-byte store per thread and peer is an NVLink packet of 64 bytes per warp, mostly header
            named_bar_sync(1, kConsumerWarps * 32);
            const int64_t base_off = p.peer.base() + b * p.osb + h_base * p.osh;
            for (int c = tid; c < rows_here * kD / 8; c += kConsumerWarps * 32) {
                const int row = (c * 8) / kD, d = (c * 8) - row * kD;
                const uint4 v = *reinterpret_cast<const uint4*>(stage_o + c * 8);
                for (int r = 0; r < p.peer.n; ++r)
                    *reinterpret_cast<uint4*>(reinterpret_cast<elem_t*>(p.peer.o[r]) + base_off + row * p.osh + d) = v;
            }
        }
        if (threadIdx.x == 0) PLI_DECODE_TRACE(4);               // output / partial written
        if (p.counters != nullptr && p.parts > 1 && p.cluster == 1) arrive_and_merge();   // (NULL: partials only)
        if (!kMulti && p.gather.n > 0 && p.gather.cta_counter != nullptr) {
            // ---- (option, off: see pli_decode_fwd_gather) the last CTA of the grid to get here publishes this rank's
            // slice and waits for the peers' ----
            named_bar_sync(1, kConsumerWarps * 32);              // every consumer thread's peer stores are issued
            if (warp == 0) {
                uint32_t last = 0;
                if (lane == 0) {
                    __threadfence_system();                      // ... and visible system-wide before this CTA counts
                    last = atomicAdd(p.gather.cta_counter, 1u) == gridDim.x * gridDim.y * gridDim.z - 1u;
                    if (last) {
                        *p.gather.cta_counter = 0u;              // zero for the next launch / graph replay
                        __threadfence_system();                  // acquire side of the other CTAs' fence + arrival
                    }
                }
                last = __shfl_sync(0xffffffffu, last, 0);
                if (last) {
                    if (lane < p.gather.n) {
                        st_release_sys(p.gather.done[lane] + p.gather.rank, step);
                        if (!wait_flag_reaches(p.gather.done[p.gather.rank] + lane, step, p.gather.timeout_ns))
                            record_peer_timeout(p.gather.status, p.gather.rank, lane, step);
                    }
                    __syncwarp();
                    if (lane == 0) *p.gather.epoch = step;       // the step is complete on this rank
                }
            }
        }
    }
    if (p.cluster > 1) {
        // ---- the unit's S = cluster splits merge through distributed shared memory ----
        // Every CTA has left its normalised partial (O, LSE) in its own shared memory (xo / xl).  After the cluster barrier
        // (ALL threads of all CTAs take part, producers included) CTA r merges the r-th slice of the unit's rows_here x kD
        // outputs, reading the S partial values of an element from the S CTAs; a second barrier keeps every CTA's shared
        // memory alive until its neighbours have read it.  Against partials in global memory + arrival atomic + bulk copy
        // this removes two L2 round trips and a device-scope release from the tail of the last CTA.
        cluster_sync_all();
        if (warp < kConsumerWarps) {
            const int C = p.cluster, r = (int)cluster_ctarank();
            const int total = rows_here * kD, per = (total + C - 1) / C;
            const uint32_t xo_addr = smem_u32(smem + kXchgOffset), xl_addr = xo_addr + 16 * kD * 4;
            if (p.gather.n > 0 && p.parts == 1) mbar_wait(peer_ok, 0);
            for (int e = r * per + (int)threadIdx.x; e < min(total, (r + 1) * per); e += kConsumerWarps * 32) {
                const int row = e / kD, d = e - row * kD;
                float lj[8], oj[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    lj[j] = j < C ? ld_shared_cluster_f32(mapa_u32(xl_addr + row * 4, j)) : -INFINITY;
                    oj[j] = j < C ? ld_shared_cluster_f32(mapa_u32(xo_addr + e * 4, j)) : 0.f;
                }
                float M = lj[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) M = fmaxf(M, lj[j]);
                float den = 0.f, o = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float w = lj[j] == -INFINITY ? 0.f : __expf(lj[j] - M);
                    den += w;
                    o = fmaf(w, oj[j], o);
                }
                const float on = den > 0.f ? o / den : 0.f;
                const float ln = den > 0.f ? M + logf(den) : -INFINITY;
                if (p.parts > 1) {
                    // several clusters per unit: this cluster's merged partial goes through the workspace
                    const int64_t prow = ((int64_t)b * p.Hq + h_base + row) * p.parts + blockIdx.x / C;
                    p.o_part[prow * kD + d] = on;
                    if (d == 0) p.lse_part[prow] = ln;
                    continue;
                }
                const elem_t val = from_f32<elem_t>(on);
                const int64_t off = b * p.osb + (h_base + row) * p.osh + d;
                if (p.peer.n > 0) {
                    const int64_t poff = p.peer.base() + off;
                    for (int q = 0; q < p.peer.n; ++q) reinterpret_cast<elem_t*>(p.peer.o[q])[poff] = val;
                } else {
                    reinterpret_cast<elem_t*>(p.o_final)[off] = val;
                }
                if (d == 0 && p.lse_final != nullptr) p.lse_final[(int64_t)b * p.Hq + h_base + row] = ln;
            }
        }
        // (also: the slices of a cluster partial written by the other CTAs happen before rank 0's arrival below)
        cluster_sync_all();
        if (p.counters != nullptr && p.parts > 1 && warp < kConsumerWarps && cluster_ctarank() == 0) arrive_and_merge();
    }
}

// ------------------------------------------------------------------------------------------------
// combine: merge S partials per (b, q head)
// ------------------------------------------------------------------------------------------------
// One CTA per (batch row, q head).  The S partial LSEs are reduced across the lanes of a warp (one or two per lane,
// S <= 64) instead of three serial passes over them, the weights go through shared memory, and the weighted sum over the
// partial outputs keeps eight independent, coalesced loads in flight per thread: with few sequences and many splits
// (B1 x L32768: 37 splits) the old serial loops cost more than the split-KV kernel they followed.
//
// The partials are written by the grid this one is programmatically launched behind: every read of them must stay BEHIND
// griddepcontrol.wait.  They are therefore NOT `const __restrict__` (loads through such pointers are "invariant" and the
// compiler hoisted them above the wait: LDG.E.CONSTANT in front of ACQBULK in the SASS, stale partials for the CTAs that
// were still running — caught by test_paged_decode_tma) and go through ld.global.cg.
template <typename T>
__global__ void __launch_bounds__(128) decode_combine_kernel(const float* o_part, const float* lse_part, T* o, float* lse,
                                                             int Hq, int D, int S, int64_t osb, int64_t osh,
                                                             const PeerScatter peer) {
    __shared__ float sw[64];
    const int h = blockIdx.x, b = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)b * Hq + h) * S;
    pdl_wait();                     // the split-KV grid before this one has completed and its partials are visible
    const float l0 = lane < S ? __ldcg(lse_part + row + lane) : -INFINITY;
    const float l1 = lane + 32 < S ? __ldcg(lse_part + row + lane + 32) : -INFINITY;
    float M = fmaxf(l0, l1);
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o2));
    const float w0 = l0 == -INFINITY ? 0.f : __expf(l0 - M);
    const float w1 = l1 == -INFINITY ? 0.f : __expf(l1 - M);
    float den = w0 + w1;
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o2);
    if (threadIdx.x < 32) {         // every warp computed the same weights; warp 0 publishes them
        sw[lane] = w0;
        sw[lane + 32] = w1;
    }
    __syncthreads();
    const float inv = den > 0.f ? 1.f / den : 0.f;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const float* src = o_part + row * D + d;
        float acc = 0.f;
        int s = 0;
        for (; s + 8 <= S; s += 8) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = __ldcg(src + (int64_t)(s + j) * D);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc = fmaf(sw[s + j], v[j], acc);
        }
        for (; s < S; ++s) acc = fmaf(sw[s], __ldcg(src + (int64_t)s * D), acc);
        const T val = from_f32<T>(acc * inv);
        if (peer.n > 0) {
            const int64_t off = peer.base() + b * osb + h * osh + d;
            for (int r = 0; r < peer.n; ++r) reinterpret_cast<T*>(peer.o[r])[off] = val;
        } else {
            o[b * osb + h * osh + d] = val;
        }
    }
    if (lse != nullptr && threadIdx.x == 0) lse[(int64_t)b * Hq + h] = den > 0.f ? M + logf(den) : -INFINITY;
}

// Runs after the scattering kernel on the same stream (whose peer stores are complete at the kernel boundary).
// Thread r tells rank r that this rank's slice of `epoch` has landed (release, system scope), then spins (acquire)
// until rank r's slice has landed here.  Publishing never waits on anybody, so this cannot deadlock.  A peer that is
// merely late (lazy module load, host GC, a checkpoint, a debugger) is waited for: the bound is wall time
// (pli_set_peer_timeout_ms, 60 s by default, 0 = forever), and when it expires the kernel does NOT trap — it records
// (this rank, the missing rank, the step) in the host-visible fault record, which pli_device_status / PeerOutput.advance
// turn into an error on the host, and lets the stream continue (the step's output is then incomplete).
__global__ void peer_publish_wait_kernel(const PeerFlags pf) {
    const int r = threadIdx.x;
    pdl_wait();                       // launched programmatically behind the storing grid: it is complete and flushed now
    const uint32_t e = *pf.epoch + 1u;
    __syncwarp();
    if (r < pf.n) {
        __threadfence_system();
        st_release_sys(pf.flags[r] + pf.rank, e);
        if (!wait_flag_reaches(pf.flags[pf.rank] + r, e, pf.timeout_ns)) record_peer_timeout(pf.status, pf.rank, r, e);
    }
    __syncwarp();
    if (r == 0) *pf.epoch = e;        // the step is complete on this rank
}

// Copy the output buffer the step that has just completed wrote (parity read from the device step counter) into a
// FIXED destination: under CUDA-graph capture the buffer a replay writes alternates, so a consumer captured in the same
// graph must read from an address that does not (pli_peer_select_copy).
__global__ void __launch_bounds__(256) peer_select_copy_kernel(const uint4* __restrict__ buf0, int64_t buffer_stride_vec,
                                                               const uint32_t* __restrict__ epoch, uint4* __restrict__ dst,
                                                               int64_t n_vec) {
    const uint4* src = buf0 + (int64_t)(*epoch & 1u) * buffer_stride_vec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------------
// KV append + page gather (16-byte vectors when aligned, else elementwise)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void kv_append_kernel(const T* __restrict__ k_new, const T* __restrict__ v_new, T* __restrict__ k_store,
                                 T* __restrict__ v_store, const int32_t* __restrict__ table,
                                 const int32_t* __restrict__ start_pos, int n_new, int Hkv, int D, int bs,
                                 int table_stride, int layer, int64_t nsb, int64_t nst, int64_t nsh, int64_t s_page,
                                 int64_t s_layer, int64_t s_slot, int64_t s_head, int vec) {
    const int b = blockIdx.z, i = blockIdx.y;                    // sequence, new-token index
    const int t = start_pos[b] + i;
    const int per_tok = Hkv * (D / vec);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < per_tok; e += gridDim.x * blockDim.x) {
        const int hk = e / (D / vec), dv = (e - hk * (D / vec)) * vec;
        const int64_t src = b * nsb + i * nst + hk * nsh + dv;
        const int64_t dst = token_offset(table, b, t, bs, table_stride, layer, hk, s_page, s_layer, s_slot, s_head) + dv;
        if (vec * sizeof(T) == 16) {
            *reinterpret_cast<uint4*>(k_store + dst) = *reinterpret_cast<const uint4*>(k_new + src);
            *reinterpret_cast<uint4*>(v_store + dst) = *reinterpret_cast<const uint4*>(v_new + src);
        } else {
            k_store[dst] = k_new[src];
            v_store[dst] = v_new[src];
        }
    }
}

template <typename T>
__global__ void paged_gather_kernel(const T* __restrict__ store, T* __restrict__ out,
                                    const int32_t* __restrict__ table, const int32_t* __restrict__ seq_lens,
                                    int max_len, int Hkv, int D, int bs, int table_stride, int layer, int64_t s_page,
                                    int64_t s_layer, int64_t s_slot, int64_t s_head) {
    const int b = blockIdx.z, t = blockIdx.y;
    const bool live = t < seq_lens[b];
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Hkv * D; e += gridDim.x * blockDim.x) {
        const int hk = e / D, d = e - hk * D;
        T val = from_f32<T>(0.f);
        if (live) val = store[token_offset(table, b, t, bs, table_stride, layer, hk, s_page, s_layer, s_slot, s_head) + d];
        out[(((int64_t)b * max_len + t) * Hkv + hk) * D + d] = val;
    }
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }
int ilog2(int x) { int l = 0; while ((1 << (l + 1)) <= x) ++l; return l; }

// Id of a split-KV launch (see unit_arrive): distinct for distinct launches of this process, never 0.
uint32_t next_launch_id() {
    static std::atomic<uint32_t> id{0x9E3779B9u};
    uint32_t v = id.fetch_add(1u, std::memory_order_relaxed) + 1u;
    return v ? v : id.fetch_add(1u, std::memory_order_relaxed) + 1u;
}

#if defined(PLI_TUNING) && PLI_TUNING
unsigned long long* g_decode_trace = nullptr;   // process-wide, unsynchronised: tuning builds are driven from one thread
int g_decode_trace_cap = 0;
#endif

bool tma_eligible(int D, int dtype, int block_size, bool paged, const int64_t* st, const void* k, const void* v) {
    if (dtype != PLI_BF16 && dtype != PLI_F16) return false;
    if (D != 64 && D != 128) return false;
    if (paged && (!is_pow2(block_size) || block_size < 8 || block_size > 256)) return false;
    if ((reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15) return false;
    // every non-unit stride must be a multiple of 16 bytes (8 elements) for the tensor map
    for (int i = 0; i < 4; ++i)
        if (st[i] % 8 != 0) return false;
    if (st[2] <= 0 || st[3] <= 0 || st[0] <= 0) return false;
    return true;
}

int make_kv_map(CUtensorMap* map, const void* base, int dtype, int D, int Hkv, bool paged, int block_size,
                int num_layers_hint, int64_t extent, int max_seq_len, const int64_t* st, int box_tokens) {
    EncodeTiledFn enc = get_encode_tiled();
    if (enc == nullptr) return set_error(PLI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const CUtensorMapDataType dt = dtype == PLI_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    // dims (fastest first): d, head, slot/token, X (layer | 1), Y (page | batch)
    cuuint64_t dims[5] = {(cuuint64_t)D, (cuuint64_t)Hkv, (cuuint64_t)(paged ? block_size : max_seq_len),
                          (cuuint64_t)(paged ? num_layers_hint : 1), (cuuint64_t)extent};
    const int64_t x_stride = paged ? st[1] : st[0];
    cuuint64_t strides[4] = {(cuuint64_t)st[3] * 2, (cuuint64_t)st[2] * 2, (cuuint64_t)(x_stride > 0 ? x_stride : st[0]) * 2,
                             (cuuint64_t)st[0] * 2};
    cuuint32_t box[5] = {64, 1, (cuuint32_t)box_tokens, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(map, dt, 5, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(PLI_ERR_CUDA, "cuTensorMapEncodeTiled(KV) failed with CUresult %d", (int)r);
    return PLI_OK;
}

template <int kD, bool kBf16, bool kRows16, bool kMulti>
int launch_tma_t(const CUtensorMap& mk, const CUtensorMap& mv, DecodeTmaParams p, dim3 grid, cudaStream_t stream) {
    auto kern = decode_tma_kernel<kD, kBf16, kRows16, kMulti>;
    constexpr int kTileBytes = (kD / 64) * kStageTokens * 128;
    const size_t merge_bytes = (size_t)(128 + 64 * (kD + 8)) * sizeof(float);
    size_t smem = (size_t)2 * kDecodeStages * kTileBytes + 2 * kDecodeStages * sizeof(uint64_t) + 24 + 1024;
    if (smem < merge_bytes + 1024) smem = merge_bytes + 1024;
    PLI_CUDA_CHECK(ensure_dynamic_smem(kern, (int)smem));
    PLI_CUDA_CHECK(bind_status_symbol());
    if (p.cluster > 1) {
        // A grid that fits the GPU in one wave as independent CTAs may not fit as clusters (the CTAs of a cluster need free
        // slots inside one GPC): 288 CTAs in clusters of four ran as two waves, 40.9 us instead of 28.6.  Ask the runtime
        // how many clusters can be resident and merge through the workspace instead when the grid would not fit.
        static int max_active[9] = {0};                     // per cluster size, this kernel instance (benign race: same value)
        if (max_active[p.cluster] == 0) {
            cudaLaunchConfig_t q = {};
            q.gridDim = dim3((unsigned)p.cluster, 1, 1);
            q.blockDim = dim3(kDecodeThreads);
            q.dynamicSmemBytes = smem;
            cudaLaunchAttribute qa[1];
            qa[0].id = cudaLaunchAttributeClusterDimension;
            qa[0].val.clusterDim.x = (unsigned)p.cluster;
            qa[0].val.clusterDim.y = 1;
            qa[0].val.clusterDim.z = 1;
            q.attrs = qa;
            q.numAttrs = 1;
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kern, &q) != cudaSuccess || n <= 0) { (void)cudaGetLastError(); n = -1; }
            max_active[p.cluster] = n;
        }
        const long long ctas = (long long)grid.x * grid.y * grid.z;
        const int sms = sm_count() > 0 ? sm_count() : 148;
        if (max_active[p.cluster] < 0 || (ctas <= 2LL * sms && ctas / p.cluster > max_active[p.cluster])) {
            p.cluster = 1;
            p.parts = p.S;
        }
    }
    {
        // Launched programmatically behind whatever precedes it on the stream: the kernel's first statement is
        // griddepcontrol.wait, so every dependency is kept and only the launch latency is hidden (the grid is resident
        // and waiting when its predecessor ends).  With 2 / 4 / 8 splits per unit the splits of a unit (consecutive
        // blockIdx.x) are one thread-block cluster.
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(kDecodeThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = stream;
        cudaLaunchAttribute attr[2];
        int na = 0;
        if (kDecodePdl) {
            attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[na].val.programmaticStreamSerializationAllowed = 1;
            ++na;
        }
        if (p.cluster > 1) {
            attr[na].id = cudaLaunchAttributeClusterDimension;
            attr[na].val.clusterDim.x = (unsigned)p.cluster;
            attr[na].val.clusterDim.y = 1;
            attr[na].val.clusterDim.z = 1;
            ++na;
        }
        cfg.attrs = attr;
        cfg.numAttrs = na;
        PLI_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, mk, mv, p));
    }
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

}  // namespace

cudaError_t bind_status_decode() { return bind_status_symbol(); }

}  // namespace pli

using namespace pli;

// Tuning builds: 16 x uint64 per CTA of the next TMA split-KV launches: SM clock stamps (0 start, 1 first loads issued,
// 2 first stage landed, 3 last stage consumed, 4 output / partial written, 5 merged output written, 8-11 last stage
// consumed by consumer warp 0-3, 12 barriers initialised, 13 first page ids known, 14 / 15 first / second barrier of the
// cross-warp merge passed) and, in word 7, the %globaltimer at the start (to place CTAs against each other); (NULL, 0)
// switches it off.  tools/decode_trace.py.
extern "C" int pli_debug_decode_trace(void* buf, int cap_ctas) {
#if defined(PLI_TUNING) && PLI_TUNING
    g_decode_trace = static_cast<unsigned long long*>(buf);
    g_decode_trace_cap = buf ? cap_ctas : 0;
    return PLI_OK;
#else
    (void)buf; (void)cap_ctas;
    return set_error(PLI_ERR_UNSUPPORTED, "pli_debug_decode_trace is compiled into tuning builds only");
#endif
}

extern "C" int pli_decode_num_splits(int B, int Hkv, int max_seq_len) {
    if (B <= 0 || Hkv <= 0 || max_seq_len <= 0) return 1;
    // The kernel is HBM-bound: what matters is enough bytes in flight (2 resident CTAs x 96 KB per SM),
    // not wave count, and every extra split costs a pipeline fill plus combine traffic (measured on C3:
    // 1 split 6.2 TB/s, 3 splits 5.5 TB/s).  So split only until one full wave of CTAs exists, with at
    // least 256 tokens per split.
    const int64_t units = (int64_t)B * Hkv;
    const int sms = sm_count() > 0 ? sm_count() : 148;
    const int64_t target = (int64_t)sms * (PLI_DECODE_STAGES > 3 ? 1 : 2);
    // floor: 256 units on 296 CTA slots stay unsplit (measured B256/Hkv1/L1k: 1 split 34.5 us, 2 splits 41.9 us)
    int by_fill = (int)(target / units);
    int by_len = (max_seq_len + 255) / 256;
    int s = by_fill < by_len ? by_fill : by_len;
    if (s < 1) s = 1;
    if (s > 64) s = 64;
    // more than eight splits: a multiple of eight, so that eight at a time merge inside a thread-block cluster (through
    // distributed shared memory) and only s / 8 partials per unit go through the workspace
    if (s > 8) s &= ~7;
    return s;
}

// Workspace: [B*Hq*S*D] partial outputs (f32), [B*Hq*S] partial LSEs (f32), then -- 8-byte aligned -- B*Hq arrival counter
// pairs (one per (b, kv head, 16-row chunk) is used) for the combine fused into the split-KV kernel.  Nothing needs
// initialising (unit_arrive).
static size_t partials_bytes(int B, int Hq, int D, int num_splits) {
    return (((size_t)B * Hq * num_splits * (size_t)(D + 1) * sizeof(float)) + 7) & ~(size_t)7;
}
extern "C" size_t pli_decode_workspace_bytes(int B, int Hq, int D, int num_splits) {
    if (B <= 0 || Hq <= 0 || D <= 0 || num_splits <= 0) return 0;
    return partials_bytes(B, Hq, D, num_splits) + (size_t)B * Hq * 2 * sizeof(unsigned long long);
}

extern "C" int pli_decode_kernel_kind(int D, int dtype, int block_size, const int64_t kv_strides[4], const void* k_store,
                                      const void* v_store) {
    return tma_eligible(D, dtype, block_size, block_size > 0, kv_strides, k_store, v_store) ? PLI_KIND_MMA_TMA
                                                                                          : PLI_KIND_SIMT;
}

static int check_decode_args(const void* q, const void* k, const void* v, const int32_t* seq_lens, int B, int Hq, int Hkv,
                             int D, int max_seq_len, int block_size, bool paged, int num_splits) {
    if (!q || !k || !v || !seq_lens) return set_error(PLI_ERR_INVALID, "null pointer argument");
    if (B <= 0 || Hq <= 0 || Hkv <= 0 || D <= 0) return set_error(PLI_ERR_INVALID, "non-positive dimension");
    if (Hq % Hkv != 0) return set_error(PLI_ERR_INVALID, "Hq (%d) must be a multiple of Hkv (%d)", Hq, Hkv);
    if (D > 256) return set_error(PLI_ERR_UNSUPPORTED, "head_dim %d > 256", D);
    if (max_seq_len <= 0) return set_error(PLI_ERR_INVALID, "max_seq_len must be positive");
    if (paged && block_size <= 0) return set_error(PLI_ERR_INVALID, "block_size must be positive for paged KV");
    if (num_splits <= 0 || num_splits > 64) return set_error(PLI_ERR_INVALID, "num_splits must be in [1, 64]");
    if (B > 65535) return set_error(PLI_ERR_UNSUPPORTED, "B > 65535");
    return PLI_OK;
}

#ifndef PLI_CLUSTER_MERGE
#define PLI_CLUSTER_MERGE 1
#endif
static constexpr bool kClusterMerge = PLI_CLUSTER_MERGE != 0;
#ifndef PLI_PUBLISH_FROM_LAST_CTA
#define PLI_PUBLISH_FROM_LAST_CTA 0
#endif
static constexpr bool kPublishFromLastCta = PLI_PUBLISH_FROM_LAST_CTA != 0;

// The TMA + mma.sync kernel serves this call (else: the SIMT kernel).
static bool tma_path_ok(const void* q, const void* k_store, const void* v_store, int D, int dtype, int block_size, bool paged,
                        const int64_t q_strides[2], const int64_t kv_strides[4], float scale) {
    return scale > 0.f && tma_eligible(D, dtype, block_size, paged, kv_strides, k_store, v_store) && (q_strides[0] % 2 == 0) &&
           (q_strides[1] % 2 == 0) && ((reinterpret_cast<uintptr_t>(q) & 3) == 0);
}

// Split-KV launch.  When o_direct is given, num_splits == 1 and the TMA kernel serves the request,
// the kernel writes the final output itself and *wrote_direct is set (the combine pass is not needed).
static int splitkv_impl(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                        const int32_t* seq_lens, int B, int Hq, int Hkv, int D, int max_seq_len, int block_size,
                        int table_stride, int layer, int64_t kv_extent, const int64_t q_strides[2],
                        const int64_t kv_strides[4], float scale, int dtype, int num_splits, void* workspace,
                        size_t workspace_bytes, cudaStream_t stream, void* o_direct, float* lse_direct,
                        const int64_t* o_strides, bool* wrote_direct, const PeerScatter* peer = nullptr,
                        const PeerGather* gather = nullptr, int q_len = 1, int64_t q_tok_stride = 0) {
    // q_len > 1 (pli_decode_fwd_multi): Hq counts virtual heads (q head * q_len + token); q_strides are q's {batch, head}
    // with q_tok_stride its token stride, o_strides are {batch, virtual head}
    const bool paged = block_table != nullptr;
    if (num_splits == 0) num_splits = pli_decode_num_splits(B, Hkv, max_seq_len);
    int rc = check_decode_args(q, k_store, v_store, seq_lens, B, Hq, Hkv, D, max_seq_len, block_size, paged, num_splits);
    if (rc) return rc;
    if (workspace == nullptr || workspace_bytes < pli_decode_workspace_bytes(B, Hq, D, num_splits))
        return set_error(PLI_ERR_INVALID, "workspace too small: need %zu bytes",
                         pli_decode_workspace_bytes(B, Hq, D, num_splits));
    if (reinterpret_cast<uintptr_t>(workspace) & 15)      // the merge bulk-copies partials out of it; counters are 8-byte words
        return set_error(PLI_ERR_INVALID, "workspace must be 16-byte aligned");
    float* o_part = static_cast<float*>(workspace);
    float* lse_part = o_part + (size_t)B * Hq * num_splits * D;
    const int G = Hq / Hkv;

    if (tma_path_ok(q, k_store, v_store, D, dtype, block_size, paged, q_strides, kv_strides, scale) &&
        (q_len == 1 || q_tok_stride % 2 == 0)) {
        const int box_tokens = paged ? (block_size < kStageTokens ? block_size : kStageTokens) : kStageTokens;
        // layers extent: the layer coordinate must be inside the tensor; layer+1 is a safe lower bound
        CUtensorMap mk, mv;
        rc = make_kv_map(&mk, k_store, dtype, D, Hkv, paged, block_size, layer + 1, kv_extent, max_seq_len, kv_strides,
                         box_tokens);
        if (rc) return rc;
        rc = make_kv_map(&mv, v_store, dtype, D, Hkv, paged, block_size, layer + 1, kv_extent, max_seq_len, kv_strides,
                         box_tokens);
        if (rc) return rc;
        DecodeTmaParams p;
#if defined(PLI_TUNING) && PLI_TUNING
        p.trace = g_decode_trace;
        p.trace_cap = g_decode_trace_cap;
#else
        p.trace = nullptr;
        p.trace_cap = 0;
#endif
        p.q = q;
        p.table = block_table;
        p.seq_lens = seq_lens;
        p.o_part = o_part;
        p.lse_part = lse_part;
        // with an output given, this one launch produces it: a single split writes it straight away, several splits are
        // merged by the last CTA of each unit to arrive (fused combine)
        const bool direct = o_direct != nullptr && num_splits == 1;
        const bool fused = o_direct != nullptr && num_splits > 1 && num_splits <= 64;
        p.o_direct = direct ? o_direct : nullptr;
        p.lse_direct = direct ? lse_direct : nullptr;
        p.osb = (direct || fused) ? o_strides[0] : 0;
        p.osh = (direct || fused) ? o_strides[1] : 0;
        p.counters = fused ? reinterpret_cast<unsigned long long*>(static_cast<char*>(workspace) +
                                                                    partials_bytes(B, Hq, D, num_splits))
                           : nullptr;
        p.launch_id = next_launch_id();
        p.o_final = fused ? o_direct : nullptr;
        p.lse_final = fused ? lse_direct : nullptr;
        p.peer_vec = 0;
        if ((direct || fused) && peer != nullptr) {
            bool ok = o_strides[0] % 8 == 0 && o_strides[1] % 8 == 0 && peer->slice_offset % 8 == 0 &&
                      peer->buffer_stride % 8 == 0 && D % 8 == 0;
            for (int r = 0; r < peer->n; ++r) ok = ok && (reinterpret_cast<uintptr_t>(peer->o[r]) & 15) == 0;
            p.peer_vec = ok ? 1 : 0;
        }
        p.gather = PeerGather{};
        if ((direct || fused) && peer != nullptr && gather != nullptr) p.gather = *gather;
        // 2, 4 or 8 splits: one thread-block cluster per unit, merged through distributed shared memory
        p.cluster = 1;
        if (fused && kClusterMerge) p.cluster = num_splits % 8 == 0 ? 8 : num_splits % 4 == 0 ? 4 : num_splits % 2 == 0 ? 2 : 1;
        p.parts = fused ? num_splits / p.cluster : num_splits;
        if (wrote_direct) *wrote_direct = direct || fused;
        p.qsb = q_strides[0];
        p.qsh = q_strides[1];
        p.qst = q_tok_stride;
        p.Hq = Hq;
        p.Hkv = Hkv;
        p.G = G;
        p.bs = paged ? block_size : 1;
        p.table_stride = table_stride;
        p.layer = layer;
        p.S = num_splits;
        p.box_tokens = box_tokens;
        p.max_len = max_seq_len;
        p.q_len = q_len;
        p.bs_shift = ilog2(p.bs);
        p.box_shift = ilog2(box_tokens);
        p.fd_splits = make_fastdiv((uint32_t)num_splits);
        p.scale_log2 = scale * kLog2e;
        p.peer = PeerScatter{};
        if ((direct || fused) && peer != nullptr) p.peer = *peer;
        const int hchunks = (G + 15) / 16;
        dim3 grid(num_splits, Hkv * hchunks, B);
        const bool rows16 = G > 8;
        const bool bf16 = dtype == PLI_BF16;
#define PLI_GO(DD, BF, R16)                                                                                         \
    return q_len > 1 ? launch_tma_t<DD, BF, R16, true>(mk, mv, p, grid, stream)                                   \
                     : launch_tma_t<DD, BF, R16, false>(mk, mv, p, grid, stream)
        if (D == 128) {
            if (bf16) { if (rows16) PLI_GO(128, true, true); else PLI_GO(128, true, false); }
            else      { if (rows16) PLI_GO(128, false, true); else PLI_GO(128, false, false); }
        } else {
            if (bf16) { if (rows16) PLI_GO(64, true, true); else PLI_GO(64, true, false); }
            else      { if (rows16) PLI_GO(64, false, true); else PLI_GO(64, false, false); }
        }
#undef PLI_GO
    }

    // generic SIMT path
    if (Hq > 65535) return set_error(PLI_ERR_UNSUPPORTED, "Hq > 65535");
    const int dc = (D + 31) / 32;
    dim3 grid(num_splits, Hq, B);
    const size_t smem = (size_t)4 * D * sizeof(float);
    const int bs = paged ? block_size : 1;
#define PLI_SIMT(T, N)                                                                                              \
    decode_simt_kernel<T, N><<<grid, 128, smem, stream>>>(                                                          \
        (const T*)q, (const T*)k_store, (const T*)v_store, block_table, seq_lens, Hq, Hkv, D, bs, table_stride,     \
        layer, q_strides[0], q_strides[1], kv_strides[0], kv_strides[1], kv_strides[2], kv_strides[3], scale,       \
        num_splits, o_part, lse_part, q_len, q_tok_stride)
#define PLI_SIMT_D(T)                   \
    if (dc <= 1) PLI_SIMT(T, 1);        \
    else if (dc <= 2) PLI_SIMT(T, 2);   \
    else if (dc <= 4) PLI_SIMT(T, 4);   \
    else PLI_SIMT(T, 8)
    if (dtype == PLI_F32) { PLI_SIMT_D(float); }
    else if (dtype == PLI_BF16) { PLI_SIMT_D(__nv_bfloat16); }
    else if (dtype == PLI_F16) { PLI_SIMT_D(__half); }
    else return set_error(PLI_ERR_INVALID, "unknown dtype %d", dtype);
#undef PLI_SIMT_D
#undef PLI_SIMT
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

extern "C" int pli_decode_splitkv(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                                  const int32_t* seq_lens, int B, int Hq, int Hkv, int D, int max_seq_len, int block_size,
                                  int table_stride, int layer, int64_t kv_extent, const int64_t q_strides[2],
                                  const int64_t kv_strides[4], float scale, int dtype, int num_splits, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    return splitkv_impl(q, k_store, v_store, block_table, seq_lens, B, Hq, Hkv, D, max_seq_len, block_size, table_stride,
                        layer, kv_extent, q_strides, kv_strides, scale, dtype, num_splits, workspace, workspace_bytes,
                        static_cast<cudaStream_t>(stream), nullptr, nullptr, nullptr, nullptr);
}

// Tuning builds (-DPLI_TUNING=1): PLI_NO_PDL=1 in the environment launches the combine pass as a plain stream-ordered
// kernel (A/B measurements).  The product build always uses the programmatic dependent launch.
#if defined(PLI_TUNING) && PLI_TUNING
static bool pdl_enabled() {
    static const bool on = [] {
        const char* e = getenv("PLI_NO_PDL");
        return !(e && e[0] == '1');
    }();
    return on;
}
#else
static constexpr bool pdl_enabled() { return true; }
#endif

static int combine_impl(const void* workspace, void* o, float* lse, int B, int Hq, int D, int num_splits,
                        const int64_t o_strides[2], int dtype, void* stream_, const PeerScatter& peer) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!workspace || (!o && peer.n == 0)) return set_error(PLI_ERR_INVALID, "null pointer argument");
    if (B <= 0 || Hq <= 0 || D <= 0 || num_splits <= 0) return set_error(PLI_ERR_INVALID, "non-positive dimension");
    if (B > 65535) return set_error(PLI_ERR_UNSUPPORTED, "B > 65535");
    const float* o_part = static_cast<const float*>(workspace);
    const float* lse_part = o_part + (size_t)B * Hq * num_splits * D;
    const int threads = D >= 128 ? 128 : (D >= 64 ? 64 : 32);
    // programmatic dependent launch behind the split-KV kernel on the same stream (the kernel waits in pdl_wait())
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(Hq, B);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const int64_t osb = o_strides[0], osh = o_strides[1];
    if (dtype == PLI_F32)
        PLI_CUDA_CHECK(cudaLaunchKernelEx(&cfg, decode_combine_kernel<float>, o_part, lse_part, (float*)o, lse, Hq, D, num_splits, osb, osh, peer));
    else if (dtype == PLI_BF16)
        PLI_CUDA_CHECK(cudaLaunchKernelEx(&cfg, decode_combine_kernel<__nv_bfloat16>, o_part, lse_part, (__nv_bfloat16*)o, lse, Hq, D, num_splits, osb, osh, peer));
    else if (dtype == PLI_F16)
        PLI_CUDA_CHECK(cudaLaunchKernelEx(&cfg, decode_combine_kernel<__half>, o_part, lse_part, (__half*)o, lse, Hq, D, num_splits, osb, osh, peer));
    else
        return set_error(PLI_ERR_INVALID, "unknown dtype %d", dtype);
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

extern "C" int pli_decode_combine(const void* workspace, void* o, float* lse, int B, int Hq, int D, int num_splits,
                                  const int64_t o_strides[2], int dtype, void* stream) {
    return combine_impl(workspace, o, lse, B, Hq, D, num_splits, o_strides, dtype, stream, PeerScatter{});
}

extern "C" int pli_decode_fwd_scatter(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                                      const int32_t* seq_lens, float* lse, int B, int Hq, int Hkv, int D, int max_seq_len,
                                      int block_size, int table_stride, int layer, int64_t kv_extent,
                                      const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                                      float scale, int dtype, int num_splits, void* workspace, size_t workspace_bytes,
                                      const pli_peer_scatter* ps, void* stream) {
    if (!ps || !o_strides) return set_error(PLI_ERR_INVALID, "null peer-scatter argument");
    if (ps->n_peers < 1 || ps->n_peers > PLI_MAX_PEERS) return set_error(PLI_ERR_INVALID, "n_peers must be in [1, %d]", PLI_MAX_PEERS);
    if (ps->rank < 0 || ps->rank >= ps->n_peers) return set_error(PLI_ERR_INVALID, "rank outside [0, n_peers)");
    PeerScatter peer{};
    for (int r = 0; r < ps->n_peers; ++r) {
        if (!ps->peer_o[r]) return set_error(PLI_ERR_INVALID, "null peer pointer for rank %d", r);
        peer.o[r] = ps->peer_o[r];
    }
    if (!ps->epoch) return set_error(PLI_ERR_INVALID, "null epoch word");
    peer.n = ps->n_peers;
    peer.epoch = ps->epoch;
    peer.buffer_stride = ps->buffer_stride;
    peer.slice_offset = ps->slice_offset;
    if (num_splits == 0) num_splits = pli_decode_num_splits(B, Hkv, max_seq_len);
    bool wrote_direct = false;
    // o_direct only selects the direct path; with a peer table the kernel never dereferences it
    int rc = splitkv_impl(q, k_store, v_store, block_table, seq_lens, B, Hq, Hkv, D, max_seq_len, block_size, table_stride,
                          layer, kv_extent, q_strides, kv_strides, scale, dtype, num_splits, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), ps->peer_o[ps->rank], lse, o_strides, &wrote_direct, &peer);
    if (rc) return rc;
    if (wrote_direct) return PLI_OK;
    return combine_impl(workspace, nullptr, lse, B, Hq, D, num_splits, o_strides, dtype, stream, peer);
}

extern "C" int pli_decode_fwd_gather(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                                     const int32_t* seq_lens, float* lse, int B, int Hq, int Hkv, int D, int max_seq_len,
                                     int block_size, int table_stride, int layer, int64_t kv_extent,
                                     const int64_t q_strides[2], const int64_t kv_strides[4], const int64_t o_strides[2],
                                     float scale, int dtype, int num_splits, void* workspace, size_t workspace_bytes,
                                     const pli_peer_scatter* ps, void* stream) {
    if (!ps || !o_strides || !q_strides || !kv_strides) return set_error(PLI_ERR_INVALID, "null argument");
    if (ps->n_peers < 1 || ps->n_peers > PLI_MAX_PEERS) return set_error(PLI_ERR_INVALID, "n_peers must be in [1, %d]", PLI_MAX_PEERS);
    if (ps->rank < 0 || ps->rank >= ps->n_peers) return set_error(PLI_ERR_INVALID, "rank outside [0, n_peers)");
    if (!ps->epoch || (kPublishFromLastCta && !ps->cta_counter))
        return set_error(PLI_ERR_INVALID, "null epoch / cta_counter word");
    if (ps->buffer_stride != 0)
        return set_error(PLI_ERR_INVALID, "the single-launch gather writes ONE buffer per rank: buffer_stride must be 0");
    if (!tma_path_ok(q, k_store, v_store, D, dtype, block_size, block_table != nullptr, q_strides, kv_strides, scale))
        return set_error(PLI_ERR_UNSUPPORTED, "this storage is served by the SIMT kernel: use pli_decode_fwd_scatter + "
                                              "pli_peer_publish_wait (two buffers)");
    PeerScatter peer{};
    PeerGather gather{};
    for (int r = 0; r < ps->n_peers; ++r) {
        if (!ps->peer_o[r] || !ps->peer_flags[r] || !ps->peer_ready[r])
            return set_error(PLI_ERR_INVALID, "null peer pointer for rank %d", r);
        peer.o[r] = ps->peer_o[r];
        gather.done[r] = ps->peer_flags[r];
        gather.ready[r] = ps->peer_ready[r];
    }
    peer.n = gather.n = ps->n_peers;
    peer.epoch = gather.epoch = ps->epoch;
    peer.buffer_stride = 0;
    peer.slice_offset = ps->slice_offset;
    // Publishing from the decode grid itself (its last CTA, found with a counter) needs a system-scope fence in EVERY CTA
    // before it counts -- ~2.5 us during which the CTA keeps its SM slot; on a 1024-CTA grid that cost 27 us against 23 for
    // the NCCL all-gather (2 GPUs, C5 ctx 1024).  The grid boundary is the cheaper fence: the one-warp publish / wait
    // kernel is launched programmatically behind the decode grid (resident and waiting in griddepcontrol.wait when it
    // ends), so a step is still one call and its second launch costs no launch latency.
    gather.cta_counter = kPublishFromLastCta ? ps->cta_counter : nullptr;
    gather.rank = ps->rank;
    gather.timeout_ns = peer_timeout_ns();
    gather.status = status_words();
    if (num_splits == 0) num_splits = pli_decode_num_splits(B, Hkv, max_seq_len);
    bool wrote_direct = false;
    int rc = splitkv_impl(q, k_store, v_store, block_table, seq_lens, B, Hq, Hkv, D, max_seq_len, block_size, table_stride,
                          layer, kv_extent, q_strides, kv_strides, scale, dtype, num_splits, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), ps->peer_o[ps->rank], lse, o_strides, &wrote_direct, &peer,
                          &gather);
    if (rc) return rc;
    if (!wrote_direct) return set_error(PLI_ERR_UNSUPPORTED, "internal: the gather launch did not take the fused path");
    if (kPublishFromLastCta) return PLI_OK;
    PeerFlags pf{};
    for (int r = 0; r < ps->n_peers; ++r) pf.flags[r] = ps->peer_flags[r];
    pf.n = ps->n_peers;
    pf.rank = ps->rank;
    pf.epoch = ps->epoch;
    pf.timeout_ns = peer_timeout_ns();
    pf.status = status_words();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(32);
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    PLI_CUDA_CHECK(cudaLaunchKernelEx(&cfg, peer_publish_wait_kernel, pf));
    count_launch();
    return PLI_OK;
}

extern "C" int pli_peer_publish_wait(const pli_peer_scatter* ps, void* stream) {
    if (!ps) return set_error(PLI_ERR_INVALID, "null peer-scatter argument");
    if (ps->n_peers < 1 || ps->n_peers > PLI_MAX_PEERS) return set_error(PLI_ERR_INVALID, "n_peers must be in [1, %d]", PLI_MAX_PEERS);
    if (ps->rank < 0 || ps->rank >= ps->n_peers) return set_error(PLI_ERR_INVALID, "rank outside [0, n_peers)");
    PeerFlags pf{};
    for (int r = 0; r < ps->n_peers; ++r) {
        if (!ps->peer_flags[r]) return set_error(PLI_ERR_INVALID, "null flag pointer for rank %d", r);
        pf.flags[r] = ps->peer_flags[r];
    }
    if (!ps->epoch) return set_error(PLI_ERR_INVALID, "null epoch word");
    pf.n = ps->n_peers;
    pf.rank = ps->rank;
    pf.epoch = ps->epoch;
    pf.timeout_ns = peer_timeout_ns();
    pf.status = status_words();
    peer_publish_wait_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(pf);
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

extern "C" int pli_peer_select_copy(const pli_peer_scatter* ps, void* dst, int64_t nbytes, int elem_size, void* stream) {
    if (!ps || !dst) return set_error(PLI_ERR_INVALID, "null argument");
    if (ps->rank < 0 || ps->rank >= ps->n_peers || ps->n_peers > PLI_MAX_PEERS) return set_error(PLI_ERR_INVALID, "bad rank");
    if (!ps->epoch || !ps->peer_o[ps->rank]) return set_error(PLI_ERR_INVALID, "null epoch word / output pointer");
    if (nbytes <= 0 || nbytes % 16 || elem_size <= 0 || (ps->buffer_stride * elem_size) % 16 ||
        ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(ps->peer_o[ps->rank])) & 15))
        return set_error(PLI_ERR_INVALID, "peer_select_copy needs 16-byte aligned buffers and sizes");
    const int64_t n_vec = nbytes / 16;
    int64_t blocks = (n_vec + 255) / 256;
    const int64_t cap = (int64_t)(sm_count() > 0 ? sm_count() : 148) * 8;
    if (blocks > cap) blocks = cap;
    peer_select_copy_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint4*>(ps->peer_o[ps->rank]), ps->buffer_stride * elem_size / 16, ps->epoch,
        static_cast<uint4*>(dst), n_vec);
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

extern "C" int pli_decode_fwd(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                              const int32_t* seq_lens, void* o, float* lse, int B, int Hq, int Hkv, int D, int max_seq_len,
                              int block_size, int table_stride, int layer, int64_t kv_extent, const int64_t q_strides[2],
                              const int64_t kv_strides[4], const int64_t o_strides[2], float scale, int dtype,
                              int num_splits, void* workspace, size_t workspace_bytes, void* stream) {
    if (num_splits == 0) num_splits = pli_decode_num_splits(B, Hkv, max_seq_len);
    if (!o || !o_strides) return set_error(PLI_ERR_INVALID, "null output argument");
    bool wrote_direct = false;
    int rc = splitkv_impl(q, k_store, v_store, block_table, seq_lens, B, Hq, Hkv, D, max_seq_len, block_size, table_stride,
                          layer, kv_extent, q_strides, kv_strides, scale, dtype, num_splits, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), o, lse, o_strides, &wrote_direct);
    if (rc) return rc;
    if (wrote_direct) return PLI_OK;
    return combine_impl(workspace, o, lse, B, Hq, D, num_splits, o_strides, dtype, stream, PeerScatter{});
}

// Split count of pli_decode_fwd_multi: the units of its TMA grid are (b, kv head, 16-row chunk of the G * q_len rows of a
// KV head); with q_len == 1 this is pli_decode_num_splits(B, Hkv, max_seq_len), the choice of pli_decode_fwd.
extern "C" int pli_decode_num_splits_multi(int B, int Hq, int Hkv, int q_len, int max_seq_len) {
    if (Hq <= 0 || Hkv <= 0 || q_len <= 1) return pli_decode_num_splits(B, Hkv, max_seq_len);
    return pli_decode_num_splits(B, Hkv * ((Hq / Hkv * q_len + 15) / 16), max_seq_len);
}

// q_len tokens per sequence: the q_len rows of a q head are virtual heads h * q_len + i of a (B, Hq * q_len, D) problem,
// so every layer of the one-token launch (GQA map v / (G * q_len) == h / G, partials, LSE layout, fused / cluster /
// two-pass merges) serves it unchanged; the kernels add the per-row causal limit and read row v of q at head v / q_len,
// token v % q_len through q's own strides.  The output is written through the virtual head stride, hence o's layout rule.
extern "C" int pli_decode_fwd_multi(const void* q, const void* k_store, const void* v_store, const int32_t* block_table,
                                    const int32_t* seq_lens, void* o, float* lse, int B, int Hq, int Hkv, int q_len, int D,
                                    int max_seq_len, int block_size, int table_stride, int layer, int64_t kv_extent,
                                    const int64_t q_strides[3], const int64_t kv_strides[4], const int64_t o_strides[3],
                                    float scale, int dtype, int num_splits, void* workspace, size_t workspace_bytes,
                                    void* stream) {
    if (!o || !q_strides || !o_strides || !kv_strides) return set_error(PLI_ERR_INVALID, "null output / stride argument");
    if (q_len < 1) return set_error(PLI_ERR_INVALID, "q_len must be positive, got %d", q_len);
    if (q_len > 16)
        return set_error(PLI_ERR_UNSUPPORTED, "decode takes at most 16 query tokens per sequence, got %d "
                                              "(use pli_prefill_paged_fwd / pli_prefill_fwd for longer chunks)", q_len);
    if (Hq <= 0 || Hkv <= 0 || Hq % Hkv != 0) return set_error(PLI_ERR_INVALID, "Hq (%d) must be a positive multiple of Hkv (%d)", Hq, Hkv);
    if (q_len > 1 && Hq > 1 && o_strides[1] != q_len * o_strides[2])
        return set_error(PLI_ERR_INVALID, "o needs head stride == q_len * token stride (a (B, Hq, q_len, D) tensor "
                                          "contiguous in its last three dimensions)");
    if ((int64_t)Hq * q_len > 65535) return set_error(PLI_ERR_UNSUPPORTED, "Hq * q_len > 65535");
    const int Hv = Hq * q_len;
    const int64_t os[2] = {o_strides[0], q_len > 1 ? o_strides[2] : o_strides[1]};
    if (num_splits == 0) num_splits = pli_decode_num_splits_multi(B, Hq, Hkv, q_len, max_seq_len);
    bool wrote_direct = false;
    int rc = splitkv_impl(q, k_store, v_store, block_table, seq_lens, B, Hv, Hkv, D, max_seq_len, block_size, table_stride,
                          layer, kv_extent, q_strides, kv_strides, scale, dtype, num_splits, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), o, lse, os, &wrote_direct, nullptr, nullptr, q_len,
                          q_strides[2]);
    if (rc) return rc;
    if (wrote_direct) return PLI_OK;
    return combine_impl(workspace, o, lse, B, Hv, D, num_splits, os, dtype, stream, PeerScatter{});
}

extern "C" int pli_kv_append(const void* k_new, const void* v_new, void* k_store, void* v_store, const int32_t* block_table,
                             const int32_t* start_pos, int B, int n_new, int Hkv, int D, int block_size, int table_stride,
                             int layer, const int64_t new_strides[3], const int64_t kv_strides[4], int dtype, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!k_new || !v_new || !k_store || !v_store || !start_pos) return set_error(PLI_ERR_INVALID, "null pointer argument");
    if (B <= 0 || Hkv <= 0 || D <= 0 || n_new < 0) return set_error(PLI_ERR_INVALID, "bad dimension");
    if (n_new == 0) return PLI_OK;
    if (B > 65535 || n_new > 65535) return set_error(PLI_ERR_UNSUPPORTED, "B and n_new must be <= 65535");
    const bool paged = block_table != nullptr;
    if (paged && block_size <= 0) return set_error(PLI_ERR_INVALID, "block_size must be positive for paged KV");
    const int esz = dtype == PLI_F32 ? 4 : 2;
    int vec = 16 / esz;
    auto aligned = [&](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    bool ok = D % vec == 0 && aligned(k_new) && aligned(v_new) && aligned(k_store) && aligned(v_store);
    for (int i = 0; i < 3; ++i) ok = ok && new_strides[i] % vec == 0;
    for (int i = 0; i < 4; ++i) ok = ok && kv_strides[i] % vec == 0;
    if (!ok) vec = 1;
    const int per_tok = Hkv * (D / vec);
    dim3 grid((per_tok + 127) / 128, n_new, B);
    const int bs = paged ? block_size : 1;
#define PLI_APPEND(T)                                                                                                 \
    kv_append_kernel<T><<<grid, 128, 0, stream>>>((const T*)k_new, (const T*)v_new, (T*)k_store, (T*)v_store,         \
                                                  block_table, start_pos, n_new, Hkv, D, bs, table_stride, layer,     \
                                                  new_strides[0], new_strides[1], new_strides[2], kv_strides[0],      \
                                                  kv_strides[1], kv_strides[2], kv_strides[3], vec)
    if (dtype == PLI_F32) PLI_APPEND(float);
    else if (dtype == PLI_BF16) PLI_APPEND(__nv_bfloat16);
    else if (dtype == PLI_F16) PLI_APPEND(__half);
    else return set_error(PLI_ERR_INVALID, "unknown dtype %d", dtype);
#undef PLI_APPEND
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}

extern "C" int pli_paged_gather(const void* store, void* out, const int32_t* block_table, const int32_t* seq_lens, int B,
                                int max_len, int Hkv, int D, int block_size, int table_stride, int layer,
                                const int64_t kv_strides[4], int dtype, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!store || !out || !seq_lens) return set_error(PLI_ERR_INVALID, "null pointer argument");
    if (B <= 0 || max_len <= 0 || Hkv <= 0 || D <= 0) return set_error(PLI_ERR_INVALID, "non-positive dimension");
    if (B > 65535 || max_len > 65535) return set_error(PLI_ERR_UNSUPPORTED, "B and max_len must be <= 65535");
    const bool paged = block_table != nullptr;
    if (paged && block_size <= 0) return set_error(PLI_ERR_INVALID, "block_size must be positive for paged KV");
    dim3 grid((Hkv * D + 255) / 256, max_len, B);
    const int bs = paged ? block_size : 1;
#define PLI_GATHER(T)                                                                                              \
    paged_gather_kernel<T><<<grid, 256, 0, stream>>>((const T*)store, (T*)out, block_table, seq_lens, max_len, Hkv, D, bs, \
                                                     table_stride, layer, kv_strides[0], kv_strides[1], kv_strides[2],  \
                                                     kv_strides[3])
    if (dtype == PLI_F32) PLI_GATHER(float);
    else if (dtype == PLI_BF16) PLI_GATHER(__nv_bfloat16);
    else if (dtype == PLI_F16) PLI_GATHER(__half);
    else return set_error(PLI_ERR_INVALID, "unknown dtype %d", dtype);
#undef PLI_GATHER
    PLI_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return PLI_OK;
}
