// engine.cu -- B200 (sm_100a) pileup engine: device buffers, the read stage,
// the column stage and the C ABI declared in include/b200_pileup.h.
//
// Data layout in HBM (one staged batch = the reads of one reference sequence
// overlapping one window, grouped by input file, file order kept):
//   raw SoA     pos i64 | flag u16 | mapq u8 | l_qseq i32 | n_cigar u32 |
//               cigar_off u64 | qual_off u64 | mtid i32 | mpos i64 | isize i64 |
//               prev_same_name i64 | rbits u8          (one array per field)
//   payload     cigar u32[] | seq4 u8[] (4-bit) | qual u8[] | ref char[]
//   derived     ReadDesc[32 B] per read, prefix-max of read ends, per-32-column
//               [lo,hi) read ranges, entry strings (2 B per read base), look-back status words, output text
//
// Column stage for text (mpileup, depth): sizes -> offsets -> bytes, no inter-CTA waiting.
//   (1) sizes.  mpileup, one input file (the default path, mpileup_ent.cuh / mpileup_ss.cuh): a READ-major entry pass formats
//       every read into 16-bit entries (eight bases per lane, SIMD within a register) and feeds order-free line-length sums
//       (coverage difference array, failing bases, extra bytes); a scan + a per-column kernel turn them into line lengths.
//       General mpileup path (several files, -O, host string columns) and depth: thread per column.
//   (2) a single-pass scan of 128-column tile totals gives every tile its byte offset;
//   (3) bytes.  Default mpileup: the gather -- a warp per 32-column group fetches the entry strings with wide loads (lanes along
//       the reads), parks them in shared-memory rows and appends them to the lines (lanes along the columns).  Other paths:
//       one thread per reference position formats its line.  Either way a tile's text is laid out in shared memory with the
//       destination's 16-byte phase and leaves the SM through cp.async.bulk (TMA) shared->global stores plus <16 B edges.
// HBM traffic per column is ~ the algorithmic bytes (+ the entry strings, written and read once).
// No tensor cores: integer/byte work.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/b200_pileup.h"
#include "plp_core.h"
#include "plp_stage.h"
#include "engine_internal.h"
#include "stage_host.h"

using namespace plp;

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    snprintf(e->err, sizeof e->err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return -1; } } while (0)

// ============================== device helpers ===============================
__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t *p)
{
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(uint64_t *p, uint64_t v)
{
    asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
#define ST_FLAG(w) ((w) >> 62)
#define ST_VAL(w) ((w) & 0x3fffffffffffffffULL)

// status words are self-contained (flag + value in one 64-bit word), so polling
// needs no acquire: relaxed gpu-scope accesses go to L2 and, unlike ld.acquire,
// do not invalidate the SM's L1 (CCTL.IVALL) under the feet of the other warps.
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t *p)
{
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t *p, uint64_t v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// decoupled look-back (sum), executed by ONE FULL WARP: 32 predecessors are
// inspected per round.  Returns the exclusive prefix of tile `t` (all lanes).
__device__ uint64_t lookback_sum(uint64_t *st, int t, uint64_t agg)
{
    const int lane = threadIdx.x & 31;
    if (t == 0) { if (lane == 0) st_relaxed_u64(&st[0], (2ULL << 62) | agg); return 0; }
    if (lane == 0) st_relaxed_u64(&st[t], (1ULL << 62) | agg);
    uint64_t excl = 0;
    for (int base = t - 1;; base -= 32) {
        const int j = base - lane;
        uint64_t w;
        unsigned m2, need;
        for (;;) {
            w = j >= 0 ? ld_relaxed_u64(&st[j]) : (2ULL << 62);      // before tile 0: inclusive prefix 0
            m2 = __ballot_sync(0xffffffffu, ST_FLAG(w) == 2);
            need = m2 ? ((2u << (__ffs(m2) - 1)) - 1u) : 0xffffffffu;  // lanes up to the nearest inclusive prefix
            if ((__ballot_sync(0xffffffffu, ST_FLAG(w) == 0) & need) == 0) break;
            __nanosleep(40);
        }
        uint64_t x = ((need >> lane) & 1u) ? ST_VAL(w) : 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        excl += x;
        if (m2) break;
    }
    if (lane == 0) st_relaxed_u64(&st[t], (2ULL << 62) | (excl + agg));
    return excl;
}

template <int T>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *warp_sums, uint32_t &total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_sums[w] = x;
    __syncthreads();
    if (w == 0) {
        uint32_t s = lane < T / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        if (lane < T / 32) warp_sums[lane] = s;
    }
    __syncthreads();
    total = warp_sums[T / 32 - 1];
    uint32_t base = w ? warp_sums[w - 1] : 0;
    return base + x - v;
}

// ============================== read stage ===================================
// (arithmetic in plp_stage.h; one thread per read)
// warp sum of a 64-bit quantity that is < 2^47 per lane: three redux.sync (16-bit limbs cannot overflow 32 lanes)
__device__ __forceinline__ unsigned long long warp_sum_u48(unsigned long long v)
{
    const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(v & 0xffffu));
    const unsigned mid = __reduce_add_sync(0xffffffffu, (unsigned)((v >> 16) & 0xffffu));
    const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(v >> 32));
    return (unsigned long long)lo + ((unsigned long long)mid << 16) + ((unsigned long long)hi << 32);
}
// Block-wide merge of the per-thread accumulators: warp reductions (single-instruction redux.sync; per-lane values are tiny:
// a read contributes 0/1 to the counters, its span / text bound / mapq to the sums), then the block's warps through shared
// memory, then ONE set of atomics per block.  The kernels that call this are grid-stride with a few blocks per SM, so a
// stage issues ~10^4 same-address atomics instead of one set per warp (3*10^5 for 1.6 M reads: they serialise in L2 and
// were most of k_build_desc's 0.18 ms).  Must be called by every thread of the block.
__device__ __forceinline__ void merge_acc(const StageAcc &a, StageAcc *g)
{
    __shared__ unsigned long long s_v[32][9];
    __shared__ int s_mx[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    unsigned long long v[9];
    v[0] = __reduce_add_sync(0xffffffffu, (unsigned)a.n_kept); v[1] = __reduce_add_sync(0xffffffffu, (unsigned)a.n_kept_in_window);
    v[2] = warp_sum_u48(a.sum_rlen); v[3] = warp_sum_u48(a.sum_indel_text);
    v[4] = __reduce_add_sync(0xffffffffu, (unsigned)a.n_reads); v[5] = __reduce_add_sync(0xffffffffu, (unsigned)a.n_selected);
    v[6] = warp_sum_u48(a.summed_mapq); v[7] = __reduce_add_sync(0xffffffffu, (unsigned)a.n_desc); v[8] = warp_sum_u48(a.sum_rlen_gen);
    const int mx = __reduce_max_sync(0xffffffffu, a.max_rend);
    if (lane == 0) { for (int k = 0; k < 9; ++k) s_v[w][k] = v[k]; s_mx[w] = mx; }
    __syncthreads();
    if (threadIdx.x < 9) {
        unsigned long long t = 0;
        for (int j = 0; j < nw; ++j) t += s_v[j][threadIdx.x];
        unsigned long long *gp[9] = {&g->n_kept, &g->n_kept_in_window, &g->sum_rlen, &g->sum_indel_text, &g->n_reads, &g->n_selected, &g->summed_mapq, &g->n_desc, &g->sum_rlen_gen};
        if (t) atomicAdd(gp[threadIdx.x], t);
    } else if (threadIdx.x == 32) {
        int m = INT32_MIN;
        for (int j = 0; j < nw; ++j) m = max(m, s_mx[j]);
        if (m != INT32_MIN) atomicMax(&g->max_rend, m);
    }
}
__global__ void k_prep1(RawSoA r, b200_stage_conf_t cf, uint8_t *state, int32_t *rlen_out, StageAcc *acc)
{
    StageAcc loc; memset(&loc, 0, sizeof loc); loc.max_rend = INT32_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < r.n; i += (int64_t)gridDim.x * blockDim.x) stage_prep1(r, cf, i, state, rlen_out, &loc);
    if (cf.mode == B200_MODE_COVERAGE) merge_acc(loc, acc);
}
__global__ void k_prep2(RawSoA r, b200_stage_conf_t cf, uint8_t *state)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < r.n) stage_prep2(r, cf, i, state);
}
__global__ void k_build_desc(RawSoA r, b200_stage_conf_t cf, const uint8_t *state, const int32_t *rlen,
                             ReadDesc *desc, int32_t *endv, StageAcc *acc, int64_t win_base, int32_t *cig_x, int32_t *cig_y)
{
    StageAcc loc; memset(&loc, 0, sizeof loc); loc.max_rend = INT32_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < r.n; i += (int64_t)gridDim.x * blockDim.x)
        stage_build_desc(r, cf, i, state, rlen, desc, endv, &loc, win_base, cig_x, cig_y);
    merge_acc(loc, acc);
}

// inclusive prefix max of endv[] (single pass, decoupled look-back, one file at a time)
__global__ void k_scan_max(const int32_t *in, int32_t *out, int64_t n, uint64_t *st, uint32_t *ticket)
{
    constexpr int T = 256, IPT = 8;
    __shared__ int s_tile;
    __shared__ int32_t s_w[T / 32];
    __shared__ int32_t s_excl;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int64_t base = (int64_t)t * T * IPT + (int64_t)threadIdx.x * IPT;
    int32_t v[IPT], m = INT32_MIN;
#pragma unroll
    for (int j = 0; j < IPT; ++j) { v[j] = base + j < n ? in[base + j] : INT32_MIN; m = max(m, v[j]); v[j] = m; }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int32_t x = m;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x = max(x, y); }
    if (lane == 31) s_w[w] = x;
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t run = INT32_MIN;
        for (int k = 0; k < T / 32; ++k) { int32_t tmp = s_w[k]; s_w[k] = run; run = max(run, tmp); }
        // publish aggregate / look back (values biased to unsigned)
        const uint64_t agg = (uint64_t)((int64_t)run - INT32_MIN);
        uint64_t excl = 0;
        if (t == 0) st_relaxed_u64(&st[0], (2ULL << 62) | agg);
        else {
            st_relaxed_u64(&st[t], (1ULL << 62) | agg);
            for (int j = t - 1;; --j) {
                uint64_t wv;
                while (ST_FLAG(wv = ld_relaxed_u64(&st[j])) == 0) { __nanosleep(20); }
                { const uint64_t pv = ST_VAL(wv); if (pv > excl) excl = pv; }
                if (ST_FLAG(wv) == 2) break;
            }
            st_relaxed_u64(&st[t], (2ULL << 62) | (excl > agg ? excl : agg));
        }
        s_excl = (int32_t)((int64_t)excl + INT32_MIN);
    }
    __syncthreads();
    int32_t pre = max(s_excl, s_w[w]);
    int32_t left = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane > 0) pre = max(pre, left);
#pragma unroll
    for (int j = 0; j < IPT; ++j) if (base + j < n) out[base + j] = max(pre, v[j]);
}

// per 32-column group: the [lo,hi) slice of each file's reads that can cover it (group_slice)
__global__ void k_ranges(const ReadDesc *desc, const int32_t *pmax, const int64_t *file_start, int n_files,
                         int32_t n_groups, int32_t *glo, int32_t *ghi, int *max_range)
{
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n_groups * n_files) return;
    const int f = (int)(idx / n_groups), g = (int)(idx % n_groups);
    int64_t first, last;
    group_slice(desc, pmax, file_start[f], file_start[f + 1], g, first, last);
    glo[idx] = (int32_t)first;
    ghi[idx] = (int32_t)last;
    atomicMax(max_range, (int)(last - first));
}

// far-reaching reads per group (ovf_span)
__global__ void k_ovf_count(const ReadDesc *desc, const int64_t *file_start, int n_files, int64_t n, int32_t n_groups, uint32_t *cnt)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ReadDesc d = desc[i];
    int32_t g0, g1;
    if (!ovf_span(d, n_groups, g0, g1)) return;
    int f = 0; while (f + 1 < n_files && i >= file_start[f + 1]) ++f;
    for (int32_t g = g0; g <= g1; ++g) atomicAdd(&cnt[(int64_t)f * n_groups + g], 1u);
}
__global__ void k_ovf_fill(const ReadDesc *desc, const int64_t *file_start, int n_files, int64_t n, int32_t n_groups,
                           const int32_t *off, uint32_t *cursor, int32_t *idx)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ReadDesc d = desc[i];
    int32_t g0, g1;
    if (!ovf_span(d, n_groups, g0, g1)) return;
    int f = 0; while (f + 1 < n_files && i >= file_start[f + 1]) ++f;
    for (int32_t g = g0; g <= g1; ++g) {
        const int64_t k = (int64_t)f * n_groups + g;
        idx[off[k] + (int32_t)atomicAdd(&cursor[k], 1u)] = (int32_t)i;
    }
}
// longest far-reaching list (enters the "can a column exceed the depth cap" bound next to the widest slice)
__global__ void k_ovf_max(const uint32_t *cnt, int64_t n_lists, int *out)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_lists && cnt[k]) atomicMax(out, (int)cnt[k]);
}
__global__ void k_ovf_sort(const int32_t *off, int32_t *idx, int64_t n_lists)   // lists are tiny: insertion sort restores file order
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_lists) return;
    int32_t *a = idx + off[k]; const int32_t m = off[k + 1] - off[k];
    for (int32_t i = 1; i < m; ++i) { const int32_t x = a[i]; int32_t j = i - 1; while (j >= 0 && a[j] > x) { a[j + 1] = a[j]; --j; } a[j + 1] = x; }
}
__global__ void k_scan_u32_excl_i32(const uint32_t *in, int32_t *out, int32_t n, uint64_t *st, uint32_t *ticket);

// ============================== column stage =================================
constexpr int TILE = 128;

// shared->global bulk store (TMA engine, SASS UBLKCP); all addresses/sizes 16 B aligned
__device__ __forceinline__ void bulk_store_s2g(void *gdst, const void *ssrc, uint32_t bytes)
{
    uint32_t saddr = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(saddr), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ---- text kernels: no inter-CTA dependency at all ---------------------------
// Fmt provides   uint32_t size(int32_t c, State&)   and   void write(int32_t c, const State&, char*)
// (1) k_*_size: every thread sizes its line; per-column {len,state} and the
//     tile total go to HBM (16-24 B per column, small next to the text itself);
// (2) a scan of the tile totals gives each tile its byte offset;
// (3) k_*_write: the tile formats its lines into shared memory, already laid
//     out with the destination's 16-byte phase, and leaves through one TMA bulk store.
template <class Fmt>
__device__ __forceinline__ void text_size_tile(const Fmt &fmt, int32_t ncols, uint32_t *len_out, typename Fmt::State *st_out,
                                               uint32_t *tile_total)
{
    __shared__ uint32_t s_ws[TILE / 32];
    const int32_t c = (int32_t)blockIdx.x * TILE + (int32_t)threadIdx.x;
    typename Fmt::State stt;
    uint32_t len = 0;
    if (c < ncols) { len = fmt.size(c, stt); len_out[c] = len; st_out[c] = stt; }
    uint32_t x = len;
#pragma unroll
    for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0) s_ws[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int k = 0; k < TILE / 32; ++k) t += s_ws[k]; tile_total[blockIdx.x] = t; }
}

template <class Fmt>
__device__ __forceinline__ void text_write_tile(const Fmt &fmt, int32_t ncols, const uint32_t *len_in, const typename Fmt::State *st_in,
                                                const uint64_t *tile_base, char *out, uint32_t smem_cap, int use_tma)
{
    extern __shared__ __align__(16) char s_text[];
    __shared__ uint32_t s_ws[TILE / 32];
    const int32_t c = (int32_t)blockIdx.x * TILE + (int32_t)threadIdx.x;
    typename Fmt::State stt;
    uint32_t len = 0;
    if (c < ncols) { len = len_in[c]; if (len) stt = st_in[c]; }
    uint32_t total;
    const uint32_t off = block_excl_scan<TILE>(len, s_ws, total);
    if (total == 0) return;
    const uint64_t base = tile_base[blockIdx.x];
    const uint32_t phase = (uint32_t)(base & 15);
    if (total + phase <= smem_cap) {
        char *sb = s_text + phase;
        if (len) fmt.write(c, stt, sb + off);
        __syncthreads();
        char *g = out + base;
        const uint32_t head = min(total, (16u - phase) & 15u);
        const uint32_t body = (total - head) & ~15u;
        const uint32_t tail = total - head - body;
        if (threadIdx.x < head) g[threadIdx.x] = sb[threadIdx.x];
        if (threadIdx.x < tail) g[head + body + threadIdx.x] = sb[head + body + threadIdx.x];
        if (body) {
            if (use_tma) {
                if (threadIdx.x == 0) bulk_store_s2g(g + head, sb + head, body);
            } else {
                const uint4 *src = reinterpret_cast<const uint4 *>(sb + head);
                uint4 *dst = reinterpret_cast<uint4 *>(g + head);
                for (uint32_t i = threadIdx.x; i < body / 16; i += TILE) dst[i] = src[i];
            }
        }
    } else if (len) {
        fmt.write(c, stt, out + base + off);
    }
}

struct MpFmt {
    View v; MpConf cf;
    typedef MpFileSz State;
    __device__ __forceinline__ uint32_t size(int32_t c, State &s) const { return mp_line_size(v, cf, c >> 5, c, s); }
    __device__ __forceinline__ void write(int32_t c, const State &s, char *p) const { mp_line_write(v, cf, c >> 5, c, s, p); }
};

__global__ void __launch_bounds__(TILE) k_mpileup_size(MpFmt fmt, uint32_t *len, MpFileSz *st, uint32_t *tile_total)
{
    text_size_tile(fmt, fmt.v.ncols, len, st, tile_total);
}
__global__ void __launch_bounds__(TILE) k_mpileup_write(MpFmt fmt, const uint32_t *len, const MpFileSz *st, const uint64_t *tile_base,
                                                        char *out, uint32_t smem_cap, int use_tma)
{
    text_write_tile(fmt, fmt.v.ncols, len, st, tile_base, out, smem_cap, use_tma);
}
#include "mpileup_ss.cuh"
#include "mpileup_ent.cuh"

// depth rows: DpFmt (plp_core.h)
__global__ void __launch_bounds__(TILE) k_depth_size(DpFmt fmt, uint32_t *len, DpFmt::State *st, uint32_t *tile_total)
{
    text_size_tile(fmt, fmt.v.ncols, len, st, tile_total);
}
__global__ void __launch_bounds__(TILE) k_depth_write(DpFmt fmt, const uint32_t *len, const DpFmt::State *st, const uint64_t *tile_base,
                                                      char *out, uint32_t smem_cap, int use_tma)
{
    text_write_tile(fmt, fmt.v.ncols, len, st, tile_base, out, smem_cap, use_tma);
}

// coverage column sums (coverage.c:622-660)
__global__ void __launch_bounds__(256) k_coverage(View v, int32_t min_baseQ, int32_t min_depth, unsigned long long *sums)
{
    const int32_t c = (int32_t)(blockIdx.x * blockDim.x + threadIdx.x);
    unsigned long long a[5] = {0, 0, 0, 0, 0};
    if (c < v.ncols) {
        CvCol o; cv_column(v, min_baseQ, c >> 5, c, o);
        a[4] = o.missing;
        if (o.count_base && o.depth >= (uint32_t)min_depth) { a[0] = 1; a[1] = o.depth; a[2] = o.sum_bq; a[3] = o.qbases; }
    }
    __shared__ unsigned long long s[5][8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        unsigned long long x = a[k];
        for (int o = 16; o; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if (lane == 0) s[k][w] = x;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        unsigned long long x = 0;
        for (int k = 0; k < 8; ++k) x += s[threadIdx.x][k];
        if (x) atomicAdd(&sums[threadIdx.x], x);
    }
}

// per-bin counters of the histogram views (coverage.c:609-660): breadth (covered columns) or depth per bin
__global__ void __launch_bounds__(256) k_coverage_hist(View v, int32_t min_baseQ, int32_t min_depth, int64_t beg_rel, int64_t bin_width, int32_t n_bins,
                                                       int plot_depth, uint32_t *hist)
{
    const int32_t c = (int32_t)(blockIdx.x * blockDim.x + threadIdx.x);
    if (c >= v.ncols) return;
    CvCol o; cv_column(v, min_baseQ, c >> 5, c, o);
    const uint32_t add = cv_hist_add(o, min_depth, plot_depth);
    if (!add) return;
    const int64_t bin = ((int64_t)c - beg_rel) / bin_width;
    if (bin >= 0 && bin < n_bins) atomicAdd(&hist[bin], add);
}

// bedcov column reducers (bedcov.c:316-331) over the staged window, per input file: sum of the per-column depth (optionally
// without deletions / reference skips) and the number of columns at or above a depth threshold (bc_any, bc_depth).
__global__ void __launch_bounds__(256) k_bedcov(View v, int skip_dn, int min_depth, unsigned long long *sums /* [n_files][2] */)
{
    const int32_t c = (int32_t)(blockIdx.x * blockDim.x + threadIdx.x);
    const bool any = c < v.ncols && bc_any(v, c);
    for (int f = 0; f < v.n_files; ++f) {
        unsigned long long pd = 0, ge = 0;
        if (any) { const int32_t d = bc_depth(v, f, c, skip_dn); pd = (unsigned long long)d; ge = (min_depth >= 0 && d >= min_depth) ? 1ull : 0ull; }
        for (int o = 16; o; o >>= 1) { pd += __shfl_xor_sync(0xffffffffu, pd, o); ge += __shfl_xor_sync(0xffffffffu, ge, o); }
        if ((threadIdx.x & 31) == 0) { if (pd) atomicAdd(&sums[2 * f], pd); if (ge) atomicAdd(&sums[2 * f + 1], ge); }
    }
}

// column-major pileup entries for the iterator tier: counts, then entries
__global__ void k_entries_count(View v, int f, int32_t c0, uint32_t *col_n)   // columns [c0, v.ncols); col_n[c - c0]
{
    const int32_t c = c0 + (int32_t)(blockIdx.x * blockDim.x + threadIdx.x);
    if (c >= v.ncols) return;
    col_n[c - c0] = column_entries<false>(v, f, c, nullptr);
}
__global__ void k_entries_fill(View v, int f, int32_t c0, const uint64_t *col_off, b200_pileup1_t *ents)
{
    const int32_t c = c0 + (int32_t)(blockIdx.x * blockDim.x + threadIdx.x);
    if (c >= v.ncols) return;
    column_entries<true>(v, f, c, ents + col_off[c - c0]);
}
__global__ void k_scan_u32_to_u64(const uint32_t *in, uint64_t *out, int32_t n, uint64_t *st, uint32_t *ticket)
{
    constexpr int T = 256;
    __shared__ uint32_t s_ws[T / 32];
    __shared__ int s_tile; __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int32_t i = t * T + (int32_t)threadIdx.x;
    uint32_t v = i < n ? in[i] : 0, total;
    uint32_t off = block_excl_scan<T>(v, s_ws, total);
    if (threadIdx.x < 32) { const uint64_t b = lookback_sum(st, t, total); if (threadIdx.x == 0) s_base = b; }
    __syncthreads();
    if (i < n) out[i] = s_base + off;
    if (i == n - 1) out[n] = s_base + off + v;
}

__global__ void k_scan_u32_excl_i32(const uint32_t *in, int32_t *out, int32_t n, uint64_t *st, uint32_t *ticket)
{
    constexpr int T = 256;
    __shared__ uint32_t s_ws[T / 32];
    __shared__ int s_tile; __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int32_t i = t * T + (int32_t)threadIdx.x;
    uint32_t v = i < n ? in[i] : 0, total;
    uint32_t off = block_excl_scan<T>(v, s_ws, total);
    if (threadIdx.x < 32) { const uint64_t b = lookback_sum(st, t, total); if (threadIdx.x == 0) s_base = b; }
    __syncthreads();
    if (i < n) out[i] = (int32_t)(s_base + off);
    if (i == n - 1) out[n] = (int32_t)(s_base + off + v);
}

// ============================== host side ====================================
template <class T> static int ensure(b200_engine *e, T *&p, size_t &cap, size_t need)
{
    if (need <= cap && p) return 0;
    if (p) cudaFree(p);
    size_t nc = need + need / 8 + 256;
    p = nullptr; cap = 0;
    CK(cudaMalloc((void **)&p, nc * sizeof(T)));
    cap = nc;
    return 0;
}
#define ENSURE(field, need) do { if (ensure(e, e->field, e->cap_##field, (need))) return -1; } while (0)

static inline int nblk(int64_t n, int t) { return (int)((n + t - 1) / t); }

#include "overlap.cuh"
#include "baq.cuh"

extern "C" const char *b200_version(void) { return "samtools_b200 0.1 (sm_100a)"; }
extern "C" const char *b200_last_error(const b200_engine_t *e) { return e ? e->err : "null engine"; }
extern "C" double b200_last_kernel_ms(const b200_engine_t *e) { return e->last_kernel_ms; }
extern "C" double b200_last_stage_ms(const b200_engine_t *e) { return e->last_stage_ms; }
extern "C" int64_t b200_launch_count(const b200_engine_t *e) { return e->launches; }
extern "C" uint64_t b200_gl_rng_draws(const b200_engine_t *e) { return e ? e->gl_rng_draws : 0; }
extern "C" void b200_last_mpileup_parts_ms(const b200_engine_t *e, double *ms3) { for (int i = 0; i < 3; ++i) ms3[i] = e->last_parts_ms[i]; }

extern "C" int b200_engine_create(int device, b200_engine_t **out)
{
    *out = nullptr;
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n <= 0) {
        fprintf(stderr, "[b200_pileup] no CUDA device: %s (this engine has no CPU fallback)\n", cudaGetErrorString(ce));
        return -1;
    }
    if (device < 0 || device >= n) { fprintf(stderr, "[b200_pileup] bad device %d of %d\n", device, n); return -1; }
    b200_engine *e = new b200_engine();
    e->device = device;
    e->err[0] = 0;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
        fprintf(stderr, "[b200_pileup] cannot initialise device %d\n", device);
        delete e;
        return -1;
    }
    cudaEventCreate(&e->ev0); cudaEventCreate(&e->ev1); cudaEventCreate(&e->evA); cudaEventCreate(&e->evB);
    cudaEventCreate(&e->evB0); cudaEventCreate(&e->evB1);
    cudaDeviceGetAttribute(&e->n_sm, cudaDevAttrMultiProcessorCount, device);
    e->smem_text = 24 * 1024;
    const char *s = getenv("B200_PLP_SMEM_TEXT"); if (s) e->smem_text = (uint32_t)atoi(s);
    s = getenv("B200_PLP_TMA"); e->use_tma = s ? atoi(s) : 1;
    s = getenv("B200_PLP_GENERAL"); e->general = s ? atoi(s) : 0;   // 1: general mpileup path (thread-per-column size + write) for every configuration
    if (e->smem_text + 16 > 48 * 1024) {   // the attribute is per function and process-wide: only ever raise it (another handle may use more)
        cudaFuncSetAttribute(k_mp_gather<7, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_mp_gather<7, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_mpileup_write, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_depth_write, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e->smem_text > 200 * 1024 - 16) e->smem_text = 200 * 1024 - 16;
    }
    cudaMalloc((void **)&e->d_acc, sizeof(StageAcc));
    cudaMalloc((void **)&e->d_misc, 64 * sizeof(unsigned long long));
    *out = e;
    return 0;
}

extern "C" void b200_engine_destroy(b200_engine_t *e)
{
    if (!e) return;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    e->free_all();
    cudaFree(e->d_acc); cudaFree(e->d_misc); if (e->d_gfmt) cudaFree(e->d_gfmt);
    cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1); cudaEventDestroy(e->evA); cudaEventDestroy(e->evB);
    cudaEventDestroy(e->evB0); cudaEventDestroy(e->evB1);
    cudaStreamDestroy(e->stream);
    delete e;
}

template <class T> static int h2d(b200_engine *e, T *&dp, size_t &cap, const T *hp, size_t n)
{
    if (ensure(e, dp, cap, n ? n : 1)) return -1;
    if (n && hp) CK(cudaMemcpyAsync(dp, hp, n * sizeof(T), cudaMemcpyHostToDevice, e->stream));
    return 0;
}
#define H2D(field, hp, n) do { if (h2d(e, e->field, e->cap_##field, (hp), (size_t)(n))) return -1; } while (0)


// Exact test for "the max-depth rule cannot fire": bam_plp_push drops a read only when more than maxcnt accepted reads of its
// file are still buffered at its start, i.e. their closed intervals [start, end] hold one position.  The largest such count is
// the maximum of the prefix sum of a +1 / -1 difference array over the kept reads (positions outside the staged columns are
// folded onto the first / last one: an over-estimate, which is the safe side).
__global__ void k_cov_diff(const uint8_t *state, const ReadDesc *desc, const int32_t *rlen, int64_t i0, int64_t i1, int32_t ncols, int32_t *diff)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1 || state[i] != ST_KEEP) return;
    const int64_t p = desc[i].rpos, q = p + (int64_t)rlen[i] + 1;
    const int32_t a = (int32_t)(p < 0 ? 0 : (p > ncols ? ncols : p)), b = (int32_t)(q < 1 ? 1 : (q > (int64_t)ncols + 1 ? (int64_t)ncols + 1 : q));
    atomicAdd(&diff[a], 1); atomicAdd(&diff[b], -1);
}
__global__ void k_max_i32(const int32_t *x, int32_t n, int *out)
{
    int m = INT32_MIN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = max(m, x[i]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}
// largest number of kept reads of one file whose closed intervals share a position (see k_cov_diff)
static int max_buffered_reads(b200_engine *e, int *out)
{
    const int32_t ncols = e->ncols_max + 1;
    ENSURE(ss_diff, (size_t)ncols + 3); ENSURE(ss_nplp, (size_t)ncols + 3);
    const int nbs = nblk((int64_t)ncols + 2, 1024);
    ENSURE(status2, (size_t)nbs + 1);
    int best = 0;
    for (int f = 0; f < e->n_files; ++f) {
        const int64_t i0 = e->h_file_start[f], i1 = e->h_file_start[f + 1];
        if (i1 <= i0) continue;
        CK(cudaMemsetAsync(e->ss_diff, 0, ((size_t)ncols + 2) * 4, e->stream));
        CK(cudaMemsetAsync(e->status2, 0, ((size_t)nbs + 1) * 8, e->stream));
        CK(cudaMemsetAsync(e->d_misc + 2, 0, 16, e->stream));
        k_cov_diff<<<nblk(i1 - i0, 256), 256, 0, e->stream>>>(e->state, e->desc, e->rlen, i0, i1, ncols, e->ss_diff); e->launches++;
        k_ss_scan<<<nbs, 256, 0, e->stream>>>(e->ss_diff, e->ss_nplp, ncols + 2, e->status2, (uint32_t *)(e->d_misc + 2)); e->launches++;
        k_max_i32<<<e->n_sm * 4, 256, 0, e->stream>>>(e->ss_nplp, ncols + 2, (int *)(e->d_misc + 3)); e->launches++;
        int m = 0;
        CK(cudaMemcpyAsync(&m, e->d_misc + 3, 4, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        if (m > best) best = m;
    }
    *out = best;
    return 0;
}

// descriptors and states of the staged reads, copied to the host for the host-side rules (stage_host.h)
static int fetch_desc_state(b200_engine *e, int64_t n, std::vector<ReadDesc> &hd, std::vector<uint8_t> &st)
{
    hd.resize((size_t)n); st.resize((size_t)n);
    CK(cudaMemcpyAsync(hd.data(), e->desc, (size_t)n * sizeof(ReadDesc), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(st.data(), e->state, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// max-depth rule of bam_plp_push (apply_maxcnt), evaluated on the host only when a column could hold more than maxcnt reads
static int apply_maxcnt_host(b200_engine *e, int64_t n, int maxcnt)
{
    std::vector<ReadDesc> hd; std::vector<uint8_t> st; std::vector<int32_t> rl((size_t)n);
    CK(cudaMemcpyAsync(rl.data(), e->rlen, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (fetch_desc_state(e, n, hd, st)) return -1;
    e->maxdrop_applied = apply_maxcnt(hd.data(), rl.data(), st.data(), e->h_file_start.data(), e->n_files, maxcnt);
    if (e->maxdrop_applied) CK(cudaMemcpyAsync(e->state, st.data(), (size_t)n, cudaMemcpyHostToDevice, e->stream));
    return 0;
}

__global__ void k_apply_maxdrop(const uint8_t *state, ReadDesc *desc, int32_t *endv, int64_t n)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (state[i] == ST_MAXDROP) { desc[i].rend = desc[i].rpos; endv[i] = INT32_MIN; }
}

static int stage_device(b200_engine *e, b200_stage_stats_t *stats);
static TextDims text_dims(const b200_engine *e) { return {e->sum_rlen, e->sum_indel_text, e->ncols_max, e->name.size(), e->n_files, e->n}; }

extern "C" int b200_stage(b200_engine_t *e, const b200_batch_t *b, const b200_stage_conf_t *cf, b200_stage_stats_t *stats)
{
    if (!e || !b || !cf) return -1;
    CK(cudaSetDevice(e->device));
    const int64_t n = b->n_reads;
    if (b->n_files < 1) { snprintf(e->err, sizeof e->err, "n_files < 1"); return -1; }
    if (n >= (1LL << 31)) { snprintf(e->err, sizeof e->err, "batch too large (%lld reads)", (long long)n); return -1; }
    if (b->qual_bytes >= (1ULL << 32) || b->n_cigar_total >= (1ULL << 32)) { snprintf(e->err, sizeof e->err, "batch payload exceeds 4 GiB: split the window"); return -1; }
    CK(cudaEventRecord(e->ev0, e->stream));
    e->n = n; e->n_files = b->n_files; e->tid = b->tid; e->tid_len = b->tid_len;
    e->name = b->tid_name ? b->tid_name : "";
    e->sconf = *cf;
    e->win_base = cf->beg > 0 ? cf->beg : 0;
    e->h_file_start.assign(b->file_start, b->file_start + b->n_files + 1);
    // ---- H2D
    H2D(pos, b->pos, n); H2D(flag, b->flag, n); H2D(mapq, b->mapq, n); H2D(l_qseq, b->l_qseq, n);
    H2D(n_cigar, b->n_cigar, n); H2D(cigar_off, b->cigar_off, n); H2D(qual_off, b->qual_off, n);
    H2D(mtid, b->mtid, n); H2D(mpos, b->mpos, n); H2D(isize, b->isize, n);
    e->has_prev = b->prev_same_name != nullptr;
    if (e->has_prev) H2D(prev, b->prev_same_name, n);
    e->has_rbits = b->rbits != nullptr;
    if (e->has_rbits) H2D(rbits, b->rbits, n);
    H2D(cigar, b->cigar, b->n_cigar_total);
    H2D(seq4, b->seq4, (b->qual_bytes + 1) / 2 + 1);
    e->qual_bytes = (size_t)b->qual_bytes + 1;
    if (e->keep_raw) {       // a pristine copy stays resident so that b200_restage() can repeat the read stage (it edits qualities / mapq in place)
        H2D(qual0, b->qual, b->qual_bytes + 1); H2D(mapq0, b->mapq, n);
        ENSURE(qual, (size_t)b->qual_bytes + 1);
    } else H2D(qual, b->qual, b->qual_bytes + 1);
    H2D(file_start, b->file_start, b->n_files + 1);
    e->has_ref = b->ref != nullptr && b->ref_len > 0;
    if (e->has_ref) H2D(ref, b->ref, b->ref_n);
    e->ref_beg = b->ref_beg; e->ref_n = b->ref_n; e->ref_len = e->has_ref ? b->ref_len : 0;
    {
        size_t nl = strlen(e->name.c_str());
        H2D(dname, e->name.c_str(), nl + 1);
    }
    e->n_cigar_total = (size_t)b->n_cigar_total;
    e->has_host_clip = false;
    if (cf->mode == B200_MODE_DEPTH && cf->d_remove_overlaps && b->depth_clip && n > 0) {
        // clip coordinates replayed by the caller (one name hash per file, across reference sequences)
        e->h_clip_tmp.resize((size_t)n);
        for (int64_t i = 0; i < n; ++i) e->h_clip_tmp[(size_t)i] = clip_rel(b->depth_clip[i], e->win_base);
        H2D(clip, e->h_clip_tmp.data(), n);
        e->has_host_clip = true;
    }
    CK(cudaEventRecord(e->evA, e->stream));
    e->uploaded = true;
    return stage_device(e, stats);
}

// Device side of the read stage: per-read filters, -6, BAQ, -C, descriptors, per-group read slices, max-depth rule,
// mate-overlap tweak.  Works on the arrays resident in device memory (b200_stage uploads them first).
static int stage_device(b200_engine *e, b200_stage_stats_t *stats)
{
    const int64_t n = e->n;
    const b200_stage_conf_t *cf = &e->sconf;
    if (e->keep_raw && n > 0) {
        CK(cudaMemcpyAsync(e->qual, e->qual0, e->qual_bytes, cudaMemcpyDeviceToDevice, e->stream));
        CK(cudaMemcpyAsync(e->mapq, e->mapq0, (size_t)n, cudaMemcpyDeviceToDevice, e->stream));
    }
    ENSURE(state, (size_t)n + 1); ENSURE(rlen, (size_t)n + 1); ENSURE(desc, (size_t)n + 1);
    ENSURE(endv, (size_t)n + 1); ENSURE(pmax, (size_t)n + 1);
    ENSURE(cig_x, e->n_cigar_total + 1); ENSURE(cig_y, e->n_cigar_total + 1);
    CK(cudaMemsetAsync(e->d_acc, 0, sizeof(StageAcc), e->stream));
    {
        StageAcc z; memset(&z, 0, sizeof z); z.max_rend = INT32_MIN;
        CK(cudaMemcpyAsync(e->d_acc, &z, sizeof z, cudaMemcpyHostToDevice, e->stream));
    }
    RawSoA r;
    r.pos = e->pos; r.flag = e->flag; r.mapq = e->mapq; r.l_qseq = e->l_qseq; r.n_cigar = e->n_cigar;
    r.cigar_off = e->cigar_off; r.qual_off = e->qual_off; r.mtid = e->mtid; r.mpos = e->mpos; r.isize = e->isize;
    r.prev = e->has_prev ? e->prev : nullptr; r.rbits = e->has_rbits ? e->rbits : nullptr;
    r.cigar = e->cigar; r.seq4 = e->seq4; r.qual = e->qual;
    r.ref = e->has_ref ? e->ref : nullptr; r.ref_beg = e->ref_beg; r.ref_n = e->ref_n; r.ref_len = e->ref_len;
    r.n = n; r.tid = e->tid;
    StageAcc *acc = (StageAcc *)e->d_acc;
    if (e->has_ref && e->ref_n > 0) {   // reference bases -> codes, once per staged batch (BAQ: 0..4, pileup_seq: nt16)
        ENSURE(ref_codes, (size_t)e->ref_n + 1);
        k_ref_codes<<<nblk(e->ref_n, 256), 256, 0, e->stream>>>(e->ref, e->ref_n, e->ref_codes); e->launches++;
    }
    if (n > 0) {
        const int gs = (int)std::min<int64_t>(nblk(n, 256), (int64_t)e->n_sm * 16);   // grid-stride: one set of accumulator atomics per block
        k_prep1<<<gs, 256, 0, e->stream>>>(r, *cf, e->state, e->rlen, acc); e->launches++;
        e->baq_ran = false;
        if (cf->mode == B200_MODE_MPILEUP && cf->baq && e->has_ref) {
            CK(cudaEventRecord(e->evB0, e->stream));
            if (launch_baq(e, r, *cf)) return -1;
            CK(cudaEventRecord(e->evB1, e->stream));
            e->baq_ran = true;
        }
        k_prep2<<<nblk(n, 256), 256, 0, e->stream>>>(r, *cf, e->state); e->launches++;
        k_build_desc<<<gs, 256, 0, e->stream>>>(r, *cf, e->state, e->rlen, e->desc, e->endv, acc, e->win_base, e->cig_x, e->cig_y); e->launches++;
    }
    CK(cudaGetLastError());
    // ---- statistics back (also the sync point that validates the batch)
    StageAcc ha;
    CK(cudaMemcpyAsync(&ha, e->d_acc, sizeof ha, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (ha.n_desc) {   // rare path: some record starts before its predecessor
        std::vector<ReadDesc> hd; std::vector<uint8_t> st;
        if (fetch_desc_state(e, n, hd, st)) return -1;
        if (const char *msg = check_sorted(hd.data(), st.data(), e->h_file_start.data(), e->n_files, cf->mode)) { snprintf(e->err, sizeof e->err, "%s", msg); return -3; }
    }
    e->acc_n_kept = (int64_t)ha.n_kept; e->max_rend = ha.n_kept ? ha.max_rend : 0;
    e->sum_rlen = ha.sum_rlen; e->sum_indel_text = ha.sum_indel_text; e->sum_rlen_gen = ha.sum_rlen_gen;
    if (!column_domain(e->max_rend, cf->end, e->tid_len, e->win_base, e->ncols_cov, e->ncols_all, e->ncols_max, e->err, sizeof e->err)) return -1;
    e->n_groups = (e->ncols_max + 31) / 32 + 1;
    ENSURE(glo, (size_t)e->n_groups * e->n_files + 1); ENSURE(ghi, (size_t)e->n_groups * e->n_files + 1);
    e->maxdrop_applied = false;
    int max_range = 0;
    if (n > 0) {
        if (build_ranges(e, &max_range)) return -1;
        // max-depth rule (bam_plp_push): only reachable when some column can hold > maxcnt reads
        bool may_fire = cf->mode != B200_MODE_DEPTH && cf->max_depth > 0 && 2LL * max_range + 1 > (int64_t)cf->max_depth;
        if (may_fire) {   // the slice bound is loose (deep amplicons): exact count on the device before falling back to the host sweep
            int mb = 0;
            if (max_buffered_reads(e, &mb)) return -1;
            may_fire = (int64_t)mb + 1 > (int64_t)cf->max_depth;
        }
        if (may_fire) {
            if (apply_maxcnt_host(e, n, cf->max_depth)) return -1;
            if (e->maxdrop_applied) {
                k_apply_maxdrop<<<nblk(n, 256), 256, 0, e->stream>>>(e->state, e->desc, e->endv, n); e->launches++;
                if (build_ranges(e, &max_range)) return -1;
            }
        }
        if (cf->mode == B200_MODE_MPILEUP && cf->overlaps && e->has_prev) { if (launch_overlap(e, r)) return -1; }
        if (e->has_host_clip) {
            e->has_clip = true;
        } else if (cf->mode == B200_MODE_DEPTH && cf->d_remove_overlaps && e->has_prev) { if (launch_depth_clip(e, r)) return -1; }
        else e->has_clip = false;
    } else {
        CK(cudaMemsetAsync(e->glo, 0, ((size_t)e->n_groups * e->n_files) * 4, e->stream));
        CK(cudaMemsetAsync(e->ghi, 0, ((size_t)e->n_groups * e->n_files) * 4, e->stream));
        ENSURE(ovf_off, (size_t)e->n_groups * e->n_files + 2); ENSURE(ovf_idx, 1);
        CK(cudaMemsetAsync(e->ovf_off, 0, ((size_t)e->n_groups * e->n_files + 2) * 4, e->stream));
        e->has_clip = false;
    }
    CK(cudaEventRecord(e->ev1, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1); e->last_stage_ms = ms;
    cudaEventElapsedTime(&ms, e->evA, e->ev1); e->last_stage_device_ms = ms;
    e->last_baq_ms = 0;
    if (e->baq_ran) { cudaEventElapsedTime(&ms, e->evB0, e->evB1); e->last_baq_ms = ms; }
    e->staged = true;
    if (stats) {
        stats->n_kept = (int64_t)ha.n_kept; stats->n_kept_in_window = (int64_t)ha.n_kept_in_window;
        stats->n_reads = ha.n_reads; stats->n_selected_reads = ha.n_selected; stats->summed_mapq = ha.summed_mapq;
        stats->out_bound = text_bound(text_dims(e), 27, 1);
        stats->n_cols = e->ncols_max;
    }
    return 0;
}

extern "C" int b200_set_keep_raw(b200_engine_t *e, int on)
{
    if (!e) return -1;
    e->keep_raw = on != 0; e->uploaded = false; e->staged = false;
    return 0;
}

extern "C" int b200_restage(b200_engine_t *e, b200_stage_stats_t *stats)
{
    if (!e) return -1;
    if (!e->uploaded || !e->keep_raw) { snprintf(e->err, sizeof e->err, "b200_restage needs b200_set_keep_raw(e, 1) before b200_stage"); return -1; }
    CK(cudaSetDevice(e->device));
    e->staged = false;
    CK(cudaEventRecord(e->ev0, e->stream));
    CK(cudaEventRecord(e->evA, e->stream));
    return stage_device(e, stats);
}
extern "C" double b200_last_stage_device_ms(const b200_engine_t *e) { return e ? e->last_stage_device_ms : 0; }
extern "C" double b200_last_baq_ms(const b200_engine_t *e) { return e ? e->last_baq_ms : 0; }

int build_ranges(b200_engine *e, int *max_range)
{
    const int64_t n = e->n;
    // prefix max of read ends, file by file
    for (int f = 0; f < e->n_files; ++f) {
        const int64_t fs = e->h_file_start[f], fn = e->h_file_start[f + 1] - fs;
        if (fn <= 0) continue;
        const int nb = nblk(fn, 256 * 8);
        ENSURE(status, (size_t)nb + 1);
        CK(cudaMemsetAsync(e->status, 0, ((size_t)nb + 1) * 8, e->stream));
        CK(cudaMemsetAsync(e->d_misc, 0, 8, e->stream));
        k_scan_max<<<nb, 256, 0, e->stream>>>(e->endv + fs, e->pmax + fs, fn, e->status, (uint32_t *)e->d_misc); e->launches++;
    }
    CK(cudaMemsetAsync(e->d_misc + 1, 0, 8, e->stream));
    const int64_t tot = (int64_t)e->n_groups * e->n_files;
    k_ranges<<<nblk(tot, 256), 256, 0, e->stream>>>(e->desc, e->pmax, e->file_start, e->n_files, e->n_groups, e->glo, e->ghi, (int *)(e->d_misc + 1));
    e->launches++;
    // far-reaching reads per group
    ENSURE(ovf_cnt, (size_t)tot + 1); ENSURE(ovf_off, (size_t)tot + 2);
    CK(cudaMemsetAsync(e->ovf_cnt, 0, ((size_t)tot + 1) * 4, e->stream));
    k_ovf_count<<<nblk(n, 256), 256, 0, e->stream>>>(e->desc, e->file_start, e->n_files, n, e->n_groups, e->ovf_cnt); e->launches++;
    k_ovf_max<<<nblk(tot, 256), 256, 0, e->stream>>>(e->ovf_cnt, tot, (int *)(e->d_misc + 1) + 1); e->launches++;
    {
        const int nb = nblk(tot, 256);
        ENSURE(status, (size_t)nb + 1);
        CK(cudaMemsetAsync(e->status, 0, ((size_t)nb + 1) * 8, e->stream));
        CK(cudaMemsetAsync(e->d_misc, 0, 8, e->stream));
        k_scan_u32_excl_i32<<<nb, 256, 0, e->stream>>>(e->ovf_cnt, e->ovf_off, (int32_t)tot, e->status, (uint32_t *)e->d_misc); e->launches++;
    }
    int32_t n_ovf = 0;
    CK(cudaMemcpyAsync(&n_ovf, e->ovf_off + tot, 4, cudaMemcpyDeviceToHost, e->stream));
    int mx[2] = {0, 0};                        // widest slice, longest far-reaching list
    CK(cudaMemcpyAsync(mx, e->d_misc + 1, sizeof mx, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    *max_range = mx[0] + mx[1];                // no column holds more reads than this
    ENSURE(ovf_idx, (size_t)n_ovf + 1);
    if (n_ovf > 0) {
        CK(cudaMemsetAsync(e->ovf_cnt, 0, ((size_t)tot + 1) * 4, e->stream));
        k_ovf_fill<<<nblk(n, 256), 256, 0, e->stream>>>(e->desc, e->file_start, e->n_files, n, e->n_groups, e->ovf_off, e->ovf_cnt, e->ovf_idx); e->launches++;
        k_ovf_sort<<<nblk(tot, 256), 256, 0, e->stream>>>(e->ovf_off, e->ovf_idx, tot); e->launches++;
    }
    CK(cudaGetLastError());
    return 0;
}

static void fill_view(b200_engine *e, View &v, const int64_t *bed_beg, const int64_t *bed_end, int n_bed, int bed_active, int all)
{
    v.desc = e->desc; v.cigar = e->cigar; v.cig_x = e->cig_x; v.cig_y = e->cig_y; v.seq4 = e->seq4; v.qual = e->qual;
    v.clip = e->has_clip ? e->clip : nullptr;
    v.ref = e->has_ref ? e->ref : nullptr;
    v.ref_off = e->ref_beg - e->win_base; v.ref_n = e->ref_n; v.ref_len_rel = e->ref_len - e->win_base;
    v.n_files = e->n_files; v.file_start = e->file_start;
    v.tile_lo = e->glo; v.tile_hi = e->ghi; v.ovf_off = e->ovf_off; v.ovf_idx = e->ovf_idx; v.n_tiles = e->n_groups; v.tile_cols = 32;
    v.win_base = e->win_base;
    v.ncols_all = all ? (int32_t)e->ncols_all : 0;
    v.ncols = (int32_t)(all ? std::max(e->ncols_cov, e->ncols_all) : e->ncols_cov);
    v.name = e->dname; v.name_len = (int32_t)e->name.size();
    v.bed_beg = bed_beg; v.bed_end = bed_end; v.n_bed = n_bed; v.bed_active = bed_active;
    v.n_x = 0; v.x_stride = 0; v.x_off = nullptr; v.x_dat = nullptr; memset(v.x_sep, 0, sizeof v.x_sep);
}

static int upload_bed(b200_engine *e, const int64_t *bb, const int64_t *be, int n, int active)
{
    if (!active) return 0;
    H2D(bed_beg, bb, n); H2D(bed_end, be, n);
    return 0;
}

// The text pass over nt 128-column tiles once the per-column buffers are in place: sizes() launches the size pass (line
// lengths into col_n / col_state, tile totals into tile_total), a scan turns the tile totals into byte offsets (col_off),
// write() launches the byte pass into e->out; then the timings, the bound check and the copy-out.
template <class Sizes, class Write>
static int text_pass(b200_engine *e, int nt, uint64_t bound, Sizes sizes, Write write, char *out, size_t out_cap, size_t *out_len)
{
    ENSURE(out, (size_t)bound + 64);
    ENSURE(tile_total, (size_t)nt + 1); ENSURE(col_off, (size_t)nt + 2);
    const int nb = nblk(nt, 256);
    ENSURE(status, (size_t)nb + 1);
    CK(cudaMemsetAsync(e->status, 0, ((size_t)nb + 1) * 8, e->stream));
    CK(cudaMemsetAsync(e->d_misc, 0, 8, e->stream));
    CK(cudaEventRecord(e->ev0, e->stream));
    if (sizes()) return -1;
    CK(cudaEventRecord(e->evA, e->stream));
    k_scan_u32_to_u64<<<nb, 256, 0, e->stream>>>(e->tile_total, e->col_off, nt, e->status, (uint32_t *)e->d_misc); e->launches++;
    CK(cudaEventRecord(e->evB, e->stream));
    if (write()) return -1;
    CK(cudaEventRecord(e->ev1, e->stream));
    unsigned long long total = 0;
    CK(cudaMemcpyAsync(&total, e->col_off + nt, 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1); e->last_kernel_ms = ms;
    cudaEventElapsedTime(&ms, e->ev0, e->evA); e->last_parts_ms[0] = ms;      // size pass
    cudaEventElapsedTime(&ms, e->evA, e->evB); e->last_parts_ms[1] = ms;      // tile-offset scan
    cudaEventElapsedTime(&ms, e->evB, e->ev1); e->last_parts_ms[2] = ms;      // write pass
    if (!within_bound(total, bound, e->err, sizeof e->err)) return -1;
    *out_len = (size_t)total;
    e->last_out_len = (size_t)total;
    if (out) {
        if (total > out_cap) { snprintf(e->err, sizeof e->err, "output buffer too small: need %llu bytes", total); return -2; }
        CK(cudaMemcpyAsync(out, e->out, (size_t)total, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
    }
    return 0;
}

// thread-per-column text: k_size / k_write over Fmt (text_size_tile / text_write_tile)
template <class Fmt, class KS, class KW>
static int run_text(b200_engine *e, KS k_size, KW k_write, const Fmt &fmt, uint64_t bound, char *out, size_t out_cap, size_t *out_len)
{
    const int32_t ncols = fmt.v.ncols;
    const int nt = (ncols + TILE - 1) / TILE;
    *out_len = 0;
    e->last_kernel_ms = 0;
    if (nt == 0) return 0;
    typedef typename Fmt::State State;
    ENSURE(col_n, (size_t)ncols + 1);                                   // per-column line length
    const size_t st_words = ((size_t)ncols * sizeof(State) + 7) / 8 + 1;
    ENSURE(col_state, st_words);                                        // per-column formatter state
    return text_pass(e, nt, bound,
        [&] { k_size<<<nt, TILE, 0, e->stream>>>(fmt, e->col_n, (State *)e->col_state, e->tile_total); e->launches++; return 0; },
        [&] { k_write<<<nt, TILE, e->smem_text + 16, e->stream>>>(fmt, e->col_n, (const State *)e->col_state, e->col_off, e->out, e->smem_text, e->use_tma); e->launches++; return 0; },
        out, out_cap, out_len);
}

extern "C" uint64_t b200_mpileup_text_bound(const b200_engine_t *e, const b200_mpileup_conf_t *c) { return (e && e->staged && c) ? mpileup_bound(text_dims(e), c) : 0; }

extern "C" int b200_mpileup_text(b200_engine_t *e, const b200_mpileup_conf_t *c, char *out, size_t out_cap, size_t *out_len)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    CK(cudaSetDevice(e->device));
    if (upload_bed(e, c->bed_beg, c->bed_end, c->n_bed, c->bed_active)) return -1;
    MpFmt fmt;
    fill_view(e, fmt.v, e->bed_beg, e->bed_end, c->n_bed, c->bed_active, c->all);
    fmt.cf.min_baseQ = c->min_baseQ; fmt.cf.all = c->all; fmt.cf.rev_del = c->rev_del; fmt.cf.no_ins = c->no_ins;
    fmt.cf.no_del = c->no_del; fmt.cf.no_ends = c->no_ends; fmt.cf.out_mapq = c->out_mapq; fmt.cf.out_qpos = c->out_qpos;
    fmt.cf.out_qpos5 = c->out_qpos5; fmt.cf.n_star_cols = c->n_star_cols;
    const uint64_t bound = mpileup_bound(text_dims(e), c);
    if (c->n_x > 0) {   // host columns: upload the per-read string tables, widen the bound by the longest per-read contribution
        if (c->n_x > PLP_MAX_X || c->n_x != c->n_star_cols || !c->x_off || (!c->x_dat && c->x_bytes)) { snprintf(e->err, sizeof e->err, "bad host-column tables"); return -1; }
        const size_t n_off = (size_t)c->n_x * ((size_t)e->n + 1);
        H2D(x_off, c->x_off, n_off); H2D(x_dat, c->x_dat, c->x_bytes ? c->x_bytes : 1);
        fmt.v.n_x = c->n_x; fmt.v.x_stride = e->n + 1; fmt.v.x_off = e->x_off; fmt.v.x_dat = e->x_dat; memcpy(fmt.v.x_sep, c->x_sep, sizeof fmt.v.x_sep);
    }
    if (e->general || e->n_files != 1 || c->out_qpos || c->out_qpos5 || c->n_x > 0)
        return run_text(e, k_mpileup_size, k_mpileup_write, fmt, bound, out, out_cap, out_len);
    // ---- default (one input file, no -O columns): entry strings + gather (mpileup_ent.cuh)
    const int32_t ncols = fmt.v.ncols;
    const int nt = (ncols + TILE - 1) / TILE;            // 128-column tiles
    *out_len = 0; e->last_kernel_ms = 0;
    if (nt == 0) return 0;
    ENSURE(col_n, (size_t)nt * TILE + 1);
    ENSURE(col_state, ((size_t)nt * TILE * sizeof(MpFileSz) + 7) / 8 + 1);
    ENSURE(ent, e->qual_bytes + 64 + ENT_PAD); ENSURE(ent2, (size_t)e->sum_rlen_gen + 64 + ENT_PAD);   // front pad + slack for the gather's 80-byte fetches
    ENSURE(ss_diff, (size_t)ncols + 2); ENSURE(ss_nplp, (size_t)ncols + 2); ENSURE(ss_fail, (size_t)ncols + 1); ENSURE(ss_extra, (size_t)ncols + 1);
    CK(cudaMemsetAsync(e->ss_diff, 0, ((size_t)ncols + 2) * 4, e->stream));
    CK(cudaMemsetAsync(e->ss_fail, 0, ((size_t)ncols + 1) * 4, e->stream));
    CK(cudaMemsetAsync(e->ss_extra, 0, ((size_t)ncols + 1) * 4, e->stream));
    const int nbs = nblk((int64_t)ncols + 1, 1024);
    ENSURE(status2, (size_t)nbs + 1);
    CK(cudaMemsetAsync(e->status2, 0, ((size_t)nbs + 1) * 8, e->stream));
    CK(cudaMemsetAsync(e->d_misc + 2, 0, 16, e->stream));      // scan ticket, cursor of the second entry array
    // entry strings + order-free line sizes
    auto sizes = [&] {
        const int64_t want_blocks = (e->n * 32 + 255) / 256;
        const int rb = (int)std::max<int64_t>(1, std::min<int64_t>(want_blocks, (int64_t)e->n_sm * 16));
        if (e->has_ref) k_mp_entries<true><<<rb, 256, 0, e->stream>>>(fmt.v, fmt.cf, e->n, e->ref_codes, e->ss_diff, e->ss_fail, e->ss_extra, e->ent + ENT_PAD, e->ent2 + ENT_PAD, e->d_misc + 3, e->desc);
        else k_mp_entries<false><<<rb, 256, 0, e->stream>>>(fmt.v, fmt.cf, e->n, nullptr, e->ss_diff, e->ss_fail, e->ss_extra, e->ent + ENT_PAD, e->ent2 + ENT_PAD, e->d_misc + 3, e->desc);
        e->launches++;
        k_ss_scan<<<nbs, 256, 0, e->stream>>>(e->ss_diff, e->ss_nplp, ncols + 1, e->status2, (uint32_t *)(e->d_misc + 2)); e->launches++;
        k_ss_cols<<<nt, TILE, 0, e->stream>>>(fmt.v, fmt.cf, e->ss_nplp, e->ss_fail, e->ss_extra, e->col_n, (MpFileSz *)e->col_state, e->tile_total); e->launches++;
        return 0;
    };
    // gather
    auto write = [&] {
        MpEntFmt gf; gf.v = fmt.v; gf.cf = fmt.cf; gf.E = e->ent + ENT_PAD; gf.E2 = e->ent2 + ENT_PAD;
        // the cold paths of the gather read the same structure from global memory (see mpileup_ent.cuh)
        if (!e->d_gfmt) CK(cudaMalloc(&e->d_gfmt, sizeof(MpEntFmt)));
        CK(cudaMemcpyAsync(e->d_gfmt, &gf, sizeof gf, cudaMemcpyHostToDevice, e->stream));
        const MpEntFmt *dg = (const MpEntFmt *)e->d_gfmt;
        // shared-memory budget of a tile's text: 9/8 of the average tile's upper bound (itself ~1.4x the text; deeper tiles format
        // straight into HBM), at most the configured cap -- a smaller footprint keeps more CTAs resident (30x/150 bp: 16 KB -> 7
        // per SM instead of 5)
        uint32_t cap = e->smem_text;
        {
            const uint64_t avg_tile = bound / (uint64_t)nt;
            const uint64_t want = std::max<uint64_t>(12 * 1024, (avg_tile * 9 / 8 + 1023) & ~1023ull);
            if (want < cap) cap = (uint32_t)want;
        }
        if (c->out_mapq) k_mp_gather<7, true><<<nt, TILE, cap + 16, e->stream>>>(gf, dg, e->col_n, (const MpFileSz *)e->col_state, e->col_off, e->out, cap, e->use_tma);
        else k_mp_gather<7, false><<<nt, TILE, cap + 16, e->stream>>>(gf, dg, e->col_n, (const MpFileSz *)e->col_state, e->col_off, e->out, cap, e->use_tma);
        e->launches++;
        return 0;
    };
    return text_pass(e, nt, bound, sizes, write, out, out_cap, out_len);
}

extern "C" int b200_depth_text(b200_engine_t *e, const b200_depth_conf_t *c, char *out, size_t out_cap, size_t *out_len)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    CK(cudaSetDevice(e->device));
    if (upload_bed(e, c->bed_beg, c->bed_end, c->n_bed, c->bed_active)) return -1;
    DpFmt fmt;
    fill_view(e, fmt.v, e->bed_beg, e->bed_end, c->n_bed, c->bed_active, c->all);
    fmt.cf.min_qual = c->min_qual; fmt.cf.count_del = c->count_del; fmt.cf.all = c->all;
    return run_text(e, k_depth_size, k_depth_write, fmt, depth_bound((uint64_t)fmt.v.ncols, e->name.size(), e->n_files), out, out_cap, out_len);
}
extern "C" uint64_t b200_depth_text_bound(const b200_engine_t *e) { return (e && e->staged) ? depth_bound((uint64_t)e->ncols_max, e->name.size(), e->n_files) : 0; }

extern "C" int b200_coverage(b200_engine_t *e, const b200_coverage_conf_t *c, b200_coverage_sums_t *sums)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    CK(cudaSetDevice(e->device));
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    memset(sums, 0, sizeof *sums);
    CK(cudaMemsetAsync(e->d_misc + 8, 0, 5 * 8, e->stream));
    CK(cudaEventRecord(e->ev0, e->stream));
    if (v.ncols > 0) { k_coverage<<<nblk(v.ncols, 256), 256, 0, e->stream>>>(v, c->min_baseQ, c->min_depth, e->d_misc + 8); e->launches++; }
    CK(cudaEventRecord(e->ev1, e->stream));
    unsigned long long h[5];
    CK(cudaMemcpyAsync(h, e->d_misc + 8, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1); e->last_kernel_ms = ms;
    sums->n_covered_bases = h[0]; sums->summed_coverage = h[1]; sums->summed_baseQ = h[2]; sums->quality_bases = h[3]; sums->missing_qual = h[4];
    return 0;
}

extern "C" int b200_coverage_hist(b200_engine_t *e, const b200_coverage_conf_t *c, int64_t beg, int64_t bin_width, int32_t n_bins, int32_t plot_depth, uint32_t *hist)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    if (!c || !hist || n_bins <= 0 || bin_width <= 0) { snprintf(e->err, sizeof e->err, "bad histogram arguments"); return -1; }
    CK(cudaSetDevice(e->device));
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    if (v.ncols <= 0) return 0;
    ENSURE(gl_n, (size_t)n_bins + 1);                     // int32 scratch shared with the GL path (never live at the same time)
    CK(cudaMemsetAsync(e->gl_n, 0, (size_t)n_bins * 4, e->stream));
    k_coverage_hist<<<nblk(v.ncols, 256), 256, 0, e->stream>>>(v, c->min_baseQ, c->min_depth, beg - e->win_base, bin_width, n_bins, plot_depth != 0, (uint32_t *)e->gl_n); e->launches++;
    std::vector<uint32_t> h((size_t)n_bins);
    CK(cudaMemcpyAsync(h.data(), e->gl_n, (size_t)n_bins * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    for (int32_t k = 0; k < n_bins; ++k) hist[k] += h[(size_t)k];
    return 0;
}

extern "C" int b200_bedcov(b200_engine_t *e, int32_t skip_del_refskip, int32_t min_depth, uint64_t *cnt, uint64_t *pcov)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    CK(cudaSetDevice(e->device));
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    const size_t nf = (size_t)e->n_files;
    for (size_t f = 0; f < nf; ++f) { cnt[f] = 0; if (pcov) pcov[f] = 0; }
    if (v.ncols <= 0) return 0;
    ENSURE(col_off, 2 * nf + 2);
    CK(cudaMemsetAsync(e->col_off, 0, 2 * nf * 8, e->stream));
    CK(cudaEventRecord(e->ev0, e->stream));
    k_bedcov<<<nblk(v.ncols, 256), 256, 0, e->stream>>>(v, (skip_del_refskip || min_depth >= 0) ? 1 : 0, min_depth, (unsigned long long *)e->col_off); e->launches++;
    CK(cudaEventRecord(e->ev1, e->stream));
    std::vector<uint64_t> h(2 * nf);
    CK(cudaMemcpyAsync(h.data(), e->col_off, 2 * nf * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1); e->last_kernel_ms = ms;
    for (size_t f = 0; f < nf; ++f) { cnt[f] = h[2 * f]; if (pcov) pcov[f] = h[2 * f + 1]; }
    return 0;
}

extern "C" int b200_fetch_qual(b200_engine_t *e, uint8_t *qual, size_t cap)
{
    if (!e || !e->staged) return -1;
    CK(cudaSetDevice(e->device));
    size_t nbytes = std::min(cap, e->cap_qual);
    CK(cudaMemcpy(qual, e->qual, nbytes, cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" int b200_fetch_mapq_keep(b200_engine_t *e, uint8_t *mapq, uint8_t *keep, size_t n)
{
    if (!e || !e->staged) return -1;
    CK(cudaSetDevice(e->device));
    n = std::min(n, (size_t)e->n);
    if (mapq) CK(cudaMemcpy(mapq, e->mapq, n, cudaMemcpyDeviceToHost));
    if (keep) CK(cudaMemcpy(keep, e->state, n, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int b200_pileup_entries(b200_engine_t *e, int32_t file, int64_t beg, int64_t end, uint32_t *col_n,
                                   b200_pileup1_t *entries, size_t cap_entries, size_t *n_entries)
{
    if (!e || !e->staged) { if (e) snprintf(e->err, sizeof e->err, "no staged batch"); return -1; }
    CK(cudaSetDevice(e->device));
    if (file < 0 || file >= e->n_files) { snprintf(e->err, sizeof e->err, "bad file index"); return -1; }
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    int64_t rb = beg - e->win_base, re = end - e->win_base;
    if (rb < 0) rb = 0;
    if (re > v.ncols) re = v.ncols;
    *n_entries = 0;
    if (re <= rb) return 0;
    // only the slab [rb,re): counts, their scan and the entries are sized by the slab, not by the contig
    v.ncols = (int32_t)re;
    const int64_t nc = re - rb;
    ENSURE(col_n, (size_t)nc + 1); ENSURE(col_off, (size_t)nc + 2);
    k_entries_count<<<nblk(nc, 256), 256, 0, e->stream>>>(v, file, (int32_t)rb, e->col_n); e->launches++;
    const int nb = nblk(nc, 256);
    ENSURE(status, (size_t)nb + 1);
    CK(cudaMemsetAsync(e->status, 0, ((size_t)nb + 1) * 8, e->stream));
    CK(cudaMemsetAsync(e->d_misc, 0, 8, e->stream));
    k_scan_u32_to_u64<<<nb, 256, 0, e->stream>>>(e->col_n, e->col_off, (int32_t)nc, e->status, (uint32_t *)e->d_misc); e->launches++;
    uint64_t tot = 0;
    CK(cudaMemcpyAsync(&tot, e->col_off + nc, 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    const size_t ne = (size_t)tot;
    *n_entries = ne;
    if (ne > cap_entries) { snprintf(e->err, sizeof e->err, "entry buffer too small: need %zu", ne); return -2; }   // before any fill work
    ENSURE(ents, ne + 1);
    k_entries_fill<<<nblk(nc, 256), 256, 0, e->stream>>>(v, file, (int32_t)rb, e->col_off, e->ents); e->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(col_n, e->col_n, (size_t)nc * 4, cudaMemcpyDeviceToHost, e->stream));
    if (ne) CK(cudaMemcpyAsync(entries, e->ents, ne * sizeof(b200_pileup1_t), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

#include "glf.cuh"
