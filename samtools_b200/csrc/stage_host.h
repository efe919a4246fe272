// stage_host.h -- host-side policy of the read stage and of the text passes, over host arrays.  Plain C++ (no CUDA
// calls): engine.cu runs it around its device copies, the emulation harness in tests/emul/ runs it as is.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <functional>
#include <queue>
#include <vector>
#include "plp_stage.h"

namespace plp {

// max-depth rule of bam_plp_push (sequential by nature; see DESIGN.md): per file, a kept read that starts at the previous
// accepted read's start while more than maxcnt accepted reads are still buffered becomes ST_MAXDROP.  Returns whether any
// read was dropped.
inline bool apply_maxcnt(const ReadDesc *desc, const int32_t *rlen, uint8_t *state, const int64_t *file_start, int n_files, int maxcnt)
{
    bool changed = false;
    for (int f = 0; f < n_files; ++f) {
        std::priority_queue<int32_t, std::vector<int32_t>, std::greater<int32_t>> ends;  // accepted reads still buffered
        bool have_prev = false; int32_t p_prev = 0;
        for (int64_t i = file_start[f]; i < file_start[f + 1]; ++i) {
            if (state[i] != ST_KEEP) continue;
            const int32_t pos = desc[i].rpos, end = desc[i].rpos + rlen[i];
            if (have_prev) {
                while (!ends.empty() && ends.top() < p_prev) ends.pop();   // buffered = accepted reads with end >= previous accepted start
                if (pos == p_prev && (int64_t)ends.size() + 1 > (int64_t)maxcnt) { state[i] = ST_MAXDROP; changed = true; continue; }
            }
            ends.push(end);
            have_prev = true; p_prev = pos;
        }
    }
    return changed;
}

// htslib's bam_plp_push rejects a PUSHED read that starts before the previous pushed read of the same file ("The input is
// not sorted", error return); reads dropped by the filters never reach the push.  The column kernels binary-search the
// descriptors by start, so unsorted input must not get through: exact check over the kept reads of each file.  depth
// (bam2depth.c:329-333) tolerates some disorder; here any disorder among its kept reads is refused ("Data is not position
// sorted") rather than risking silently wrong counts.  Returns the error message, or nullptr when every file is sorted.
inline const char *check_sorted(const ReadDesc *desc, const uint8_t *state, const int64_t *file_start, int n_files, int mode)
{
    for (int f = 0; f < n_files; ++f) {
        bool have = false; int32_t last = 0;
        for (int64_t i = file_start[f]; i < file_start[f + 1]; ++i) {
            if (state[i] != ST_KEEP) continue;
            if (have && desc[i].rpos < last) return mode == B200_MODE_DEPTH ? "Data is not position sorted" : "The input is not sorted (reads out of order)";
            have = true; last = desc[i].rpos;
        }
    }
    return nullptr;
}

// Columns of a staged window, relative to win_base: [0,cov) can hold kept reads (max_rend: 0 if none is kept), [0,all) is
// what -a prints.  Fails, with the message in err, when the window needs more columns than 32-bit indices allow.
inline bool column_domain(int64_t max_rend, int64_t end, int64_t tid_len, int64_t win_base, int64_t &cov, int64_t &all, int32_t &ncols_max,
                          char *err, size_t err_cap)
{
    const int64_t wend = end - win_base;                         // exclusive, relative
    cov = max_rend > 0 ? max_rend : 0;
    if (cov > wend) cov = wend;
    all = (end < tid_len ? end : tid_len) - win_base;
    if (all < 0) all = 0;
    const int64_t nc = cov > all ? cov : all;
    if (nc >= (1LL << 31) - 4096) { snprintf(err, err_cap, "window too wide (%lld columns)", (long long)nc); return false; }
    ncols_max = (int32_t)nc;
    return true;
}

// depth -s: the clip coordinate the caller replayed for a read (absolute, 0: none) as a relative column, clamped to int32
inline int32_t clip_rel(int64_t cabs, int64_t win_base)
{
    int64_t rel = cabs ? cabs - win_base : (int64_t)INT32_MIN;
    if (rel > INT32_MAX) rel = INT32_MAX;
    if (rel < INT32_MIN) rel = INT32_MIN;
    return (int32_t)rel;
}

// text bounds: callers size their output buffers from these, and a text pass that emits more fails (within_bound).
struct TextDims {   // the StageAcc sums, ncols_max, contig name length, files, reads
    uint64_t sum_rlen, sum_indel_text; int64_t ncols; uint64_t name_len; int32_t n_files; int64_t n_reads;
};

// any line-per-column text with at most per_entry bytes per (read, column) entry and per_file_extra more bytes per file
inline uint64_t text_bound(const TextDims &t, int per_entry, int per_file_extra)
{
    return t.sum_rlen * (uint64_t)per_entry + t.sum_indel_text +
           (uint64_t)t.ncols * (t.name_len + 24 + (uint64_t)t.n_files * (16 + (uint64_t)per_file_extra)) + 64;
}

inline uint64_t mpileup_bound(const TextDims &t, const b200_mpileup_conf_t *c)
{
    const int per = 2 + (c->out_mapq ? 1 : 0) + (c->out_qpos ? 12 : 0) + (c->out_qpos5 ? 13 : 0);
    uint64_t b = text_bound(t, per, 1 + 2 * (3 + c->n_star_cols));
    if (c->n_x > 0 && c->x_off) {   // host columns: every (read, column) entry can add the read's strings + separators
        uint64_t worst = 0;
        for (int64_t i = 0; i < t.n_reads; ++i) {
            uint64_t w = 0;
            for (int k = 0; k < c->n_x; ++k) { const uint32_t *o = c->x_off + (size_t)k * ((size_t)t.n_reads + 1) + (size_t)i; w += (uint64_t)(o[1] - o[0]) + 1; }
            if (w > worst) worst = w;
        }
        b += t.sum_rlen * worst;
    }
    return b;
}

// depth rows over ncols columns: name, tab, position, (tab, depth) per file, newline
inline uint64_t depth_bound(uint64_t ncols, uint64_t name_len, int n_files)
{
    return ncols * (name_len + 1 + 20 + (uint64_t)n_files * 12 + 1) + 64;
}

// Returns false, with the message in err, when a text pass emitted more than its bound.
inline bool within_bound(uint64_t total, uint64_t bound, char *err, size_t err_cap)
{
    if (total <= bound) return true;
    snprintf(err, err_cap, "internal: output %llu exceeds bound %llu", (unsigned long long)total, (unsigned long long)bound);
    return false;
}

}  // namespace plp
