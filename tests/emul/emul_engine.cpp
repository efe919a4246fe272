// emul_engine.cpp -- DEBUG HARNESS, NOT PART OF THE PRODUCT.
//
// Implements the C ABI of include/b200_pileup.h by stepping the very same __host__ __device__ per-read / per-column
// functions the CUDA kernels call (samtools_b200/csrc/plp_core.h, plp_stage.h) and the engine's host-side policy
// (stage_host.h).  Of its own it has only sequential loops in place of the kernel grids, a host prefix max in place of the
// device scans, and the cross-checks below (reference implementations).  It exists so that the column arithmetic and the
// host drivers can be debugged on a machine without a GPU.  It is built only by tests/emul/build.sh, is never linked into
// libb200pileup.so or b200samtools, is never used as a fallback, and is not a measured or shipped path.
// BAQ (warp-cooperative kernel) and GL are NOT emulated: calls needing them fail.
#include "../../include/b200_pileup.h"
#include "../../samtools_b200/csrc/stage_host.h"
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace plp;

struct b200_engine {
    std::string err, name;
    b200_batch_t b; b200_stage_conf_t cf;
    std::vector<uint8_t> qual, seq4, mapq, state; std::vector<int32_t> rlen, endv, pmax, glo, ghi, clip, cig_x, cig_y, ovf_off, ovf_idx; std::vector<ReadDesc> desc;
    std::vector<int64_t> next, bedb, bede;
    std::string ref;
    StageAcc acc;
    int64_t win_base = 0, ncols_cov = 0, ncols_all = 0; int32_t ncols_max = 0, n_groups = 0;
    bool staged = false, has_clip = false;
};

extern "C" {
const char *b200_version(void) { return "emulation harness (debug only)"; }
const char *b200_last_error(const b200_engine_t *e) { return e->err.c_str(); }
double b200_last_kernel_ms(const b200_engine_t *) { return 0; }
double b200_last_stage_ms(const b200_engine_t *) { return 0; }
int64_t b200_launch_count(const b200_engine_t *) { return 0; }
uint64_t b200_gl_rng_draws(const b200_engine_t *) { return 0; }
double b200_last_baq_ms(const b200_engine_t *) { return 0; }
void b200_last_mpileup_parts_ms(const b200_engine_t *, double *ms3) { ms3[0] = ms3[1] = ms3[2] = 0; }
int b200_engine_create(int, b200_engine_t **out) { *out = new b200_engine(); return 0; }
void b200_engine_destroy(b200_engine_t *e) { delete e; }

static RawSoA raw(b200_engine *e)
{
    const b200_batch_t &b = e->b;
    RawSoA r;
    r.pos = b.pos; r.flag = b.flag; r.mapq = e->mapq.data(); r.l_qseq = b.l_qseq; r.n_cigar = b.n_cigar; r.cigar_off = b.cigar_off;
    r.qual_off = b.qual_off; r.mtid = b.mtid; r.mpos = b.mpos; r.isize = b.isize; r.prev = b.prev_same_name; r.rbits = b.rbits;
    r.cigar = b.cigar; r.seq4 = e->seq4.data(); r.qual = e->qual.data();
    r.ref = b.ref && b.ref_len > 0 ? e->ref.data() : nullptr; r.ref_beg = b.ref_beg; r.ref_n = b.ref_n; r.ref_len = r.ref ? b.ref_len : 0;
    r.n = b.n_reads; r.tid = b.tid;
    return r;
}

// k_scan_max + k_ranges + k_ovf_*: a host prefix max in place of the device scan, then the same group_slice / ovf_span
static void build_ranges(b200_engine *e, int *max_range)
{
    const b200_batch_t &b = e->b;
    const int64_t n = b.n_reads;
    e->pmax.assign((size_t)n + 1, INT32_MIN);
    for (int f = 0; f < b.n_files; ++f) {
        int32_t m = INT32_MIN;
        for (int64_t i = b.file_start[f]; i < b.file_start[f + 1]; ++i) { m = std::max(m, e->endv[(size_t)i]); e->pmax[(size_t)i] = m; }
    }
    e->glo.assign((size_t)e->n_groups * b.n_files + 1, 0); e->ghi = e->glo;
    *max_range = 0;
    for (int f = 0; f < b.n_files; ++f)
        for (int g = 0; g < e->n_groups; ++g) {
            int64_t first, last;
            group_slice(e->desc.data(), e->pmax.data(), b.file_start[f], b.file_start[f + 1], g, first, last);
            e->glo[(size_t)f * e->n_groups + g] = (int32_t)first; e->ghi[(size_t)f * e->n_groups + g] = (int32_t)last;
            *max_range = std::max(*max_range, (int)(last - first));
        }
    // far-reaching reads per group, in file order
    std::vector<std::vector<int32_t>> lists((size_t)e->n_groups * b.n_files);
    for (int f = 0; f < b.n_files; ++f)
        for (int64_t i = b.file_start[f]; i < b.file_start[f + 1]; ++i) {
            int32_t g0, g1;
            if (!ovf_span(e->desc[(size_t)i], e->n_groups, g0, g1)) continue;
            for (int32_t g = g0; g <= g1; ++g) lists[(size_t)f * e->n_groups + g].push_back((int32_t)i);
        }
    { size_t mo = 0; for (auto &l : lists) mo = std::max(mo, l.size()); *max_range += (int)mo; }
    e->ovf_off.assign(lists.size() + 2, 0); e->ovf_idx.clear();
    for (size_t k = 0; k < lists.size(); ++k) { e->ovf_off[k] = (int32_t)e->ovf_idx.size(); e->ovf_idx.insert(e->ovf_idx.end(), lists[k].begin(), lists[k].end()); }
    e->ovf_off[lists.size()] = (int32_t)e->ovf_idx.size(); e->ovf_off[lists.size() + 1] = (int32_t)e->ovf_idx.size();
    e->ovf_idx.push_back(0);
}

static TextDims text_dims(const b200_engine *e) { return {e->acc.sum_rlen, e->acc.sum_indel_text, e->ncols_max, e->name.size(), e->b.n_files, e->b.n_reads}; }

int b200_stage(b200_engine_t *e, const b200_batch_t *b, const b200_stage_conf_t *cf, b200_stage_stats_t *stats)
{
    e->b = *b; e->cf = *cf; e->name = b->tid_name ? b->tid_name : "";
    const int64_t n = b->n_reads;
    e->qual.assign(b->qual, b->qual + b->qual_bytes); e->qual.resize(b->qual_bytes + 16, 0);
    e->seq4.assign(b->seq4, b->seq4 + (b->qual_bytes + 1) / 2 + 1); e->seq4.resize(e->seq4.size() + 16, 0);
    e->mapq.assign(b->mapq, b->mapq + n); e->mapq.resize((size_t)n + 1);
    e->ref.assign(b->ref ? b->ref : "", b->ref ? (size_t)b->ref_n : 0);
    e->state.assign((size_t)n + 1, 0); e->rlen.assign((size_t)n + 1, 0); e->desc.assign((size_t)n + 1, ReadDesc());
    e->endv.assign((size_t)n + 1, INT32_MIN);
    e->cig_x.assign((size_t)b->n_cigar_total + 1, 0); e->cig_y.assign((size_t)b->n_cigar_total + 1, 0);
    memset(&e->acc, 0, sizeof e->acc); e->acc.max_rend = INT32_MIN;
    e->win_base = cf->beg > 0 ? cf->beg : 0;
    RawSoA r = raw(e);
    for (int64_t i = 0; i < n; ++i) stage_prep1(r, *cf, i, e->state.data(), e->rlen.data(), &e->acc);
    if (cf->mode == B200_MODE_MPILEUP && cf->baq && r.ref) {
        for (int64_t i = 0; i < n; ++i)
            if (e->state[(size_t)i] == ST_ALIVE && !(b->rbits && (b->rbits[i] & B200_RB_BAQ_DONE)) && b->l_qseq[i] > 0 && e->qual[b->qual_off[i]] != 0xff) {
                e->err = "emulation harness: the BAQ kernel is not emulated"; return -1;
            }
    }
    for (int64_t i = 0; i < n; ++i) stage_prep2(r, *cf, i, e->state.data());
    for (int64_t i = 0; i < n; ++i) stage_build_desc(r, *cf, i, e->state.data(), e->rlen.data(), e->desc.data(), e->endv.data(), &e->acc, e->win_base, e->cig_x.data(), e->cig_y.data());
    if (e->acc.n_desc)
        if (const char *msg = check_sorted(e->desc.data(), e->state.data(), b->file_start, b->n_files, cf->mode)) { e->err = msg; return -3; }
    char msg[128];
    if (!column_domain(e->acc.n_kept ? e->acc.max_rend : 0, cf->end, b->tid_len, e->win_base, e->ncols_cov, e->ncols_all, e->ncols_max, msg, sizeof msg)) {
        e->err = msg; return -1;
    }
    e->n_groups = (e->ncols_max + 31) / 32 + 1;
    int max_range = 0;
    build_ranges(e, &max_range);
    if (cf->mode != B200_MODE_DEPTH && cf->max_depth > 0 && 2LL * max_range + 1 > (int64_t)cf->max_depth) {
        if (apply_maxcnt(e->desc.data(), e->rlen.data(), e->state.data(), b->file_start, b->n_files, cf->max_depth)) {
            for (int64_t i = 0; i < n; ++i) if (e->state[(size_t)i] == ST_MAXDROP) { e->desc[(size_t)i].rend = e->desc[(size_t)i].rpos; e->endv[(size_t)i] = INT32_MIN; }
            build_ranges(e, &max_range);
        }
    }
    e->has_clip = false;
    if (cf->mode == B200_MODE_DEPTH && cf->d_remove_overlaps && b->depth_clip) {
        e->clip.assign((size_t)n + 1, INT32_MIN);
        for (int64_t i = 0; i < n; ++i) e->clip[(size_t)i] = clip_rel(b->depth_clip[i], e->win_base);
        e->has_clip = true;
    } else if (b->prev_same_name && ((cf->mode == B200_MODE_MPILEUP && cf->overlaps) || (cf->mode == B200_MODE_DEPTH && cf->d_remove_overlaps))) {
        e->next.assign((size_t)n + 1, -1);
        for (int64_t i = 0; i < n; ++i) if (b->prev_same_name[i] >= 0) e->next[(size_t)b->prev_same_name[i]] = i;
        if (cf->mode == B200_MODE_MPILEUP) {
            int bad = 0;   // cross-check of the device's simple-pair fast path (plp_stage.h overlap_span_simple / tweak_pos)
            for (int64_t i = 0; i < n; ++i) overlap_chain(r, i, e->next.data(), e->state.data(), e->rlen.data(), b->file_start, b->n_files, nullptr, nullptr, e->desc.data(), &bad);
            if (bad) { e->err = "emulation harness: per-position overlap tweak differs from the lock-step walk"; return -1; }
        } else {
            e->clip.assign((size_t)n + 1, INT32_MIN);
            for (int64_t i = 0; i < n; ++i) depth_clip_chain(r, i, e->next.data(), e->state.data(), e->rlen.data(), e->clip.data(), e->win_base);
            e->has_clip = true;
        }
    }
    e->staged = true;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_kept = (int64_t)e->acc.n_kept; stats->n_kept_in_window = (int64_t)e->acc.n_kept_in_window;
        stats->n_reads = e->acc.n_reads; stats->n_selected_reads = e->acc.n_selected; stats->summed_mapq = e->acc.summed_mapq;
        stats->out_bound = text_bound(text_dims(e), 27, 1); stats->n_cols = e->ncols_max;
    }
    return 0;
}

static void fill_view(b200_engine *e, View &v, const int64_t *bb, const int64_t *be, int nb, int active, int all)
{
    const b200_batch_t &b = e->b;
    v.desc = e->desc.data(); v.cigar = b.cigar; v.cig_x = e->cig_x.data(); v.cig_y = e->cig_y.data(); v.seq4 = e->seq4.data(); v.qual = e->qual.data();
    v.clip = e->has_clip ? e->clip.data() : nullptr;
    v.ref = (b.ref && b.ref_len > 0) ? e->ref.data() : nullptr;
    v.ref_off = b.ref_beg - e->win_base; v.ref_n = b.ref_n; v.ref_len_rel = (v.ref ? b.ref_len : 0) - e->win_base;
    v.n_files = b.n_files; v.file_start = b.file_start; v.tile_lo = e->glo.data(); v.tile_hi = e->ghi.data(); v.ovf_off = e->ovf_off.data(); v.ovf_idx = e->ovf_idx.data();
    v.n_tiles = e->n_groups; v.tile_cols = 32; v.win_base = e->win_base;
    v.ncols_all = all ? (int32_t)e->ncols_all : 0;
    v.ncols = (int32_t)(all ? std::max(e->ncols_cov, e->ncols_all) : e->ncols_cov);
    v.name = e->name.c_str(); v.name_len = (int32_t)e->name.size();
    v.bed_beg = bb; v.bed_end = be; v.n_bed = nb; v.bed_active = active;
    v.n_x = 0; v.x_stride = 0; v.x_off = nullptr; v.x_dat = nullptr; memset(v.x_sep, 0, sizeof v.x_sep);
}

// the tail of the engine's text pass: bound check, then the copy-out
static int emit(b200_engine *e, const std::string &s, uint64_t bound, char *out, size_t cap, size_t *out_len)
{
    char msg[128];
    if (!within_bound(s.size(), bound, msg, sizeof msg)) { e->err = msg; return -1; }
    *out_len = s.size();
    if (out) { if (s.size() > cap) { e->err = "output buffer too small"; return -2; } memcpy(out, s.data(), s.size()); }
    return 0;
}

int b200_mpileup_text(b200_engine_t *e, const b200_mpileup_conf_t *c, char *out, size_t cap, size_t *out_len)
{
    View v; fill_view(e, v, c->bed_beg, c->bed_end, c->n_bed, c->bed_active, c->all);
    MpConf cf{c->min_baseQ, c->all, c->rev_del, c->no_ins, c->no_del, c->no_ends, c->out_mapq, c->out_qpos, c->out_qpos5, c->n_star_cols};
    std::string s;
    // default path (one file, no -O columns): sequential replay of mpileup_ent.cuh -- the read-major entry pass (scalar
    // walk over the same per-base functions), the order-free line sizes, then mp_line_write_ent per column.
    // EMUL_GENERAL=1 replays the general path (mp_line_size + mp_line_write) like B200_PLP_GENERAL=1 on the device.
    const char *gen = getenv("EMUL_GENERAL");
    if (c->n_x > 0) { v.n_x = c->n_x; v.x_stride = e->b.n_reads + 1; v.x_off = c->x_off; v.x_dat = c->x_dat; memcpy(v.x_sep, c->x_sep, sizeof v.x_sep); }
    const bool use_ent = !(gen && atoi(gen) == 1) && v.n_files == 1 && !cf.out_qpos && !cf.out_qpos5 && c->n_x == 0;
    std::vector<uint16_t> E, E2; std::vector<int32_t> diff; std::vector<uint32_t> fail, extra;
    if (use_ent) {
        const uint8_t *tab = (const uint8_t *)".ACMGRSVTWYHKDBN,acmgrsvtwyhkdbn";
        E.assign(e->qual.size() + 16, 0xdead); diff.assign((size_t)v.ncols + 2, 0); fail.assign((size_t)v.ncols + 1, 0); extra.assign((size_t)v.ncols + 1, 0);
        size_t e2n = 0;
        for (int64_t i = 0; i < e->b.n_reads; ++i) { const ReadDesc &d = e->desc[(size_t)i]; if (d.rend > d.rpos && !(d.fl & RD_SIMPLE)) e2n += (size_t)(d.rend - d.rpos); }
        E2.assign(e2n + 16, 0xdead);
        size_t cursor = 0;
        for (int64_t i = 0; i < e->b.n_reads; ++i) {
            ReadDesc &d = e->desc[(size_t)i];
            if (d.rend <= d.rpos) continue;
            const int32_t a = d.rpos > 0 ? d.rpos : 0, b = d.rend < v.ncols ? d.rend : v.ncols;
            if (a >= b) continue;
            diff[(size_t)a] += 1; diff[(size_t)b] -= 1;
            const uint32_t rev = (d.fl & RD_REV) ? 1u : 0u;
            if (d.fl & RD_SIMPLE) {
                const uint32_t q0 = d.qoff + (uint32_t)d.qstart, qtail = q0 + (uint32_t)(d.rend - d.rpos) - 1u;
                for (int32_t c = a; c < b; ++c) {
                    const uint32_t qi = q0 + (uint32_t)(c - d.rpos);
                    uint32_t fl = 0;
                    if (!cf.no_ends) fl = (qi == q0 ? 0x80u : 0u) | (qi == qtail ? 0x8000u : 0u);
                    const uint32_t x = ent_plain(v.qual[qi], (uint32_t)base4(v.seq4, 0, (int32_t)qi), ent_ref_code(v, c), rev, cf.min_baseQ, fl, tab);
                    E[qi] = (uint16_t)x;
                    if (!x) fail[(size_t)c]++;
                    else if (fl) extra[(size_t)c] += ((fl & 0x80u) ? 2u : 0u) + ((fl & 0x8000u) ? 1u : 0u);
                }
                // cross-check of the SIMD-in-word formatter the device entry pass uses (ent_group8_swar) against the per-base ent_plain
                if (cf.min_baseQ <= 127) {
                    const uint32_t lo = q0 + (uint32_t)(a - d.rpos), hi = q0 + (uint32_t)(b - d.rpos);
                    const EntTab etab = ent_tab(rev);
                    const uint32_t minq4 = (uint32_t)(cf.min_baseQ > 0 ? cf.min_baseQ : 0) * 0x01010101u;
                    for (uint32_t g = lo & ~7u; g < hi; g += 8) {
                        uint32_t qx = 0, qy = 0, s4 = 0, r8 = 0;
                        for (uint32_t k = 0; k < 8; ++k) {
                            const size_t qi = (size_t)g + k;
                            const uint32_t q = qi < e->qual.size() ? e->qual[qi] : 0;
                            if (k < 4) qx |= q << (8 * k); else qy |= q << (8 * (k - 4));
                            const int32_t cc = d.rpos + (int32_t)(g + k - q0);
                            r8 |= (ent_ref_code(v, cc) & 0xfu) << (4 * k);
                        }
                        for (uint32_t k = 0; k < 4; ++k) { const size_t bi = (size_t)(g >> 1) + k; s4 |= (uint32_t)(bi < e->seq4.size() ? e->seq4[bi] : 0) << (8 * k); }
                        uint32_t w[4];
                        const uint32_t fm = ent_group8_swar(qx, qy, s4, v.ref != nullptr, r8, etab, minq4, w);
                        for (uint32_t k = 0; k < 8; ++k) {
                            const uint32_t qi = g + k;
                            if (qi < lo || qi >= hi) continue;
                            const uint32_t got = (w[k >> 1] >> (16 * (k & 1))) & 0xffffu, want = E[qi] & 0x7f7fu;
                            if (got != want || (((fm >> k) & 1u) != (want == 0 ? 1u : 0u))) {
                                e->err = "emulation harness: ent_group8_swar differs from ent_plain at query index " + std::to_string(qi); return -1;
                            }
                        }
                    }
                }
            } else {
                d.pad_ = (uint32_t)cursor; cursor += (size_t)(d.rend - d.rpos);
                for (int32_t c = a; c < b; ++c) {
                    uint32_t xb;
                    const uint32_t x = ent_generic(v, cf, d, c, ent_ref_code(v, c), tab, xb);
                    E2[d.pad_ + (uint32_t)(c - d.rpos)] = (uint16_t)x;
                    if (!x) fail[(size_t)c]++; else extra[(size_t)c] += xb;
                }
            }
        }
    }
    int32_t cov = 0;
    for (int32_t col = 0; col < v.ncols; ++col) {
        MpFileSz s0;
        uint32_t len = mp_line_size(v, cf, col >> 5, col, s0);
        if (use_ent) {   // the sums the device derives the line length from must reproduce mp_line_size
            cov += diff[(size_t)col];
            MpFileSz s1; s1.nplp = cov; s1.cnt = cov - (int32_t)fail[(size_t)col]; s1.seq_len = (uint32_t)s1.cnt + extra[(size_t)col]; s1.bp_len = 0; s1.bp5_len = 0;
            uint32_t len1 = 0;
            if ((s1.nplp > 0 || (cf.all && col < v.ncols_all)) && bed_pass(v, col)) len1 = mp_head_len(v, col) + mp_file_section_len(cf, s1) + 1;
            if (len1 != len || (len && (s1.nplp != s0.nplp || s1.cnt != s0.cnt || s1.seq_len != s0.seq_len))) {
                e->err = "emulation harness: order-free line size differs from mp_line_size at column " + std::to_string(col); return -1;
            }
            s0 = s1;
        }
        if (!len) continue;
        size_t at = s.size(); s.resize(at + len, '?');
        if (use_ent) mp_line_write_ent(v, cf, col, s0, &s[at], E.data(), E2.data());
        else mp_line_write(v, cf, col >> 5, col, s0, &s[at]);
    }
    return emit(e, s, mpileup_bound(text_dims(e), c), out, cap, out_len);
}

uint64_t b200_mpileup_text_bound(const b200_engine_t *e, const b200_mpileup_conf_t *c) { return e->staged && c ? mpileup_bound(text_dims(e), c) : 0; }
uint64_t b200_depth_text_bound(const b200_engine_t *e) { return e->staged ? depth_bound((uint64_t)e->ncols_max, e->name.size(), e->b.n_files) : 0; }
int b200_depth_text(b200_engine_t *e, const b200_depth_conf_t *c, char *out, size_t cap, size_t *out_len)
{
    DpFmt fmt; fill_view(e, fmt.v, c->bed_beg, c->bed_end, c->n_bed, c->bed_active, c->all);
    fmt.cf = DpConf{c->min_qual, c->count_del, c->all};
    std::string s;
    for (int32_t col = 0; col < fmt.v.ncols; ++col) {
        DpFmt::State st{};
        const uint32_t len = fmt.size(col, st);
        if (!len) continue;
        const size_t at = s.size(); s.resize(at + len, '?');
        fmt.write(col, st, &s[at]);
    }
    return emit(e, s, depth_bound((uint64_t)fmt.v.ncols, e->name.size(), fmt.v.n_files), out, cap, out_len);
}

int b200_coverage(b200_engine_t *e, const b200_coverage_conf_t *c, b200_coverage_sums_t *sums)
{
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    memset(sums, 0, sizeof *sums);
    for (int32_t col = 0; col < v.ncols; ++col) {
        CvCol o; cv_column(v, c->min_baseQ, col >> 5, col, o);
        sums->missing_qual += o.missing;
        if (o.count_base && o.depth >= (uint32_t)c->min_depth) { sums->n_covered_bases++; sums->summed_coverage += o.depth; sums->summed_baseQ += o.sum_bq; sums->quality_bases += o.qbases; }
    }
    return 0;
}
int b200_coverage_hist(b200_engine_t *e, const b200_coverage_conf_t *c, int64_t beg, int64_t bin_width, int32_t n_bins, int32_t plot_depth, uint32_t *hist)
{
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    for (int32_t col = 0; col < v.ncols; ++col) {
        CvCol o; cv_column(v, c->min_baseQ, col >> 5, col, o);
        const uint32_t add = cv_hist_add(o, c->min_depth, plot_depth);
        const int64_t bin = ((int64_t)col - (beg - v.win_base)) / bin_width;
        if (add && bin >= 0 && bin < n_bins) hist[bin] += add;
    }
    return 0;
}
int b200_bedcov(b200_engine_t *e, int32_t skip_dn, int32_t min_depth, uint64_t *cnt, uint64_t *pcov)
{
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    const int dn = skip_dn || min_depth >= 0;
    for (int f = 0; f < v.n_files; ++f) { cnt[f] = 0; if (pcov) pcov[f] = 0; }
    for (int32_t c = 0; c < v.ncols; ++c) {
        if (!bc_any(v, c)) continue;
        for (int f = 0; f < v.n_files; ++f) {
            const int32_t d = bc_depth(v, f, c, dn);
            cnt[f] += (uint64_t)d;
            if (pcov && min_depth >= 0 && d >= min_depth) pcov[f]++;
        }
    }
    return 0;
}
int b200_glf(b200_engine_t *e, int32_t, int64_t *, int64_t *, int32_t *, float *, float *, size_t) { e->err = "emulation harness: GL not emulated"; return -1; }
int b200_fetch_qual(b200_engine_t *e, uint8_t *q, size_t cap) { memcpy(q, e->qual.data(), std::min(cap, e->qual.size())); return 0; }
int b200_fetch_mapq_keep(b200_engine_t *e, uint8_t *m, uint8_t *k, size_t n) { n = std::min(n, (size_t)e->b.n_reads); if (m) memcpy(m, e->mapq.data(), n); if (k) memcpy(k, e->state.data(), n); return 0; }
// column-major (read, column) entries: column_entries per column, counts first (k_entries_count / k_entries_fill in engine.cu)
int b200_pileup_entries(b200_engine_t *e, int32_t file, int64_t beg, int64_t end, uint32_t *col_n, b200_pileup1_t *ents, size_t cap, size_t *n_out)
{
    if (!e->staged) { e->err = "no staged batch"; return -1; }
    if (file < 0 || file >= e->b.n_files) { e->err = "bad file index"; return -1; }
    View v; fill_view(e, v, nullptr, nullptr, 0, 0, 0);
    int64_t rb = beg - e->win_base, re = end - e->win_base;
    if (rb < 0) rb = 0;
    if (re > v.ncols) re = v.ncols;
    *n_out = 0;
    if (re <= rb) return 0;
    size_t ne = 0;
    for (int64_t c = rb; c < re; ++c) { col_n[c - rb] = column_entries<false>(v, file, (int32_t)c, nullptr); ne += col_n[c - rb]; }
    *n_out = ne;
    if (ne > cap) { e->err = "entry buffer too small"; return -2; }
    for (int64_t c = rb; c < re; ++c) ents += column_entries<true>(v, file, (int32_t)c, ents);
    return 0;
}
}
