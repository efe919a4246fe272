// plp_stage.h -- per-read stage arithmetic (filters, geometry, descriptors,
// mate-overlap replay) as __host__ __device__ functions; the kernels in
// engine.cu / overlap.cuh are thin wrappers.  See plp_core.h for why.
//
// Reference behaviour restated here (file:line into /root/reference):
//   stage_prep1   mplp_func pre-BAQ filters  bam_plcmd.c:413-445
//                 fastdepth_core filters      bam2depth.c:552-570, qlen_used :124-159
//                 read_bam filters + stats    coverage.c:185-193
//   cap_mapq      htslib realn.c sam_cap_mapq (doc/samtools-mpileup.1:219-241)
//   stage_prep2   mplp_func post-BAQ filters bam_plcmd.c:452-458
//   tweak_overlap htslib sam.c tweak_overlap_quality (doc/samtools-mpileup.1:353-365)
//   overlap_chain htslib sam.c overlap_push / overlap_remove
//   depth_clip_chain  olap_hash logic         bam2depth.c:598-623
#pragma once
#include <math.h>
#include "../../include/b200_pileup.h"
#include "plp_core.h"

// The per-read functions add into a StageAcc that is PRIVATE to the caller (a thread-local copy in
// the kernels, which then merge with one warp-reduced atomic per warp: five atomics per read on the
// same five addresses serialise in L2 and cost ~1 ms per 800 k reads; the emulation harness passes
// its single accumulator directly).
#define PLP_ADD64(p, v) (*(p) += (unsigned long long)(v))
#define PLP_MAX32(p, v) (*(p) = *(p) > (int)(v) ? *(p) : (int)(v))

namespace plp {

struct RawSoA {
    const int64_t *pos; const uint16_t *flag; uint8_t *mapq; const int32_t *l_qseq; const uint32_t *n_cigar;
    const uint64_t *cigar_off, *qual_off; const int32_t *mtid; const int64_t *mpos, *isize, *prev; const uint8_t *rbits;
    const uint32_t *cigar; const uint8_t *seq4; uint8_t *qual;
    const char *ref; int64_t ref_beg, ref_n, ref_len;
    int64_t n; int32_t tid;
};

struct StageAcc {   // device-side accumulators (one instance per stage call)
    unsigned long long n_kept, n_kept_in_window, sum_rlen, sum_indel_text, n_reads, n_selected, summed_mapq;
    unsigned long long sum_rlen_gen;   // reference span of the kept reads that are not of the simple shape (entries of the second array, mpileup_ent.cuh)
    unsigned long long n_desc;   // records whose start lies before the previous record's (any file, any state): triggers the exact sortedness check
    int max_rend;
};

enum { ST_DEAD = 0, ST_ALIVE = 1, ST_KEEP = 2, ST_MAXDROP = 3 };

// geometry + filters that precede BAQ (bam_plcmd.c:413-445; bam2depth.c:552-570; coverage.c:185-190)
PLP_HD void stage_prep1(const RawSoA &r, const b200_stage_conf_t &cf, int64_t i, uint8_t *state, int32_t *rlen_out, StageAcc *acc)
{
    const uint16_t fl = r.flag[i];
    const uint8_t rb = r.rbits ? r.rbits[i] : 0;
    const uint32_t *cg = r.cigar + r.cigar_off[i];
    const int n = (int)r.n_cigar[i];
    int32_t rl = 0;
    for (int k = 0; k < n; ++k) { int op = cg[k] & 0xf; if (is_refop(op)) rl += (int)(cg[k] >> 4); }
    rlen_out[i] = rl;
    bool alive = true;
    if (cf.mode == B200_MODE_MPILEUP) {
        if (fl & 4) alive = false;
        if (cf.rflag_require && !(cf.rflag_require & fl)) alive = false;
        if (cf.rflag_filter && (cf.rflag_filter & fl)) alive = false;
        if (rb & B200_RB_HOST_SKIP) alive = false;
        if (alive && cf.illumina13 && !(rb & B200_RB_BAQ_DONE)) {   // host already applied -6 before its BQ:Z integer path
            uint8_t *q = r.qual + r.qual_off[i];
            for (int j = 0; j < r.l_qseq[i]; ++j) q[j] = q[j] > 31 ? q[j] - 31 : 0;
        }
        if (r.ref_len > 0 && r.ref_len <= r.pos[i]) alive = false;   // "outside of the reference" skip
    } else if (cf.mode == B200_MODE_DEPTH) {
        if (fl & cf.d_flag_excl) alive = false;
        if (cf.d_flag_incl && (fl & cf.d_flag_incl) == 0) alive = false;
        if ((fl & cf.d_flag_require) != cf.d_flag_require) alive = false;
        if (r.mapq[i] < cf.d_min_mapq) alive = false;
        if (alive && cf.d_min_len) {   // qlen_used (bam2depth.c:124-159)
            int64_t l;
            if (r.l_qseq[i]) {
                l = r.l_qseq[i];
                int kl, kr;
                for (kl = 0; kl < n; kl++) { if ((cg[kl] & 0xf) == OP_S) l -= cg[kl] >> 4; else break; }
                for (kr = n - 1; kr > kl; kr--) { if ((cg[kr] & 0xf) == OP_S) l -= cg[kr] >> 4; else break; }
            } else {
                l = 0;
                for (int k = 0; k < n; k++) { int op = cg[k] & 0xf; if (op == OP_M || op == OP_I || op == OP_EQ || op == OP_X) l += cg[k] >> 4; }
            }
            if (l < cf.d_min_len) alive = false;
        }
    } else {  // coverage
        const bool counted = !(rb & B200_RB_HALO);   // a read staged again by the next column window is counted once
        if (counted) PLP_ADD64(&acc->n_reads, 1);
        if (cf.rflag_filter && (fl & cf.rflag_filter)) alive = false;
        if (cf.rflag_require && !(fl & cf.rflag_require)) alive = false;
        if (r.mapq[i] < cf.min_mq) alive = false;
        if (alive && cf.c_min_len) {
            int64_t l = 0;
            for (int k = 0; k < n; k++) { int op = cg[k] & 0xf; if (op == OP_M || op == OP_I || op == OP_S || op == OP_EQ || op == OP_X) l += cg[k] >> 4; }
            if (l < cf.c_min_len) alive = false;
        }
        if (alive && counted) { PLP_ADD64(&acc->n_selected, 1); PLP_ADD64(&acc->summed_mapq, r.mapq[i]); }
        if (fl & 4) alive = false;   // bam_plp_push ignores unmapped reads
    }
    state[i] = alive ? ST_ALIVE : ST_DEAD;
}

// sam_cap_mapq (htslib realn.c; formula doc/samtools-mpileup.1:219-241)
PLP_HD int cap_mapq(const RawSoA &r, int64_t i, int thres)
{
    const uint8_t *qual = r.qual + r.qual_off[i];
    const uint64_t qoff = r.qual_off[i];
    const uint32_t *cg = r.cigar + r.cigar_off[i];
    const int n = (int)r.n_cigar[i];
    int y = 0, mm = 0, q = 0, len = 0, clip_q = 0;
    int64_t x = r.pos[i];
    if (thres < 0) thres = 40;
    for (int k = 0; k < n; ++k) {
        int j, l = (int)(cg[k] >> 4), op = cg[k] & 0xf;
        if (is_mop(op)) {
            for (j = 0; j < l; ++j) {
                int z = y + j;
                int64_t rp = x + j;
                if (rp >= r.ref_len) break;
                int64_t ri = rp - r.ref_beg;
                char rc = (ri >= 0 && ri < r.ref_n) ? r.ref[ri] : 'N';
                if (rc == '\0') break;
                int c1 = base4(r.seq4, qoff, z), c2 = nt16_of((unsigned char)rc);
                if (c2 != 15 && c1 != 15 && qual[z] >= 13) {
                    ++len;
                    if (c1 && c1 != c2 && qual[z] >= 13) { ++mm; q += qual[z] > 33 ? 33 : qual[z]; }
                }
            }
            if (j < l) break;
            x += l; y += l; len += l;
        } else if (op == OP_D) {
            for (j = 0; j < l; ++j) if (x + j >= r.ref_len) break;
            if (j < l) break;
            x += l;
        } else if (op == OP_S) { for (j = 0; j < l; ++j) clip_q += qual[y + j]; y += l; }
        else if (op == OP_H) clip_q += 13 * l;
        else if (op == OP_I) y += l;
        else if (op == OP_N) x += l;
    }
    double t = 1;
    for (int k = 0; k < mm; ++k) t *= (double)len / (k + 1);
    t = q - 4.343 * log(t) + clip_q / 5.;
    if (t > thres) return -1;
    if (t < 0) t = 0;
    t = sqrt((thres - t) / thres) * thres;
    return (int)(t + .499);
}

// filters that follow BAQ (bam_plcmd.c:452-458)
PLP_HD void stage_prep2(const RawSoA &r, const b200_stage_conf_t &cf, int64_t i, uint8_t *state)
{
    if (state[i] != ST_ALIVE) return;
    bool keep = true;
    if (cf.mode == B200_MODE_MPILEUP) {
        const uint16_t fl = r.flag[i];
        if (r.ref && r.ref_len > 0 && cf.capq_thres > 10) {
            int q = cap_mapq(r, i, cf.capq_thres);
            if (q < 0) keep = false;
            else if (r.mapq[i] > q) r.mapq[i] = (uint8_t)q;
        }
        if (r.mapq[i] < cf.min_mq) keep = false;
        else if (cf.no_orphan && (fl & 1) && !(fl & 2)) keep = false;
    }
    state[i] = keep ? ST_KEEP : ST_DEAD;
}

// read descriptors + batch statistics
PLP_HD void stage_build_desc(const RawSoA &r, const b200_stage_conf_t &cf, int64_t i, const uint8_t *state, const int32_t *rlen,
                             ReadDesc *desc, int32_t *endv, StageAcc *acc, int64_t win_base,
                             int32_t *cig_x, int32_t *cig_y)
{
    const uint32_t *cg = r.cigar + r.cigar_off[i];
    const int n = (int)r.n_cigar[i];
    ReadDesc d;
    d.rpos = (int32_t)(r.pos[i] - win_base);
    const bool keep = state[i] == ST_KEEP;
    int32_t rl = rlen[i];
    int32_t span = rl;
    if (cf.mode == B200_MODE_DEPTH) span = ((r.flag[i] & 4) || n == 0 || rl == 0) ? 1 : rl;   // bam_endpos
    d.rend = keep ? d.rpos + span : d.rpos;
    d.qoff = (uint32_t)r.qual_off[i];
    d.cig_off = (uint32_t)r.cigar_off[i];
    d.l_qseq = r.l_qseq[i];
    d.n_cigar = (uint32_t)n; d.pad_ = 0;
    d.mapq = r.mapq[i];
    d.fl = (r.flag[i] & 16) ? RD_REV : 0;
    d.qstart = 0;
    // simple shape: [H]*[S]?(M|=|X)[S]?[H]*
    {
        int k = 0, qs = 0;
        while (k < n && (cg[k] & 0xf) == OP_H) ++k;
        if (k < n && (cg[k] & 0xf) == OP_S) { qs = (int)(cg[k] >> 4); ++k; }
        if (k < n && is_mop(cg[k] & 0xf) && (int)(cg[k] >> 4) == rl && rl > 0) {
            ++k;
            if (k < n && (cg[k] & 0xf) == OP_S) ++k;
            while (k < n && (cg[k] & 0xf) == OP_H) ++k;
            if (k == n && qs <= 65535 && qs + rl <= r.l_qseq[i]) { d.fl |= RD_SIMPLE; d.qstart = (uint16_t)qs; }
        }
    }
    if (n > kCigarWalkMax) {   // per-op prefix arrays for long CIGARs (see plp_core.h locate())
        int32_t x = d.rpos, y = 0;
        for (int k = 0; k < n; ++k) {
            const int op = cg[k] & 0xf; const int len = (int)(cg[k] >> 4);
            cig_x[d.cig_off + k] = x; cig_y[d.cig_off + k] = y;
            if (is_refop(op)) { x += len; if (is_mop(op)) y += len; }
            else if (op == OP_I || op == OP_S) y += len;
        }
    }
    desc[i] = d;
    if (i > 0 && r.pos[i] < r.pos[i - 1]) PLP_ADD64(&acc->n_desc, 1);   // bam_plp_push rejects unsorted input; see check_sorted() in stage_host.h
    // end used for the running max that bounds the per-group read slices: capped at rpos + kReach, because from
    // there on the read is served through the far-reaching lists (k_ovf_*) and must not widen the slices under it
    endv[i] = d.rend > d.rpos ? (d.rend - d.rpos > kReach ? d.rpos + kReach : d.rend) : INT32_MIN;
    if (keep) {
        PLP_ADD64(&acc->n_kept, 1);
        const int64_t wend = cf.end - win_base;   // may overflow int32 only on purpose-built inputs
        if (d.rend > d.rpos && d.rend > 0 && (int64_t)d.rpos < wend) PLP_ADD64(&acc->n_kept_in_window, 1);
        PLP_ADD64(&acc->sum_rlen, span);
        if (!(d.fl & RD_SIMPLE)) PLP_ADD64(&acc->sum_rlen_gen, span);
        unsigned long long it = 3;
        if (!(d.fl & RD_SIMPLE))
            for (int k = 0; k < n; ++k) { int op = cg[k] & 0xf; if (op == OP_I || op == OP_P || op == OP_D) it += 12 + (cg[k] >> 4); }
        PLP_ADD64(&acc->sum_indel_text, it);
        PLP_MAX32(&acc->max_rend, d.rend);
    }
}


// ---- mate overlap ---------------------------------------------------------
struct CWalk { const uint32_t *c, *c0, *cmax; int64_t icig, iseq, iref; };

PLP_HD int cw_set(CWalk &w)
{
    int64_t pos = w.iref;
    if (pos < 0) return -1;
    w.icig = 0; w.iseq = 0; w.iref = 0;
    while (w.c < w.cmax) {
        const int op = *w.c & 0xf; const int n = (int)(*w.c >> 4);
        if (op == OP_S) { w.c++; w.iseq += n; w.icig = 0; continue; }
        if (op == OP_H || op == OP_P) { w.c++; w.icig = 0; continue; }
        if (is_mop(op)) {
            pos -= n;
            if (pos < 0) { w.icig = n + pos; w.iseq += w.icig; w.iref += w.icig; return OP_M; }
            w.c++; w.iseq += n; w.icig = 0; w.iref += n;
            continue;
        }
        if (op == OP_I) { w.c++; w.iseq += n; w.icig = 0; continue; }
        if (op == OP_D || op == OP_N) { pos -= n; if (pos < 0) pos = 0; w.c++; w.iref += n; continue; }
        return -2;
    }
    w.iseq = -1;
    return -1;
}
PLP_HD int cw_next(CWalk &w)
{
    while (w.c < w.cmax) {
        const int op = *w.c & 0xf; const int n = (int)(*w.c >> 4);
        if (is_mop(op)) {
            if (w.icig >= n - 1) { w.icig = -1; w.c++; continue; }
            w.iseq++; w.icig++; w.iref++;
            return OP_M;
        }
        if (op == OP_D || op == OP_N) { w.c++; w.iref += n; w.icig = -1; continue; }
        if (op == OP_I || op == OP_S) { w.c++; w.iseq += n; w.icig = -1; continue; }
        if (op == OP_H || op == OP_P) { w.c++; w.icig = -1; continue; }
        return -2;
    }
    w.iseq = -1; w.iref = -1;
    return -1;
}

// the rule for one reference position where both mates have a base (htslib tweak_overlap_quality): equal bases pool their
// qualities (capped at 200) onto the mate the name hash picks, the other gets 0; different bases: the better one keeps
// 0.8 of its quality, the other gets 0
PLP_HD void tweak_pos(const uint8_t *seq4, uint8_t *aq, uint8_t *bq, uint64_t aoff, uint64_t boff, int32_t ja, int32_t jb, int amul)
{
    const int bmul = 1 - amul;
    const int qa = aq[ja], qb = bq[jb];
    if (base4(seq4, aoff, ja) == base4(seq4, boff, jb)) {
        int q = qa + qb; if (q > 200) q = 200;
        aq[ja] = (uint8_t)(amul * q); bq[jb] = (uint8_t)(bmul * q);
    } else if (qa > qb) { aq[ja] = (uint8_t)(0.8 * qa); bq[jb] = 0; }
    else if (qa < qb) { bq[jb] = (uint8_t)(0.8 * qb); aq[ja] = 0; }
    else { aq[ja] = (uint8_t)(amul * 0.8 * qa); bq[jb] = (uint8_t)(bmul * 0.8 * qb); }
}

// a = mate buffered first, b = mate arriving now
PLP_HD void tweak_overlap(const RawSoA &r, int64_t ia, int64_t ib)
{
    const int64_t apos = r.pos[ia], bpos = r.pos[ib];
    CWalk A, B;
    A.c = A.c0 = r.cigar + r.cigar_off[ia]; A.cmax = A.c + r.n_cigar[ia];
    B.c = B.c0 = r.cigar + r.cigar_off[ib]; B.cmax = B.c + r.n_cigar[ib];
    int64_t iref = bpos;
    A.iref = iref - apos; B.iref = iref - bpos; A.icig = A.iseq = B.icig = B.iseq = 0;
    int ra = cw_set(A);
    if (ra < 0) return;
    int rb = cw_set(B);
    if (rb < 0) return;
    uint8_t *aq = r.qual + r.qual_off[ia], *bq = r.qual + r.qual_off[ib];
    const uint64_t aoff = r.qual_off[ia], boff = r.qual_off[ib];
    const int alq = r.l_qseq[ia], blq = r.l_qseq[ib];
    const int amul = (r.rbits && (r.rbits[ia] & B200_RB_NAME_ODD)) ? 1 : 0, bmul = 1 - amul;
    for (;;) {
        while (ra >= 0 && A.iref >= 0 && A.iref < iref - apos) ra = cw_next(A);
        if (ra < 0) break;
        while (rb >= 0 && B.iref >= 0 && B.iref < iref - bpos) rb = cw_next(B);
        if (rb < 0) break;
        if (iref < A.iref + apos) iref = A.iref + apos;
        if (iref < B.iref + bpos) iref = B.iref + bpos;
        iref++;
        if (A.iref + apos != B.iref + bpos) {
            if (A.iref + apos < B.iref + bpos && B.c > B.c0 && (B.c[-1] & 0xf) == OP_D) {
                do {
                    aq[A.iseq] = amul ? (uint8_t)(aq[A.iseq] * 0.8) : 0;
                    ra = cw_next(A);
                    if (ra < 0) return;
                } while (A.iref + apos < B.iref + bpos);
            } else if (A.c > A.c0 && (A.c[-1] & 0xf) == OP_D) {
                do {
                    bq[B.iseq] = bmul ? (uint8_t)(bq[B.iseq] * 0.8) : 0;
                    rb = cw_next(B);
                    if (rb < 0) return;
                } while (B.iref + bpos < A.iref + apos);
            } else continue;
        }
        if (A.iseq > alq || B.iseq > blq) return;
        tweak_pos(r.seq4, aq, bq, aoff, boff, (int32_t)A.iseq, (int32_t)B.iseq, amul);
    }
}

// Both mates of the shape [H][S]<n>M[S][H] (RD_SIMPLE): over the shared reference span [bpos, min(aend, bend)) every position
// has a base in both reads and the rule above is applied position by position, independently -- position k of the span is
// query base a0 + k of the first mate and b0 + k of the second (what the lock-step CIGAR walk of tweak_overlap visits, in
// the same order).  The device gives a warp to a pair and a lane to every 32nd position.
struct OvSpan { int32_t a0, b0, n; };
PLP_HD OvSpan overlap_span_simple(const RawSoA &r, const ReadDesc &da, const ReadDesc &db, const int32_t *rlen, int64_t ia, int64_t ib)
{
    OvSpan s;
    const int64_t apos = r.pos[ia], bpos = r.pos[ib];
    const int64_t aend = apos + rlen[ia], bend = bpos + rlen[ib];
    const int64_t e = aend < bend ? aend : bend;
    s.a0 = (int32_t)da.qstart + (int32_t)(bpos - apos); s.b0 = (int32_t)db.qstart;
    s.n = (bpos >= apos && e > bpos) ? (int32_t)(e - bpos) : 0;
    return s;
}

// one thread per name chain: replay overlap_push / overlap_remove.  pairs == nullptr: the quality tweak of a pair runs
// right here (emulation harness); else the pair (first mate, second mate) is appended to pairs[] and tweaked by a second
// kernel with one thread per PAIR -- a read takes part in at most one tweak, so the pairs are independent, and a warp
// of tweaks keeps all its lanes busy where a warp of chains has ~15 % of them walking CIGARs.
PLP_HD void overlap_chain(const RawSoA &r, int64_t i, const int64_t *next, const uint8_t *state, const int32_t *rlen,
                          const int64_t *file_start, int n_files, int32_t *pairs = nullptr, unsigned int *n_pairs = nullptr,
                          const ReadDesc *desc = nullptr, int *xcheck_bad = nullptr)
{
    if (r.prev[i] >= 0 || next[i] < 0) return;   // not the head of a chain of >= 2
    int f = 0;
    while (f + 1 < n_files && i >= file_start[f + 1]) ++f;
    const int64_t fs = file_start[f];
    int64_t stored = -1;
    for (int64_t x = i; x >= 0; x = next[x]) {
        const uint8_t st = state[x];
        if (st == ST_MAXDROP) { stored = -1; continue; }   // rejected inside bam_plp_push: overlap_remove(name)
        if (st != ST_KEEP) continue;                        // filtered before the push: invisible
        const uint16_t fl = r.flag[x];
        const int64_t pos = r.pos[x], end = pos + rlen[x];
        if (stored >= 0) {
            // the buffered mate left the buffer (and the hash) once a column >= its end was
            // processed, i.e. once a read starting beyond its end had been pushed
            int64_t j = x - 1;
            while (j >= fs && state[j] != ST_KEEP) --j;
            const int64_t a_end = r.pos[stored] + rlen[stored];
            if (j >= fs && r.pos[j] > a_end) stored = -1;
        }
        if ((fl & 8) || !(fl & 2)) continue;               // mate unmapped / not a proper pair
        const int64_t is = r.isize[x] < 0 ? -r.isize[x] : r.isize[x];
        if ((r.mtid[x] >= 0 && r.tid != r.mtid[x]) || (is >= 2LL * r.l_qseq[x] && r.mpos[x] >= end)) continue;
        if (stored < 0) {
            if (r.mpos[x] >= pos || ((fl & 1) && r.mpos[x] == -1)) stored = x;
        } else {
            if (pairs) {
#if defined(__CUDA_ARCH__)
                const unsigned int k = atomicAdd(n_pairs, 1u);
                pairs[2 * (size_t)k] = (int32_t)stored; pairs[2 * (size_t)k + 1] = (int32_t)x;
#endif
            } else {
#if !defined(__CUDA_ARCH__)
                // emulation harness: the per-position fast path the device uses for two simple mates must rewrite the
                // qualities exactly like the lock-step walk
                if (desc && xcheck_bad && (desc[stored].fl & RD_SIMPLE) && (desc[x].fl & RD_SIMPLE)) {
                    const int la = r.l_qseq[stored], lb = r.l_qseq[x];
                    uint8_t *aq = r.qual + r.qual_off[stored], *bq = r.qual + r.qual_off[x];
                    uint8_t ca[1024], cb[1024];
                    if (la <= 1024 && lb <= 1024) {
                        for (int k = 0; k < la; ++k) ca[k] = aq[k];
                        for (int k = 0; k < lb; ++k) cb[k] = bq[k];
                        const OvSpan sp = overlap_span_simple(r, desc[stored], desc[x], rlen, stored, x);
                        const int amul = (r.rbits && (r.rbits[stored] & B200_RB_NAME_ODD)) ? 1 : 0;
                        // on copies laid out like the originals: tweak_pos addresses bases through the nibble offsets
                        for (int k = 0; k < sp.n; ++k) {
                            uint8_t *pa = ca - 0, *pb = cb - 0;
                            tweak_pos(r.seq4, pa, pb, r.qual_off[stored], r.qual_off[x], sp.a0 + k, sp.b0 + k, amul);
                        }
                        tweak_overlap(r, stored, x);
                        for (int k = 0; k < la; ++k) if (ca[k] != aq[k]) ++*xcheck_bad;
                        for (int k = 0; k < lb; ++k) if (cb[k] != bq[k]) ++*xcheck_bad;
                        stored = -1;
                        continue;
                    }
                }
#endif
                tweak_overlap(r, stored, x);
            }
            stored = -1;
        }
    }
}

// depth -s: second mate is clipped at the first mate's end (bam2depth.c:598-623)
PLP_HD void depth_clip_chain(const RawSoA &r, int64_t i, const int64_t *next, const uint8_t *state, const int32_t *rlen, int32_t *clip, int64_t win_base)
{
    if (r.prev[i] >= 0 || next[i] < 0) return;
    bool have = false; int64_t stored_end = 0;
    for (int64_t x = i; x >= 0; x = next[x]) {
        if (state[x] != ST_KEEP) continue;
        const uint16_t fl = r.flag[x];
        if (!(fl & 1) || (fl & 8)) continue;
        if (!have) {
            const int32_t rl = rlen[x];
            const int64_t endpos = r.pos[x] + (((fl & 4) || r.n_cigar[x] == 0 || rl == 0) ? 1 : rl);
            if (r.mpos[x] == -1 || (r.tid == r.mtid[x] && r.mpos[x] <= endpos)) { have = true; stored_end = endpos; }
        } else {
            clip[x] = (int32_t)(stored_end - win_base);
            have = false;
        }
    }
}

// column-major pileup entries for the iterator tier: the number of file f's reads over column c, and, with Fill, their
// entries in file order at o
template <bool Fill>
PLP_HD uint32_t column_entries(const View &v, int f, int32_t c, b200_pileup1_t *o)
{
    const ReadRange rr = read_range(v, f, c >> 5);
    uint32_t n = 0;
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        const ReadDesc d = v.desc[i];
        if (c < d.rpos || c >= d.rend) continue;
        ++n;
        if (!Fill) continue;
        Ent e; resolve(v, d, c, e);
        if (e.k < 0) {   // simple read: the op index of its match
            const uint32_t *cg = v.cigar + d.cig_off; int k = 0;
            while (!is_mop(cg[k] & 0xf)) ++k;
            e.k = k;
        }
        b200_pileup1_t p;
        p.read = i; p.qpos = e.qpos; p.indel = e.indel; p.cigar_ind = e.k;
        p.is_del = e.is_del; p.is_head = e.is_head; p.is_tail = e.is_tail; p.is_refskip = e.is_refskip;
        *o++ = p;
    }
    return n;
}

}  // namespace plp
