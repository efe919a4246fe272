// plp_core.h -- per-column pileup arithmetic shared by all kernels.
//
// Everything here is a pure function of (staged batch, column): no state is
// carried from column to column, unlike htslib's incremental CIGAR cursor
// (resolve_cigar2) -- that is what lets one GPU thread own one reference
// position.  Functions are __host__ __device__ so the exact same code can be
// single-stepped on the CPU by the debug harness in tests/emul/ (not shipped,
// not linked into the product library).
//
// Reference behaviour restated here (file:line into /root/reference):
//   resolve()            htslib sam.c resolve_cigar2       (SURVEY.md A2)
//   ins_scan()/ins_write htslib sam.c bam_plp_insertion_mod (SURVEY.md A3)
//   mp_entry_*           pileup_seq                bam_plcmd.c:54-169
//   mp_file_size/write   column loop per file      bam_plcmd.c:669-797
//   mp_empty_*           print_empty_pileup        bam_plcmd.c:372-398
//   dp_*                 add_depth / flush rows    bam2depth.c:209-477
//   cv_column            coverage reducers         coverage.c:622-660
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PLP_HD __host__ __device__ __forceinline__
#define PLP_HD_COLD __host__ __device__ __noinline__
#else
#define PLP_HD inline
#define PLP_HD_COLD inline
#endif

namespace plp {

// CIGAR ops, BAM encoding
enum { OP_M = 0, OP_I, OP_D, OP_N, OP_S, OP_H, OP_P, OP_EQ, OP_X };

// 32-byte read descriptor built on the device by the read stage.  The first 16 bytes are all
// a column needs for the common read shape ([S]<n>M[S], RD_SIMPLE); the second half is only
// fetched for reads with indels / clips-with-pads / skips and for a few optional columns.
struct alignas(16) ReadDesc {
    int32_t rpos;      // leftmost column, relative to the window base
    int32_t rend;      // one past the last column the read can appear in (== rpos: never)
    uint32_t qoff;     // offset of qual[0]; nibble offset of the first base
    uint16_t qstart;   // RD_SIMPLE: query index aligned to rpos (qstart + span <= l_qseq is guaranteed)
    uint8_t mapq;
    uint8_t fl;        // RD_* bits
    // ---- second half
    uint32_t cig_off;  // first CIGAR op
    int32_t l_qseq;
    uint32_t n_cigar;
    uint32_t pad_;
};
enum { RD_REV = 1, RD_SIMPLE = 2 };

PLP_HD ReadDesc load_desc(const ReadDesc *p)
{
#if defined(__CUDA_ARCH__)
    union { uint4 w[2]; ReadDesc d; } u;
    u.w[0] = __ldg(reinterpret_cast<const uint4 *>(p));
    u.w[1] = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
    return u.d;
#else
    return *p;
#endif
}
// first half only (second half zero)
PLP_HD ReadDesc load_hot(const ReadDesc *p)
{
#if defined(__CUDA_ARCH__)
    union { uint4 w[2]; ReadDesc d; } u;
    u.w[0] = __ldg(reinterpret_cast<const uint4 *>(p));
    u.w[1] = make_uint4(0, 0, 0, 0);
    return u.d;
#else
    ReadDesc d = *p; d.cig_off = 0; d.l_qseq = 0; d.n_cigar = 0; d.pad_ = 0;
    return d;
#endif
}
PLP_HD void load_cold(ReadDesc &d, const ReadDesc *p)
{
#if defined(__CUDA_ARCH__)
    const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
    d.cig_off = w.x; d.l_qseq = (int32_t)w.y; d.n_cigar = w.z;
#else
    d.cig_off = p->cig_off; d.l_qseq = p->l_qseq; d.n_cigar = p->n_cigar;
#endif
}

// base character of the pileup sequence column: ".ACMGRSVTWYHKDBN" / ",acmgrsvtwyhkdbn"[code]
// from packed immediates (no table load in the inner loop)
PLP_HD char base_char(int code, bool rev)
{
    // bytes little-endian: index 0 is the lowest byte
    const uint64_t fwd_lo = ((uint64_t)'.') | ((uint64_t)'A' << 8) | ((uint64_t)'C' << 16) | ((uint64_t)'M' << 24) | ((uint64_t)'G' << 32) |
                            ((uint64_t)'R' << 40) | ((uint64_t)'S' << 48) | ((uint64_t)'V' << 56);
    const uint64_t fwd_hi = ((uint64_t)'T') | ((uint64_t)'W' << 8) | ((uint64_t)'Y' << 16) | ((uint64_t)'H' << 24) | ((uint64_t)'K' << 32) |
                            ((uint64_t)'D' << 40) | ((uint64_t)'B' << 48) | ((uint64_t)'N' << 56);
    const uint64_t rev_lo = (fwd_lo | 0x2020202020202000ull) & ~0xffull | (uint64_t)',';
    const uint64_t rev_hi = fwd_hi | 0x2020202020202020ull;
    const uint64_t w = (code & 8) ? (rev ? rev_hi : fwd_hi) : (rev ? rev_lo : fwd_lo);
    return (char)(w >> ((code & 7) * 8));
}

struct View {
    const ReadDesc *desc;
    const uint32_t *cigar;
    const int32_t *cig_x;      // per CIGAR op: first column of the op (relative), parallel to cigar[]
    const int32_t *cig_y;      // per CIGAR op: query offset at the start of the op
    const uint8_t *seq4;
    const uint8_t *qual;
    const int32_t *clip;       // depth -s: per-read overlap clip (relative), or nullptr
    const char *ref;           // reference bases or nullptr
    int64_t ref_off;           // relative column of ref[0]
    int64_t ref_n;             // bytes available in ref
    int64_t ref_len_rel;       // contig length in the FASTA, relative to the window base
    int32_t n_files;
    const int64_t *file_start; // [n_files+1]
    const int32_t *tile_lo;    // [n_files][n_tiles] first read to inspect
    const int32_t *tile_hi;    // [n_files][n_tiles] one past the last
    const int32_t *ovf_off;    // [n_files*n_tiles+1] far-reaching reads that start before tile_lo but still cover the group
    const int32_t *ovf_idx;    //   their read indices, ascending
    int32_t n_tiles;
    int32_t tile_cols;
    int64_t win_base;          // absolute coordinate of relative column 0
    int32_t ncols;             // columns [0,ncols) are candidates for output
    int32_t ncols_all;         // -a: columns [0,ncols_all) are emitted even if empty
    const char *name; int32_t name_len;
    const int64_t *bed_beg, *bed_end; int32_t n_bed; int32_t bed_active;
    // per-read strings of the host columns (--output-QNAME, --output-extra fields and tags; bam_plcmd.c:727-855): column k
    // of read i is x_dat[x_off[k * (n_reads + 1) + i] .. x_off[k * (n_reads + 1) + i + 1]); entries of one pileup column
    // are joined with x_sep[k].  n_x == 0: none (then MpConf::n_star_cols only produces "*" place holders)
    int32_t n_x; int64_t x_stride; const uint32_t *x_off; const char *x_dat; char x_sep[16];
};
constexpr int PLP_MAX_X = 16;

// Reads that can cover a 32-column group = far-reaching reads (index < lo, e.g. spliced or
// long-deletion alignments; usually none) followed by the contiguous slice [lo,hi).  Both parts
// are in file order and every index of the first part is below lo, so one pass over the
// concatenation visits the covering reads in file order.
constexpr int32_t kReach = 512;   // a read registers as far-reaching for groups starting >= rpos + kReach
struct ReadRange { int32_t n_ovf, lo, n; const int32_t *ovf; };
PLP_HD ReadRange read_range(const View &v, int f, int g)
{
    const int64_t k = (int64_t)f * v.n_tiles + g;
    ReadRange r;
    const int32_t o0 = v.ovf_off[k];
    r.n_ovf = v.ovf_off[k + 1] - o0;
    r.ovf = v.ovf_idx + o0;
    r.lo = v.tile_lo[k];
    r.n = r.n_ovf + (v.tile_hi[k] - r.lo);
    return r;
}
PLP_HD int32_t range_at(const ReadRange &r, int32_t t) { return t < r.n_ovf ? r.ovf[t] : r.lo + (t - r.n_ovf); }

// The [first,last) slice of a file's reads [fs,fe) that can cover group g.  first is the later of (a) the first read whose
// running max end (pmax, prefix max over the file) exceeds the group start and (b) the first read starting within kReach
// columns of it; reads before (b) that still reach the group are listed separately (ovf_span), so one spliced read cannot
// widen the slice of every group under it.
PLP_HD void group_slice(const ReadDesc *desc, const int32_t *pmax, int64_t fs, int64_t fe, int32_t g, int64_t &first, int64_t &last)
{
    const int32_t c0 = g * 32, c1 = c0 + 31;
    int64_t lo = fs, hi = fe;
    while (lo < hi) { int64_t m = (lo + hi) >> 1; if (pmax[m] > c0) hi = m; else lo = m + 1; }   // first read whose running max end exceeds c0
    first = lo;
    lo = first; hi = fe;
    while (lo < hi) { int64_t m = (lo + hi) >> 1; if (desc[m].rpos > c0 - kReach) hi = m; else lo = m + 1; }  // first read within reach
    if (lo > first) first = lo;
    lo = first; hi = fe;
    while (lo < hi) { int64_t m = (lo + hi) >> 1; if (desc[m].rpos > c1) hi = m; else lo = m + 1; }  // first read starting beyond c1
    last = lo > first ? lo : first;
}

// far-reaching reads: d is listed for the groups [g0,g1], those with 32g >= rpos + kReach and 32g < rend (false: none)
PLP_HD bool ovf_span(const ReadDesc &d, int32_t n_groups, int32_t &g0, int32_t &g1)
{
    if ((int64_t)d.rend - d.rpos <= kReach) return false;
    const int64_t a = (int64_t)d.rpos + kReach;
    g0 = (int32_t)(a <= 0 ? 0 : (a + 31) >> 5);
    g1 = d.rend > 0 ? (d.rend - 1) >> 5 : -1;
    if (g1 >= n_groups) g1 = n_groups - 1;
    return true;
}

struct MpConf {
    int32_t min_baseQ, all, rev_del, no_ins, no_del, no_ends, out_mapq, out_qpos, out_qpos5, n_star_cols;
};
struct DpConf { int32_t min_qual, count_del, all; };

struct Ent {
    int32_t qpos, indel, k;
    uint8_t is_del, is_refskip, is_head, is_tail;
};

PLP_HD int ndigits32(uint32_t v)
{
    return v < 10u ? 1 : v < 100u ? 2 : v < 1000u ? 3 : v < 10000u ? 4 : v < 100000u ? 5 : v < 1000000u ? 6
         : v < 10000000u ? 7 : v < 100000000u ? 8 : v < 1000000000u ? 9 : 10;
}
PLP_HD int ndigits(uint64_t v)
{
    if (v <= 0xffffffffull) return ndigits32((uint32_t)v);
    int n = 1;
    while (v >= 10) { v /= 10; ++n; }
    return n;
}
PLP_HD int put_u64(char *p, uint64_t v)
{
    const int n = ndigits(v);
    if (v <= 0xffffffffull) {
        uint32_t w = (uint32_t)v;
        for (int i = n - 1; i >= 0; --i) { const uint32_t q = w / 10u; p[i] = (char)('0' + (w - q * 10u)); w = q; }
        return n;
    }
    for (int i = n - 1; i >= 0; --i) { p[i] = (char)('0' + v % 10); v /= 10; }
    return n;
}
PLP_HD int base4(const uint8_t *seq4, uint32_t qoff, int32_t i)
{
    const uint32_t n = qoff + (uint32_t)i;
    return (seq4[n >> 1] >> ((~n & 1) << 2)) & 0xf;
}
PLP_HD bool is_refop(int op) { return op == OP_M || op == OP_D || op == OP_N || op == OP_EQ || op == OP_X; }
PLP_HD bool is_mop(int op) { return op == OP_M || op == OP_EQ || op == OP_X; }

// IUPAC character -> 4-bit code (htslib seq_nt16_table), computed not tabled
PLP_HD int nt16_of(unsigned char ch)
{
    switch (ch | 0x20) {  // case-insensitive letters
    case 'a': return 1; case 'c': return 2; case 'm': return 3; case 'g': return 4; case 'r': return 5;
    case 's': return 6; case 'v': return 7; case 't': return 8; case 'w': return 9; case 'y': return 10;
    case 'h': return 11; case 'k': return 12; case 'd': return 13; case 'b': return 14; case 'n': return 15;
    default: break;
    }
    if (ch == '=') return 0;
    if (ch == '0') return 1;
    if (ch == '1') return 2;
    if (ch == '2') return 4;
    if (ch == '3') return 8;
    return 15;
}
PLP_HD int nt16_int_of(int b4)
{
    return b4 == 1 ? 0 : b4 == 2 ? 1 : b4 == 4 ? 2 : b4 == 8 ? 3 : 4;
}
PLP_HD char up(char c) { return (c >= 'a' && c <= 'z') ? (char)(c - 32) : c; }
PLP_HD char lo(char c) { return (c >= 'A' && c <= 'Z') ? (char)(c + 32) : c; }

// reference character at relative column c as the reference prints it
// ("(ref && pos < ref_len) ? ref[pos] : 'N'", bam_plcmd.c:667)
PLP_HD char ref_char(const View &v, int64_t c)
{
    if (!v.ref || c >= v.ref_len_rel) return 'N';
    int64_t i = c - v.ref_off;
    if (i < 0 || i >= v.ref_n) return 'N';
    return v.ref[i];
}

// per-column BED test: bed_overlap(bed, name, pos, pos+1) (bedidx.c:183-191).
// The reference scans its sorted interval list from a linear-index hint; the
// hint never skips an interval that contains pos, so the result is exactly
// "some interval has beg <= pos < end".  The host passes the per-contig
// intervals merged into a disjoint sorted union, which keeps that predicate.
PLP_HD bool bed_pass(const View &v, int64_t c)
{
    if (!v.bed_active) return true;
    const int64_t p = c + v.win_base;
    int lo_ = 0, hi_ = v.n_bed;
    while (lo_ < hi_) { int m = (lo_ + hi_) >> 1; if (v.bed_beg[m] <= p) lo_ = m + 1; else hi_ = m; }
    return lo_ > 0 && v.bed_end[lo_ - 1] > p;
}

// ---- CIGAR -> column (stateless resolve_cigar2) -----------------------------
// Finds the reference-consuming op that holds column c: its index k, first
// column x and query offset y.  Short CIGARs are walked; long ones (long reads,
// thousands of ops) use the per-op prefix arrays built by the read stage, so a
// column costs O(log n_cigar) instead of O(n_cigar).
constexpr int kCigarWalkMax = 8;
PLP_HD void locate(const View &v, const ReadDesc &d, int32_t c, int &k, int32_t &x, int32_t &y, int &op, int &len)
{
    const uint32_t *cg = v.cigar + d.cig_off;
    const int n = (int)d.n_cigar;
    if (n > kCigarWalkMax) {
        const int32_t *cx = v.cig_x + d.cig_off;
        int lo_ = 0, hi_ = n;
        while (lo_ < hi_) { const int m = (lo_ + hi_) >> 1; if (cx[m] <= c) lo_ = m + 1; else hi_ = m; }
        k = lo_ - 1; x = cx[k]; y = v.cig_y[d.cig_off + k];
        op = cg[k] & 0xf; len = (int)(cg[k] >> 4);
        return;
    }
    x = d.rpos; y = 0; op = 0; len = 0;
    for (k = 0; k < n; ++k) {
        op = cg[k] & 0xf; len = (int)(cg[k] >> 4);
        if (is_refop(op)) {
            if (c < x + len) break;
            x += len;
            if (is_mop(op)) y += len;
        } else if (op == OP_I || op == OP_S) y += len;
    }
}

PLP_HD void resolve(const View &v, const ReadDesc &d, int32_t c, Ent &e)
{
    e.is_head = (c == d.rpos);
    e.is_tail = (c == d.rend - 1);
    e.indel = 0; e.is_del = 0; e.is_refskip = 0;
    if (d.fl & RD_SIMPLE) {  // [H][S] M [S][H]
        e.qpos = (int32_t)d.qstart + (c - d.rpos);
        e.k = -1;            // only needed for insertions, which a simple read has none of
        return;
    }
    const uint32_t *cg = v.cigar + d.cig_off;
    const int n = (int)d.n_cigar;
    int32_t x, y; int k, op, len;
    locate(v, d, c, k, x, y, op, len);
    e.k = k;
    if (x + len - 1 == c && k + 1 < n) {  // last column of op k: look ahead
        int op2 = cg[k + 1] & 0xf, l2 = (int)(cg[k + 1] >> 4);
        if (op2 == OP_D && op != OP_D) {
            e.indel = -l2;
            for (int j = k + 2; j < n; ++j) { if ((cg[j] & 0xf) == OP_D) e.indel -= (int)(cg[j] >> 4); else break; }
        } else if (op2 == OP_I) {
            e.indel = l2;
            for (int j = k + 2; j < n; ++j) {
                int o = cg[j] & 0xf;
                if (o == OP_I) e.indel += (int)(cg[j] >> 4);
                else if (o != OP_P) break;
            }
        } else if (op2 == OP_P && k + 2 < n) {
            int l3 = 0;
            for (int j = k + 2; j < n; ++j) {
                int o = cg[j] & 0xf;
                if (o == OP_I) l3 += (int)(cg[j] >> 4);
                else if (o == OP_D || o == OP_M || o == OP_N || o == OP_EQ || o == OP_X) break;
            }
            if (l3 > 0) e.indel = l3;
        }
    }
    if (is_mop(op)) e.qpos = y + (c - x);
    else { e.is_del = 1; e.qpos = y; e.is_refskip = (op == OP_N); }
}

// insertion after op k: number of printed symbols (pads + bases) and the
// length of a deletion that follows directly (bam_plp_insertion_mod)
PLP_HD int ins_scan(const ReadDesc &d, const uint32_t *cg, int k, int &del_len)
{
    int nb = 0;
    del_len = 0;
    for (int j = k + 1; j < (int)d.n_cigar; ++j) {
        int op = cg[j] & 0xf, l = (int)(cg[j] >> 4);
        if (op == OP_P || op == OP_I) nb += l;
        else { if (op == OP_D) del_len = l; break; }
    }
    return nb;
}

// base quality the reference tests against -Q ("qpos < l_qseq ? qual[qpos] : 0")
PLP_HD int ent_qual(const View &v, const ReadDesc &d, const Ent &e)
{
    return e.qpos < d.l_qseq ? (int)v.qual[d.qoff + (uint32_t)e.qpos] : 0;
}

// ---- mpileup text for one (read, column) ------------------------------------
PLP_HD int mp_entry_size(const MpConf &cf, const ReadDesc &d, const uint32_t *cg, const Ent &e)
{
    int sz = 1;
    if (!cf.no_ends && e.is_head) sz += 2;
    int del_len = -e.indel;
    if (e.indel > 0) {
        int len = ins_scan(d, cg, e.k, del_len);
        if (cf.no_ins < 2) sz += 1 + ndigits((uint64_t)len);
        if (!cf.no_ins) sz += len;
    }
    if (del_len > 0) {
        if (cf.no_del < 2) sz += 1 + ndigits((uint64_t)del_len);
        if (!cf.no_del) sz += del_len;
    }
    if (!cf.no_ends && e.is_tail) sz += 1;
    return sz;
}

PLP_HD int mp_entry_write(const View &v, const MpConf &cf, const ReadDesc &d, const uint32_t *cg, const Ent &e,
                          int32_t c, char *p)
{
    char *p0 = p;
    const bool rev = d.fl & RD_REV;
    if (!cf.no_ends && e.is_head) { *p++ = '^'; *p++ = (char)(d.mapq > 93 ? 126 : d.mapq + 33); }
    if (!e.is_del) {
        int ch = e.qpos < d.l_qseq ? base4(v.seq4, d.qoff, e.qpos) : 15;
        if (v.ref) {
            int rb = 15;
            if ((int64_t)c < v.ref_len_rel) {
                int64_t i = (int64_t)c - v.ref_off;
                if (i >= 0 && i < v.ref_n) rb = nt16_of((unsigned char)v.ref[i]);
            }
            if (ch == rb) ch = 0;
        }
        *p++ = base_char(ch, rev);
    } else *p++ = e.is_refskip ? (rev ? '<' : '>') : ((rev && cf.rev_del) ? '#' : '*');
    int del_len = -e.indel;
    if (e.indel > 0) {
        int len = ins_scan(d, cg, e.k, del_len);
        if (cf.no_ins < 2) { *p++ = '+'; p += put_u64(p, (uint64_t)len); }
        if (!cf.no_ins) {
            int j = 1;
            for (int kk = e.k + 1; kk < (int)d.n_cigar; ++kk) {
                int op = cg[kk] & 0xf, l = (int)(cg[kk] >> 4);
                if (op == OP_P) { for (int i = 0; i < l; ++i) *p++ = (rev && cf.rev_del) ? '#' : '*'; }
                else if (op == OP_I) {
                    for (int i = 0; i < l; ++i, ++j) {
                        int q = e.qpos + j - (int)e.is_del;
                        char b = q < d.l_qseq ? "=ACMGRSVTWYHKDBN"[base4(v.seq4, d.qoff, q)] : 'N';
                        *p++ = rev ? lo(b) : up(b);
                    }
                } else break;
            }
        }
    }
    if (del_len > 0) {
        if (cf.no_del < 2) { *p++ = '-'; p += put_u64(p, (uint64_t)del_len); }
        if (!cf.no_del)
            for (int j = 1; j <= del_len; ++j) {
                // "(ref && (int)pos+j < ref_len) ? ref[pos+j] : 'N'" (bam_plcmd.c:158)
                char b = ref_char(v, (int64_t)c + j);
                *p++ = rev ? lo(b) : up(b);
            }
    }
    if (!cf.no_ends && e.is_tail) *p++ = '$';
    return (int)(p - p0);
}

// per (column, file) sizes
struct MpFileSz {
    int32_t nplp, cnt;
    uint32_t seq_len, bp_len, bp5_len;
};

PLP_HD int32_t qpos5_of(const ReadDesc &d, const Ent &e)
{
    return (d.fl & RD_REV) ? d.l_qseq - e.qpos + (int)e.is_del : e.qpos + 1;
}

// quality the reference tests against -Q for read d at column c (simple reads without the cursor)
PLP_HD int col_qual(const View &v, const ReadDesc &d, int32_t i, int32_t c)
{
    if (d.fl & RD_SIMPLE) return (int)v.qual[d.qoff + (uint32_t)d.qstart + (uint32_t)(c - d.rpos)];
    ReadDesc dd = d; load_cold(dd, v.desc + i);
    Ent e; resolve(v, dd, c, e);
    return ent_qual(v, dd, e);
}
// bytes of every host column of file f at column c (contents only: strings of the reads that pass -Q plus separators)
PLP_HD void mp_x_sizes(const View &v, const MpConf &cf, int f, int tile, int32_t c, uint32_t *xl)
{
    for (int k = 0; k < v.n_x; ++k) xl[k] = 0;
    const ReadRange rr = read_range(v, f, tile);
    int n = 0;
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        const ReadDesc d = load_hot(v.desc + i);
        if ((uint32_t)(c - d.rpos) >= (uint32_t)(d.rend - d.rpos)) continue;
        if (col_qual(v, d, i, c) < cf.min_baseQ) continue;
        for (int k = 0; k < v.n_x; ++k) { const uint32_t *o = v.x_off + (int64_t)k * v.x_stride + i; xl[k] += (o[1] - o[0]) + (n ? 1u : 0u); }
        ++n;
    }
}
PLP_HD uint32_t mp_x_section_len(const View &v, const MpConf &cf, int f, int tile, int32_t c, const MpFileSz &s)
{
    if (!v.n_x || s.nplp == 0 || s.cnt == 0) return 0;     // the "\t*" place holders are already in mp_file_section_len
    uint32_t xl[PLP_MAX_X];
    mp_x_sizes(v, cf, f, tile, c, xl);
    uint32_t n = 0;
    for (int k = 0; k < v.n_x; ++k) n += xl[k];
    return n - (uint32_t)v.n_x;                            // instead of the one-byte "*" of each column
}
// the host columns of file f at column c, written at p (which points just behind the last device column)
PLP_HD char *mp_x_write(const View &v, const MpConf &cf, int f, int tile, int32_t c, char *p)
{
    uint32_t xl[PLP_MAX_X];
    mp_x_sizes(v, cf, f, tile, c, xl);
    char *px[PLP_MAX_X];
    for (int k = 0; k < v.n_x; ++k) { *p++ = '\t'; px[k] = p; p += xl[k]; }
    const ReadRange rr = read_range(v, f, tile);
    int n = 0;
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        const ReadDesc d = load_hot(v.desc + i);
        if ((uint32_t)(c - d.rpos) >= (uint32_t)(d.rend - d.rpos)) continue;
        if (col_qual(v, d, i, c) < cf.min_baseQ) continue;
        for (int k = 0; k < v.n_x; ++k) {
            const uint32_t *o = v.x_off + (int64_t)k * v.x_stride + i;
            if (n) *px[k]++ = v.x_sep[k];
            for (uint32_t j = o[0]; j < o[1]; ++j) *px[k]++ = v.x_dat[j];
        }
        ++n;
    }
    return p;
}

PLP_HD void mp_file_size(const View &v, const MpConf &cf, int f, int tile, int32_t c, MpFileSz &s)
{
    s.nplp = 0; s.cnt = 0; s.seq_len = 0; s.bp_len = 0; s.bp5_len = 0;
    const ReadRange rr = read_range(v, f, tile);
    const uint32_t ends = cf.no_ends ? 0u : 1u;
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        ReadDesc d = load_hot(v.desc + i);
        const uint32_t rel = (uint32_t)(c - d.rpos);
        if (rel >= (uint32_t)(d.rend - d.rpos)) continue;
        ++s.nplp;
        if (!(d.fl & RD_SIMPLE) || cf.out_qpos5) load_cold(d, v.desc + i);
        if (d.fl & RD_SIMPLE) {
            // the common case ([S]<n>M[S]): one base, no indel text; 2 extra bytes at the read's
            // first column ("^" + mapq), 1 at its last ("$")
            const int32_t qpos = (int32_t)d.qstart + (int32_t)rel;
            const int q = (int)v.qual[d.qoff + (uint32_t)qpos];
            if (q < cf.min_baseQ) continue;
            ++s.cnt;
            s.seq_len += 1u + (ends & (uint32_t)(rel == 0)) * 2u + (ends & (uint32_t)(c == d.rend - 1));
            if (cf.out_qpos) s.bp_len += (uint32_t)ndigits32((uint32_t)(qpos + 1)) + 1;
            if (cf.out_qpos5) { const int32_t q5 = (d.fl & RD_REV) ? d.l_qseq - qpos : qpos + 1; s.bp5_len += (uint32_t)(q5 < 0 ? 1 + ndigits32((uint32_t)(-q5)) : ndigits32((uint32_t)q5)) + 1; }
            continue;
        }
        const uint32_t *cg = v.cigar + d.cig_off;
        Ent e;
        resolve(v, d, c, e);
        if (ent_qual(v, d, e) < cf.min_baseQ) continue;
        ++s.cnt;
        s.seq_len += (uint32_t)mp_entry_size(cf, d, cg, e);
        if (cf.out_qpos) s.bp_len += (uint32_t)ndigits((uint64_t)(e.qpos + 1)) + 1;
        if (cf.out_qpos5) { int32_t q5 = qpos5_of(d, e); s.bp5_len += (uint32_t)(q5 < 0 ? 1 + ndigits((uint64_t)(-(int64_t)q5)) : ndigits((uint64_t)q5)) + 1; }
    }
}

PLP_HD int mp_n_opt_cols(const MpConf &cf) { return (cf.out_mapq != 0) + (cf.out_qpos != 0) + (cf.out_qpos5 != 0) + cf.n_star_cols; }

// bytes of the per-file section "\tcnt\tseq\tqual[\topt]*"
PLP_HD uint32_t mp_file_section_len(const MpConf &cf, const MpFileSz &s)
{
    uint32_t n = 1 + (uint32_t)ndigits((uint64_t)s.cnt) + 1;
    if (s.nplp == 0) return n + 3 + 2u * (uint32_t)mp_n_opt_cols(cf);
    n += (s.seq_len ? s.seq_len : 1) + 1 + (s.cnt ? (uint32_t)s.cnt : 1);
    if (cf.out_mapq) n += 1 + (s.cnt ? (uint32_t)s.cnt : 1);
    if (cf.out_qpos) n += 1 + (s.cnt ? s.bp_len - 1 : 1);
    if (cf.out_qpos5) n += 1 + (s.cnt ? s.bp5_len - 1 : 1);
    n += 2u * (uint32_t)cf.n_star_cols;   // host-side columns are not produced here
    return n;
}

PLP_HD int put_i32(char *p, int32_t v)
{
    if (v < 0) { *p = '-'; return 1 + put_u64(p + 1, (uint64_t)(-(int64_t)v)); }
    return put_u64(p, (uint64_t)v);
}

// writes the per-file section; s must come from mp_file_size for the same column
PLP_HD char *mp_file_write(const View &v, const MpConf &cf, int f, int tile, int32_t c, const MpFileSz &s, char *p)
{
    *p++ = '\t'; p += put_u64(p, (uint64_t)s.cnt); *p++ = '\t';
    if (s.nplp == 0) {
        *p++ = '*'; *p++ = '\t'; *p++ = '*';
        for (int i = 0; i < mp_n_opt_cols(cf); ++i) { *p++ = '\t'; *p++ = '*'; }
        return p;
    }
    char *ps = p;                                   // sequence column
    char *pq = ps + (s.seq_len ? s.seq_len : 1) + 1; // quality column
    char *pm = pq + (s.cnt ? s.cnt : 1);             // optional columns follow
    char *pb = pm, *pb5;
    if (cf.out_mapq) pb = pm + 1 + (s.cnt ? s.cnt : 1);
    pb5 = pb;
    if (cf.out_qpos) pb5 = pb + 1 + (s.cnt ? s.bp_len - 1 : 1);
    char *pend = pb5;
    if (cf.out_qpos5) pend = pb5 + 1 + (s.cnt ? s.bp5_len - 1 : 1);
    if (!s.cnt) {
        *ps = '*'; *pq = '*';
        if (cf.out_mapq) { pm[0] = '\t'; pm[1] = '*'; }
        if (cf.out_qpos) { pb[0] = '\t'; pb[1] = '*'; }
        if (cf.out_qpos5) { pb5[0] = '\t'; pb5[1] = '*'; }
    } else {
        if (cf.out_mapq) *pm++ = '\t';
        if (cf.out_qpos) *pb++ = '\t';
        if (cf.out_qpos5) *pb5++ = '\t';
        const ReadRange rr = read_range(v, f, tile);
        int n = 0;
        // reference base of this column, once (bam_plcmd.c:74-80)
        int rb = -1;
        if (v.ref) {
            rb = 15;
            if ((int64_t)c < v.ref_len_rel) { const int64_t ri = (int64_t)c - v.ref_off; if (ri >= 0 && ri < v.ref_n) rb = nt16_of((unsigned char)v.ref[ri]); }
        }
        const bool ends = !cf.no_ends, extras = (cf.out_mapq | cf.out_qpos | cf.out_qpos5) != 0;
        const int minq = cf.min_baseQ;
        // Descriptors travel through the loop as four raw words (rpos, rend, qoff, qstart | mapq << 16 | flags << 24):
        // rotating a struct with sub-word fields through the software pipeline costs ~25 byte-permute / move instructions
        // per iteration.  Reads that are not of the simple shape reload their full descriptor in the (rare) generic branch.
        struct Raw { int32_t rpos, rend; uint32_t qoff, pk; };
        auto load_raw = [&](int32_t i) -> Raw {
            Raw r;
#if defined(__CUDA_ARCH__)
            const uint4 w = __ldg(reinterpret_cast<const uint4 *>(v.desc + i));
            r.rpos = (int32_t)w.x; r.rend = (int32_t)w.y; r.qoff = w.z; r.pk = w.w;
#else
            const ReadDesc &d = v.desc[i];
            r.rpos = d.rpos; r.rend = d.rend; r.qoff = d.qoff; r.pk = (uint32_t)d.qstart | (uint32_t)d.mapq << 16 | (uint32_t)d.fl << 24;
#endif
            return r;
        };
        const uint32_t kSimple = (uint32_t)RD_SIMPLE << 24, kRev = (uint32_t)RD_REV << 24;
        // operands of a simple read's entry, fetched one iteration ahead of their use
        struct Pre { int q; uint32_t sb; };
        auto prefetch = [&](const Raw &d) -> Pre {
            Pre o; o.q = 0; o.sb = 0;
            const uint32_t rel = (uint32_t)(c - d.rpos);
            if (rel < (uint32_t)(d.rend - d.rpos) && (d.pk & kSimple)) {
                const uint32_t qi = d.qoff + (d.pk & 0xffffu) + rel;
                o.q = (int)v.qual[qi];
                o.sb = v.seq4[qi >> 1];
            }
            return o;
        };
        auto body = [&](const Raw &r, int32_t i, const Pre &pre) {
            const uint32_t rel = (uint32_t)(c - r.rpos);
            if (rel >= (uint32_t)(r.rend - r.rpos)) return;
            int q, qpos1 = 0; int32_t q5 = 0;
            const int mapq = (int)((r.pk >> 16) & 0xffu);
            if (r.pk & kSimple) {
                q = pre.q;
                if (q < minq) return;
                const bool rev = (r.pk & kRev) != 0;
                const uint32_t par = (r.qoff ^ r.pk ^ rel) & 1u;          // parity of the query index qoff + qstart + rel
                if (ends && rel == 0) { *ps++ = '^'; *ps++ = (char)(mapq > 93 ? 126 : mapq + 33); }
                int ch = (int)((pre.sb >> ((par ^ 1u) << 2)) & 0xfu);
                if (ch == rb) ch = 0;
                *ps++ = base_char(ch, rev);
                if (ends && c == r.rend - 1) *ps++ = '$';
                if (extras) {
                    const int32_t qpos = (int32_t)(r.pk & 0xffffu) + (int32_t)rel;
                    qpos1 = qpos + 1;
                    if (cf.out_qpos5) { ReadDesc d; load_cold(d, v.desc + i); q5 = rev ? d.l_qseq - qpos : qpos + 1; }
                }
            } else {
                const ReadDesc d = load_desc(v.desc + i);
                const uint32_t *cg = v.cigar + d.cig_off;
                Ent e;
                resolve(v, d, c, e);
                q = ent_qual(v, d, e);
                if (q < minq) return;
                ps += mp_entry_write(v, cf, d, cg, e, c, ps);
                qpos1 = e.qpos + 1; q5 = qpos5_of(d, e);
            }
            *pq++ = (char)(q + 33 < 126 ? q + 33 : 126);
            if (extras) {
                if (cf.out_mapq) { int m = mapq + 33; *pm++ = (char)(m > 126 ? 126 : m); }
                if (cf.out_qpos) { if (n) *pb++ = ','; pb += put_i32(pb, qpos1); }
                if (cf.out_qpos5) { if (n) *pb5++ = ','; pb5 += put_i32(pb5, q5); }
                ++n;
            }
        };
        for (int32_t t_ = 0; t_ < rr.n_ovf; ++t_) { const int32_t i = rr.ovf[t_]; const Raw d = load_raw(i); body(d, i, prefetch(d)); }
        const int32_t hi_ = rr.lo + (rr.n - rr.n_ovf);
        if (rr.lo < hi_) {
            // two-deep software pipeline: while entry i is formatted, the quality/base bytes of read i+1 and the
            // descriptor of read i+2 are in flight (the loop is bound by dependent-load latency otherwise)
            Raw d0 = load_raw(rr.lo);
            Raw d1 = rr.lo + 1 < hi_ ? load_raw(rr.lo + 1) : d0;
            Pre p0 = prefetch(d0);
            for (int32_t i = rr.lo; i < hi_; ++i) {
                const Raw d = d0; const Pre pr = p0;
                d0 = d1;
                if (i + 1 < hi_) p0 = prefetch(d0);
                if (i + 2 < hi_) d1 = load_raw(i + 2);
                body(d, i, pr);
            }
        }
    }
    pq = p + (s.seq_len ? s.seq_len : 1);
    *pq = '\t';
    p = pend;
    if (v.n_x && s.cnt) return mp_x_write(v, cf, f, tile, c, p);
    for (int i = 0; i < cf.n_star_cols; ++i) { *p++ = '\t'; *p++ = '*'; }
    return p;
}

PLP_HD uint32_t mp_head_len(const View &v, int32_t c)
{
    return (uint32_t)v.name_len + 1 + (uint32_t)ndigits((uint64_t)(v.win_base + c + 1)) + 2;
}
PLP_HD char *mp_head_write(const View &v, int32_t c, char *p)
{
    for (int i = 0; i < v.name_len; ++i) *p++ = v.name[i];
    *p++ = '\t';
    p += put_u64(p, (uint64_t)(v.win_base + c + 1));
    *p++ = '\t';
    *p++ = ref_char(v, c);
    return p;
}

// full line length for column c (0: the column is not reported)
PLP_HD uint32_t mp_line_size(const View &v, const MpConf &cf, int tile, int32_t c, MpFileSz &s0)
{
    uint32_t body = 0;
    bool any = false;
    for (int f = 0; f < v.n_files; ++f) {
        MpFileSz s;
        mp_file_size(v, cf, f, tile, c, s);
        if (f == 0) s0 = s;
        any |= s.nplp > 0;
        body += mp_file_section_len(cf, s) + mp_x_section_len(v, cf, f, tile, c, s);
    }
    if (!any && !(cf.all && c < v.ncols_all)) return 0;
    if (!bed_pass(v, c)) return 0;
    return mp_head_len(v, c) + body + 1;
}

PLP_HD void mp_line_write(const View &v, const MpConf &cf, int tile, int32_t c, const MpFileSz &s0, char *p)
{
    p = mp_head_write(v, c, p);
    for (int f = 0; f < v.n_files; ++f) {
        MpFileSz s;
        if (f == 0) s = s0; else mp_file_size(v, cf, f, tile, c, s);
        p = mp_file_write(v, cf, f, tile, c, s, p);
    }
    *p = '\n';
}

// ---- entry strings: the default single-file mpileup path (mpileup_ent.cuh) ------------------
// pileup_seq (bam_plcmd.c:54-169) emits, for almost every (read, column), ONE sequence character and ONE
// quality character.  A read-major pass (lanes along the read: wide coalesced loads, no per-column
// searching) therefore pre-formats every read into a string of 16-bit entries, one per reference column
// the read spans, and the column pass only gathers them in file order:
//   0x0000          nothing to print: the base fails -Q (bam_plcmd.c:676-679)
//   0xffff          special: the entry carries indel text; the column pass runs the generic formatter
//   otherwise       bits 0-6 sequence character, bit 7 "^"+mapq goes first (read's first column),
//                   bits 8-14 quality character, bit 15 "$" follows (read's last column)
// Reads of the simple shape ([S]<n>M[S], RD_SIMPLE) keep the entry of query base qi at E[qi] -- the index of
// its quality byte, so no offsets have to be computed or stored; the other reads get a slice of a second
// array, one entry per spanned column, whose start is kept in the descriptor's spare word.
constexpr uint32_t ENT_SPECIAL = 0xffffu;

PLP_HD uint32_t umin32(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return min(a, b);
#else
    return a < b ? a : b;
#endif
}

// reference code of column c as pileup_seq compares it (bam_plcmd.c:74-80); 0x10 without a FASTA
PLP_HD uint32_t ent_ref_code(const View &v, int32_t c)
{
    if (!v.ref) return 0x10u;
    if ((int64_t)c < v.ref_len_rel) { const int64_t ri = (int64_t)c - v.ref_off; if (ri >= 0 && ri < v.ref_n) return (uint32_t)nt16_of((unsigned char)v.ref[ri]); }
    return 15u;
}

// entry of one aligned base: q quality byte, code 4-bit base, rb reference code of the column (0x10: none),
// tab = ".ACMGRSVTWYHKDBN,acmgrsvtwyhkdbn" (forward strand, then reverse), flags = 0x80 (head) | 0x8000 (tail)
PLP_HD uint32_t ent_plain(uint32_t q, uint32_t code, uint32_t rb, uint32_t rev, int minq, uint32_t flags, const uint8_t *tab)
{
    if ((int)q < minq) return 0;
    if (code == rb) code = 0;
    return (uint32_t)tab[rev * 16u + code] | umin32(q + 33u, 126u) << 8 | flags;
}

// ---- eight entries at once, SIMD within 32-bit words (the read-major entry pass of mpileup_ent.cuh).
// byte permute: result byte i = byte (sel nibble i) of the 8 bytes {b:7..4, a:3..0}  (PRMT on the device)
PLP_HD uint32_t bperm(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t w = (uint64_t)b << 32 | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((w >> (8 * ((sel >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
    return r;
#endif
}
// the 16 sequence characters of one strand as four words of a register table: t[k] holds codes 4k .. 4k+3
struct EntTab { uint32_t t0, t1, t2, t3; };
PLP_HD EntTab ent_tab(uint32_t rev)
{
    EntTab t;   // ".ACM" "GRSV" "TWYH" "KDBN" little-endian; the reverse strand is the lower-case row with ','
    t.t0 = 0x4d43412eu; t.t1 = 0x56535247u; t.t2 = 0x48595754u; t.t3 = 0x4e42444bu;
    if (rev) { t.t0 = 0x6d63612cu; t.t1 |= 0x20202020u; t.t2 |= 0x20202020u; t.t3 |= 0x20202020u; }
    return t;
}
// quality characters of four quality bytes: min(q + 33, 126) per byte
PLP_HD uint32_t ent_qchar4(uint32_t q)
{
    const uint32_t t = (q & 0x7f7f7f7fu) + 0x21212121u;                       // q7 + 33 <= 160: no carry between bytes
    const uint32_t m = ((((t + 0x01010101u) | q) & 0x80808080u) >> 7) * 0xffu;  // bytes with q7 + 33 >= 127 or q >= 128
    return (t & ~m) | (0x7e7e7e7eu & m);
}
// 0xff in every byte whose quality is below minq (0 <= minq <= 127; bytes >= 128 never fail)
PLP_HD uint32_t ent_fail4(uint32_t q, uint32_t minq4)
{
    const uint32_t ge = ((((q & 0x7f7f7f7fu) | 0x80808080u) - minq4) | q) & 0x80808080u;   // bit 7: q >= minq
    return ((ge ^ 0x80808080u) >> 7) * 0xffu;
}
// sequence characters of the four codes in nibbles 0..3 of h (natural order), through the register table
PLP_HD uint32_t ent_schar4(uint32_t h, const EntTab &t)
{
    const uint32_t sel = h & 0x7777u;
    const uint32_t lo = bperm(t.t0, t.t1, sel), hi = bperm(t.t2, t.t3, sel);
    return bperm(lo, hi, ((h & 0x8888u) >> 1) | 0x3210u);
}
// Eight consecutive bases: qx/qy their quality bytes, s4 their four sequence bytes (even base in the high nibble, BAM order),
// r8 the reference codes of their columns as eight nibbles in natural order (has_ref; a base equal to it prints '.' / ','),
// minq4 = minq in every byte (0..127).  Entries leave as four words (entry k in half k&1 of word k>>1), WITHOUT the
// "^" / "$" flags; returns bit k set when base k fails -Q.
PLP_HD uint32_t ent_group8_swar(uint32_t qx, uint32_t qy, uint32_t s4, bool has_ref, uint32_t r8, const EntTab &t, uint32_t minq4, uint32_t (&w)[4])
{
    uint32_t n = ((s4 & 0x0f0f0f0fu) << 4) | ((s4 >> 4) & 0x0f0f0f0fu);         // nibble k = code of base k
    if (has_ref) {
        const uint32_t z = n ^ r8;
        const uint32_t ne = (((z & 0x77777777u) + 0x77777777u) | z) & 0x88888888u;   // bit 3 of a nibble: codes differ
        n &= ~(((ne ^ 0x88888888u) >> 3) * 0xfu);
    }
    const uint32_t fx = ent_fail4(qx, minq4), fy = ent_fail4(qy, minq4);
    const uint32_t cx = ent_schar4(n, t) & ~fx, cy = ent_schar4(n >> 16, t) & ~fy;
    const uint32_t ax = ent_qchar4(qx) & ~fx, ay = ent_qchar4(qy) & ~fy;
    w[0] = bperm(cx, ax, 0x5140u); w[1] = bperm(cx, ax, 0x7362u);
    w[2] = bperm(cy, ay, 0x5140u); w[3] = bperm(cy, ay, 0x7362u);
    // one bit per failing base: bits 0,8,16,24 of (f >> 7) gathered by a multiply (partial products never collide)
    return ((((fx & 0x01010101u) * 0x00204081u) >> 21) & 0xfu) | ((((fy & 0x01010101u) * 0x00204081u) >> 17) & 0xf0u);
}

// entry of read d (any shape) at column c through the generic cursor; extra = bytes the entry prints beyond its
// one sequence character ("^"+mapq, "$", indel text): what the size pass adds to the column
PLP_HD uint32_t ent_generic(const View &v, const MpConf &cf, const ReadDesc &d, int32_t c, uint32_t rb, const uint8_t *tab, uint32_t &extra)
{
    Ent e;
    resolve(v, d, c, e);
    extra = 0;
    const int q = ent_qual(v, d, e);
    if (q < cf.min_baseQ) return 0;
    extra = (uint32_t)mp_entry_size(cf, d, v.cigar + d.cig_off, e) - 1u;
    if (e.indel != 0) return ENT_SPECIAL;
    const uint32_t rev = (d.fl & RD_REV) ? 1u : 0u;
    uint32_t ch;
    if (!e.is_del) {
        uint32_t code = e.qpos < d.l_qseq ? (uint32_t)base4(v.seq4, d.qoff, e.qpos) : 15u;
        if (code == rb) code = 0;
        ch = tab[rev * 16u + code];
    } else ch = (uint32_t)(e.is_refskip ? (rev ? '<' : '>') : ((rev && cf.rev_del) ? '#' : '*'));
    uint32_t x = ch | umin32((uint32_t)q + 33u, 126u) << 8;
    if (!cf.no_ends) x |= (e.is_head ? 0x80u : 0u) | (e.is_tail ? 0x8000u : 0u);
    return x;
}

// Everything of a single-file line except the entries: header, count, separators, "*" place
// holders, newline.  Returns the cursors the entries are appended through (ps == nullptr: none).
struct EntCur { char *ps, *pq, *pm; };
PLP_HD EntCur ent_layout(const View &v, const MpConf &cf, int32_t c, const MpFileSz &s, char *p)
{
    EntCur k; k.ps = nullptr; k.pq = nullptr; k.pm = nullptr;
    p = mp_head_write(v, c, p);
    *p++ = '\t'; p += put_u64(p, (uint64_t)s.cnt); *p++ = '\t';
    if (s.nplp == 0) {
        *p++ = '*'; *p++ = '\t'; *p++ = '*';
        for (int i = 0; i < mp_n_opt_cols(cf); ++i) { *p++ = '\t'; *p++ = '*'; }
    } else {
        char *ps = p, *pq = ps + (s.seq_len ? s.seq_len : 1) + 1, *pm = pq + (s.cnt ? s.cnt : 1);
        char *pend = cf.out_mapq ? pm + 1 + (s.cnt ? s.cnt : 1) : pm;
        pq[-1] = '\t';
        if (!s.cnt) { *ps = '*'; *pq = '*'; if (cf.out_mapq) { pm[0] = '\t'; pm[1] = '*'; } }
        else { if (cf.out_mapq) *pm++ = '\t'; k.ps = ps; k.pq = pq; k.pm = pm; }
        p = pend;
        for (int i = 0; i < cf.n_star_cols; ++i) { *p++ = '\t'; *p++ = '*'; }
    }
    *p = '\n';
    return k;
}

// special entry (indel text) of read i at column c through the generic formatter: ONE out-of-line copy, so that the
// gather loop stays a few dozen instructions.  Appends the sequence text at ps, returns its length; q = quality.
PLP_HD_COLD int ent_special(const View &v, const MpConf &cf, int32_t i, int32_t c, char *ps, int &q)
{
    const ReadDesc d = load_desc(v.desc + i);
    Ent en;
    resolve(v, d, c, en);
    q = ent_qual(v, d, en);
    return mp_entry_write(v, cf, d, v.cigar + d.cig_off, en, c, ps);
}

// The column pass: line of column c from the entry strings (single file; -s supported, -O / --output-BP-5 not).
// E: entries of simple reads at their quality-byte index; E2: the slices of the other reads (start in desc.pad_).
// Cursors are byte offsets from p (one base register: shared-memory stores on the device).
PLP_HD void mp_line_write_ent(const View &v, const MpConf &cf, int32_t c, const MpFileSz &s, char *p, const uint16_t *E, const uint16_t *E2)
{
    const EntCur cur = ent_layout(v, cf, c, s, p);
    if (!cur.ps) return;
    uint32_t so = (uint32_t)(cur.ps - p), qo = (uint32_t)(cur.pq - p), mo = (uint32_t)(cur.pm - p);
    const ReadRange rr = read_range(v, 0, c >> 5);
    const uint32_t kSimple = (uint32_t)RD_SIMPLE << 24;
    const bool out_mapq = cf.out_mapq != 0;
    struct Raw { int32_t rpos, rend; uint32_t qoff, pk; };
    auto load_raw = [&](int32_t i) -> Raw {
        Raw r;
#if defined(__CUDA_ARCH__)
        const uint4 w = __ldg(reinterpret_cast<const uint4 *>(v.desc + i));
        r.rpos = (int32_t)w.x; r.rend = (int32_t)w.y; r.qoff = w.z; r.pk = w.w;
#else
        const ReadDesc &d = v.desc[i];
        r.rpos = d.rpos; r.rend = d.rend; r.qoff = d.qoff; r.pk = (uint32_t)d.qstart | (uint32_t)d.mapq << 16 | (uint32_t)d.fl << 24;
#endif
        return r;
    };
    auto emit = [&](const Raw &r, int32_t i, uint32_t e) {
        if (!e) return;
        const uint32_t mapq = (r.pk >> 16) & 0xffu;
        if (e == ENT_SPECIAL) {
            int q;
            so += (uint32_t)ent_special(v, cf, i, c, p + so, q);
            p[qo++] = (char)(q + 33 < 126 ? q + 33 : 126);
        } else {
            if (e & 0x8080u) {
                if (e & 0x80u) { p[so++] = '^'; p[so++] = (char)(mapq > 93u ? 126u : mapq + 33u); }
                p[so++] = (char)(e & 0x7fu);
                if (e & 0x8000u) p[so++] = '$';
            } else p[so++] = (char)e;
            p[qo++] = (char)((e >> 8) & 0x7fu);
        }
        if (out_mapq) p[mo++] = (char)umin32(mapq + 33u, 126u);
    };
    // entry of read i (descriptor r) at this column through the general route (any shape)
    auto entry_of = [&](const Raw &r, int32_t i) -> uint32_t {
        const uint32_t rel = (uint32_t)(c - r.rpos);
        if (rel >= (uint32_t)(r.rend - r.rpos)) return 0;
        if (r.pk & kSimple) return E[r.qoff + (r.pk & 0xffffu) + rel];
        return E2[v.desc[i].pad_ + rel];
    };
    // far-reaching reads first (usually none): all of them precede the slice in file order
    for (int32_t t = 0; t < rr.n_ovf; ++t) { const int32_t i = rr.ovf[t]; const Raw r = load_raw(i); emit(r, i, entry_of(r, i)); }
    // the slice, four reads per step: four descriptor loads, then four entry loads in flight (branch-free for simple
    // reads: a read that is not over the column loads entry 0 of the array and discards it), then the appends
    const int32_t hi = rr.lo + (rr.n - rr.n_ovf);
    int32_t i = rr.lo;
    for (; i + 4 <= hi; i += 4) {
        Raw r[4]; uint32_t rel[4], e[4]; bool in[4];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = 0; k < 4; ++k) r[k] = load_raw(i + k);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = 0; k < 4; ++k) {
            rel[k] = (uint32_t)(c - r[k].rpos);
            in[k] = rel[k] < (uint32_t)(r[k].rend - r[k].rpos);
            const bool fast = in[k] && (r[k].pk & kSimple);
            const uint32_t idx = fast ? r[k].qoff + (r[k].pk & 0xffffu) + rel[k] : 0u;
            e[k] = E[idx];
            if (!fast) e[k] = 0;
        }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = 0; k < 4; ++k) {
            if (in[k] && !(r[k].pk & kSimple)) e[k] = E2[v.desc[i + k].pad_ + rel[k]];
            emit(r[k], i + k, e[k]);
        }
    }
    for (; i < hi; ++i) { const Raw r = load_raw(i); emit(r, i, entry_of(r, i)); }
}

// ---- depth (bam2depth.c) ------------------------------------------------------
// In depth mode ReadDesc.rend is bam_endpos (zero-length reads span one column).
struct DpCol { int32_t depth; bool spanned; };

PLP_HD void dp_file_column(const View &v, const DpConf &cf, int f, int tile, int32_t c, DpCol &o)
{
    o.depth = 0; o.spanned = false;
    const ReadRange rr = read_range(v, f, tile);
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        ReadDesc d = load_hot(v.desc + i);
        if ((uint32_t)(c - d.rpos) >= (uint32_t)(d.rend - d.rpos)) continue;
        o.spanned = true;
        if (!(d.fl & RD_SIMPLE)) load_cold(d, v.desc + i);
        const int32_t clip = v.clip ? v.clip[i] : INT32_MIN;
        if (d.fl & RD_SIMPLE) {
            if (c < clip) continue;
            int q = (int)d.qstart + (c - d.rpos);
            if (!cf.min_qual || v.qual[d.qoff + (uint32_t)q] >= cf.min_qual) ++o.depth;
            continue;
        }
        int32_t x, y; int k, op, len;
        locate(v, d, c, k, x, y, op, len);
        if (k >= (int)d.n_cigar || c < clip) continue;
        if (is_mop(op)) {
            int q = y + (c - x);
            if (!cf.min_qual || v.qual[d.qoff + (uint32_t)q] >= cf.min_qual) ++o.depth;
        } else if (op == OP_D && cf.count_del) {
            // -J: a deletion column borrows the quality of the next query base (bam2depth.c:418-423)
            if (y < d.l_qseq) { if (v.qual[d.qoff + (uint32_t)y] >= cf.min_qual) ++o.depth; }
            else ++o.depth;
        }
    }
}

// ---- coverage (coverage.c:622-660) --------------------------------------------
struct CvCol { uint32_t depth; uint32_t qbases; uint64_t sum_bq; uint32_t missing; bool count_base; };

PLP_HD void cv_column(const View &v, int32_t min_baseQ, int tile, int32_t c, CvCol &o)
{
    o.depth = 0; o.qbases = 0; o.sum_bq = 0; o.missing = 0; o.count_base = false;
    for (int f = 0; f < v.n_files; ++f) {
        const ReadRange rr = read_range(v, f, tile);
        int32_t dpos = 0;
        for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
            ReadDesc d = load_hot(v.desc + i);
            if ((uint32_t)(c - d.rpos) >= (uint32_t)(d.rend - d.rpos)) continue;
            ++dpos;
            if (d.fl & RD_SIMPLE) {
                const int q = v.qual[d.qoff + (uint32_t)d.qstart + (uint32_t)(c - d.rpos)];
                if (q < min_baseQ) --dpos;
                else { o.sum_bq += (uint64_t)q; ++o.qbases; }
                continue;
            }
            load_cold(d, v.desc + i);
            Ent e;
            resolve(v, d, c, e);
            if (e.is_del || e.is_refskip) --dpos;
            else if (e.qpos < d.l_qseq) {
                int q = v.qual[d.qoff + (uint32_t)e.qpos];
                if (q < min_baseQ) --dpos;
                else { o.sum_bq += (uint64_t)q; ++o.qbases; }
            } else ++o.missing;
        }
        if (dpos > 0) { o.count_base = true; o.depth += (uint32_t)dpos; }
    }
}

// what a column adds to its bin of the histogram views (coverage.c:609-660): its depth, or 1 if covered (breadth)
PLP_HD uint32_t cv_hist_add(const CvCol &o, int32_t min_depth, int plot_depth)
{
    return plot_depth ? o.depth : ((o.count_base && o.depth >= (uint32_t)min_depth) ? 1u : 0u);
}

// bedcov (bedcov.c:316-331): a column takes part when the multi-file iterator would return it (any file has a read over it)
PLP_HD bool bc_any(const View &v, int32_t c)
{
    bool any = false;
    for (int f = 0; f < v.n_files && !any; ++f) {
        const ReadRange rr = read_range(v, f, c >> 5);
        for (int32_t t_ = 0; t_ < rr.n && !any; ++t_) { const ReadDesc d = load_hot(v.desc + range_at(rr, t_)); any = (uint32_t)(c - d.rpos) < (uint32_t)(d.rend - d.rpos); }
    }
    return any;
}
// depth of file f at column c, without deletions / reference skips when skip_dn (simple reads have neither)
PLP_HD int32_t bc_depth(const View &v, int f, int32_t c, int skip_dn)
{
    const ReadRange rr = read_range(v, f, c >> 5);
    int32_t np = 0, m = 0;
    for (int32_t t_ = 0; t_ < rr.n; ++t_) {
        const int32_t i = range_at(rr, t_);
        ReadDesc d = load_hot(v.desc + i);
        if ((uint32_t)(c - d.rpos) >= (uint32_t)(d.rend - d.rpos)) continue;
        ++np;
        if (skip_dn && !(d.fl & RD_SIMPLE)) { load_cold(d, v.desc + i); Ent e; resolve(v, d, c, e); if (e.is_del || e.is_refskip) ++m; }
    }
    return np - m;
}

// depth rows "name\tpos(\tdepth)*\n" (bam2depth.c:234-244); size() keeps the first file's depth for write()
struct DpFmt {
    View v; DpConf cf;
    struct State { int32_t d0; };
    PLP_HD uint32_t size(int32_t c, State &s) const
    {
        bool any = false; uint32_t body = 0;
        for (int f = 0; f < v.n_files; ++f) {
            DpCol o; dp_file_column(v, cf, f, c >> 5, c, o);
            if (f == 0) s.d0 = o.depth;
            any |= o.spanned;
            body += 1 + (uint32_t)ndigits((uint64_t)o.depth);
        }
        if (!any && !(cf.all && c < v.ncols_all)) return 0;
        if (!bed_pass(v, c)) return 0;
        return (uint32_t)v.name_len + 1 + (uint32_t)ndigits((uint64_t)(v.win_base + c + 1)) + body + 1;
    }
    PLP_HD void write(int32_t c, const State &s, char *p) const
    {
        for (int i = 0; i < v.name_len; ++i) *p++ = v.name[i];
        *p++ = '\t';
        p += put_u64(p, (uint64_t)(v.win_base + c + 1));
        for (int f = 0; f < v.n_files; ++f) {
            int32_t d = s.d0;
            if (f) { DpCol o; dp_file_column(v, cf, f, c >> 5, c, o); d = o.depth; }
            *p++ = '\t';
            p += put_u64(p, (uint64_t)d);
        }
        *p = '\n';
    }
};

}  // namespace plp
