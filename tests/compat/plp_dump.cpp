// plp_dump.cpp -- test client of the htslib-compatible iterator tier (include/b200_htslib_compat.h).
// Written the way an htslib user writes a pileup loop (cf. coverage.c:572-589): a pull callback
// fills bam1_t records, bam_mplp64_auto() hands out columns.  Prints every bam_pileup1_t field so the
// test can diff it against the CPU oracle's iterator (`plp_oracle pileup-dump`).
#include "fill_bam1.hpp"
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>

// -c: exercise the client-data hooks: the constructor numbers the reads, every entry must carry its read's number,
// and every constructed read must be destructed exactly once
static long n_ctor = 0, n_dtor = 0, cd_bad = 0;
static int ctor(void *, const bam1_t *, bam_pileup_cd *cd) { cd->i = ++n_ctor; return 0; }
static std::map<const bam1_t *, int64_t> seen;     // client data last seen with a live read (the iterator may recycle a freed read's address)
static int dtor(void *, const bam1_t *b, bam_pileup_cd *cd) { if (cd->i < 1 || cd->i > n_ctor) ++cd_bad; cd->i = -1; ++n_dtor; seen.erase(b); return 0; }

static void print_entry(const bam_pileup1_t *p, const char *ins, int il, int dl)
{
    int q = p->qpos < p->b->core.l_qseq ? bam_get_qual(p->b)[p->qpos] : -1;
    printf(" %s/%d/%d/%d%d%d%d/%d/%d/%s/%d", bam_get_qname(p->b), p->qpos, p->indel, p->is_del, p->is_head, p->is_tail, p->is_refskip,
           p->cigar_ind, q, il > 0 ? ins : "-", dl);
}

static void print_column(int tid, hts_pos_t pos, int n_plp, const bam_pileup1_t *plp)
{
    char ins[4096];
    printf("%d\t%lld\t%d:", tid, (long long)pos, n_plp);
    for (int j = 0; j < n_plp; ++j) {
        int dl = 0, il = b200_plp_insertion(plp + j, ins, sizeof ins, &dl);
        print_entry(plp + j, ins, il, dl);
    }
    putchar('\n');
}

// -p: one file through the push interface, the way a callback-style buffer over the iterator (samtools' bam_plbuf layer)
// drives it: every record goes in with bam_plp_push and the columns it completes are drained with bam_plp64_next right
// away; a NULL push marks the end of input and the last drain flushes what is left
static int push_dump(const char *fn)
{
    Src src; src.rd = b200::AlnReader::open(fn);
    if (!src.rd) return 1;
    bam_plp_t it = bam_plp_init(nullptr, nullptr);
    if (!it) { fprintf(stderr, "plp_dump: no pileup engine\n"); return 1; }
    bam1_t *b = bam_init1();
    int ret, tid, n_plp; hts_pos_t pos; const bam_pileup1_t *plp;
    bool eof = false;
    while (!eof) {
        ret = pull(&src, b);
        if (ret < -1) break;
        eof = ret == -1;
        if (bam_plp_push(it, eof ? nullptr : b) < 0) { ret = -2; break; }
        while ((plp = bam_plp64_next(it, &tid, &pos, &n_plp)) != nullptr) print_column(tid, pos, n_plp, plp);
        if (n_plp < 0) { ret = -2; break; }
    }
    bam_destroy1(b);
    bam_plp_destroy(it);
    return ret < -1 ? 1 : 0;
}

int main(int argc, char **argv)
{
    bool overlaps = false, hooks = false, push = false; int maxcnt = 8000; int a = 1;
    for (; a < argc && argv[a][0] == '-'; ++a) {
        if (!strcmp(argv[a], "-o")) overlaps = true;
        else if (!strcmp(argv[a], "-c")) hooks = true;
        else if (!strcmp(argv[a], "-p")) push = true;
        else if (!strcmp(argv[a], "-d") && a + 1 < argc) maxcnt = atoi(argv[++a]);
    }
    const int n = argc - a;
    if (n < 1 || (push && n != 1)) { fprintf(stderr, "usage: plp_dump [-o] [-c] [-d maxcnt] in.sam [in2.sam ...] | plp_dump -p in.sam\n"); return 1; }
    if (push) return push_dump(argv[a]);
    std::vector<Src> src((size_t)n); std::vector<void *> data;
    for (int i = 0; i < n; ++i) { src[(size_t)i].rd = b200::AlnReader::open(argv[a + i]); if (!src[(size_t)i].rd) return 1; data.push_back(&src[(size_t)i]); }
    bam_mplp_t it = bam_mplp_init(n, pull, data.data());
    if (!it) { fprintf(stderr, "plp_dump: no CUDA pileup engine\n"); return 1; }
    if (overlaps) bam_mplp_init_overlaps(it);
    if (hooks) { bam_mplp_constructor(it, ctor); bam_mplp_destructor(it, dtor); }
    kstring_t ks = {0, 0, nullptr};
    bam_mplp_set_maxcnt(it, maxcnt);
    std::vector<int> n_plp((size_t)n); std::vector<const bam_pileup1_t *> plp((size_t)n);
    int tid, ret; hts_pos_t pos; char ins[4096];
    while ((ret = bam_mplp64_auto(it, &tid, &pos, n_plp.data(), plp.data())) > 0) {
        printf("%d\t%lld", tid, (long long)pos);
        for (int i = 0; i < n; ++i) {
            printf("\t%d:", n_plp[(size_t)i]);
            for (int j = 0; j < n_plp[(size_t)i]; ++j) {
                const bam_pileup1_t *p = plp[(size_t)i] + j;
                int il, dl = 0;
                if (hooks) {   // htslib's own insertion signature + the client data of the read
                    il = bam_plp_insertion(p, &ks, &dl);
                    snprintf(ins, sizeof ins, "%s", il > 0 ? ks.s : "");
                    auto f = seen.find(p->b);
                    if (p->cd.i < 1 || p->cd.i > n_ctor || (f != seen.end() && f->second != p->cd.i)) ++cd_bad;
                    seen[p->b] = p->cd.i;
                } else il = b200_plp_insertion(p, ins, sizeof ins, &dl);
                print_entry(p, ins, il, dl);
            }
        }
        putchar('\n');
    }
    bam_mplp_destroy(it);
    free(ks.s);
    if (hooks) {
        fprintf(stderr, "hooks: ctor=%ld dtor=%ld bad=%ld\n", n_ctor, n_dtor, cd_bad);
        if (n_ctor != n_dtor || cd_bad || n_ctor == 0) return 2;
    }
    return ret < 0 ? 1 : 0;
}
