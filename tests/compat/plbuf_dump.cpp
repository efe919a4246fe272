// plbuf_dump.cpp -- client of samtools' own bam_plbuf layer (bam_plbuf.h:32-51), which is compiled UNMODIFIED from a
// samtools source tree against tests/compat/shim/htslib/sam.h -> include/b200_htslib_compat.h by
// tests/golden/make_plbuf_golden.py.  Shows that the layer riding on the iterator API keeps working (SURVEY.md section 8b).
// Same dump format as plp_dump.
#include "fill_bam1.hpp"
#include <cstdio>
extern "C" {
#include "bam_plbuf.h"
}

static int on_column(uint32_t tid, hts_pos_t pos, int n, const bam_pileup1_t *pl, void *)
{
    char ins[4096];
    printf("%u\t%lld\t%d:", tid, (long long)pos, n);
    for (int j = 0; j < n; ++j) {
        const bam_pileup1_t *p = pl + j;
        int q = p->qpos < p->b->core.l_qseq ? bam_get_qual(p->b)[p->qpos] : -1, dl = 0;
        int il = b200_plp_insertion(p, ins, sizeof ins, &dl);
        printf(" %s/%d/%d/%d%d%d%d/%d/%d/%s/%d", bam_get_qname(p->b), p->qpos, p->indel, p->is_del, p->is_head, p->is_tail, p->is_refskip,
               p->cigar_ind, q, il > 0 ? ins : "-", dl);
    }
    putchar('\n');
    return 0;
}

int main(int argc, char **argv)
{
    if (argc != 2) { fprintf(stderr, "usage: plbuf_dump in.sam\n"); return 1; }
    Src src; src.rd = b200::AlnReader::open(argv[1]);
    if (!src.rd) return 1;
    bam_plbuf_t *buf = bam_plbuf_init(on_column, nullptr);
    if (!buf || !buf->iter) { fprintf(stderr, "plbuf_dump: no pileup engine\n"); return 1; }
    bam1_t *b = bam_init1();
    int ret;
    while ((ret = pull(&src, b)) >= 0) if (bam_plbuf_push(b, buf) < 0) return 1;
    if (ret < -1) return 1;
    bam_plbuf_push(nullptr, buf);            // flush (bam_plbuf.c:59-71)
    bam_plbuf_destroy(buf);
    bam_destroy1(b);
    return 0;
}
