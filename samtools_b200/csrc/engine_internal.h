// engine_internal.h -- the engine handle: grow-only HBM buffers + batch state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/b200_pileup.h"
#include "plp_core.h"

#define DBUF(type, name) type *name = nullptr; size_t cap_##name = 0

struct b200_engine {
    int device = 0, n_sm = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evA = nullptr, evB = nullptr, evB0 = nullptr, evB1 = nullptr;
    bool baq_ran = false; double last_baq_ms = 0;
    double last_parts_ms[3] = {0, 0, 0};
    char err[512];
    int64_t launches = 0;
    double last_kernel_ms = 0, last_stage_ms = 0, last_stage_device_ms = 0;
    bool keep_raw = false, uploaded = false, has_host_clip = false;
    size_t qual_bytes = 0, n_cigar_total = 0;
    uint32_t smem_text = 24 * 1024;
    void *d_gfmt = nullptr;      // device copy of the gather's parameter block (cold paths)
    bool baq_attr_set = false;   // k_baq_reg's dynamic shared-memory attribute has been raised on this handle's device
    int use_tma = 1, general = 0;

    // raw SoA image of the staged records
    DBUF(int64_t, pos); DBUF(uint16_t, flag); DBUF(uint8_t, mapq); DBUF(int32_t, l_qseq); DBUF(uint32_t, n_cigar);
    DBUF(uint64_t, cigar_off); DBUF(uint64_t, qual_off); DBUF(int32_t, mtid); DBUF(int64_t, mpos); DBUF(int64_t, isize);
    DBUF(int64_t, prev); DBUF(uint8_t, rbits);
    DBUF(uint32_t, cigar); DBUF(uint8_t, seq4); DBUF(uint8_t, qual); DBUF(char, ref); DBUF(char, dname);
    DBUF(int64_t, file_start);
    DBUF(uint8_t, qual0); DBUF(uint8_t, mapq0);   // pristine copies for b200_restage (b200_set_keep_raw)
    // derived
    DBUF(uint8_t, state); DBUF(int32_t, rlen); DBUF(plp::ReadDesc, desc); DBUF(int32_t, endv); DBUF(int32_t, pmax);
    DBUF(int32_t, glo); DBUF(int32_t, ghi); DBUF(uint64_t, status); DBUF(char, out);
    DBUF(int64_t, bed_beg); DBUF(int64_t, bed_end);
    DBUF(uint32_t, col_n); DBUF(uint64_t, col_off); DBUF(uint64_t, col_state); DBUF(uint32_t, tile_total);
    DBUF(uint32_t, ovf_cnt); DBUF(int32_t, ovf_off); DBUF(int32_t, ovf_idx);
    DBUF(int32_t, ss_diff); DBUF(int32_t, ss_nplp); DBUF(uint32_t, ss_fail); DBUF(uint32_t, ss_extra); DBUF(uint64_t, status2); DBUF(b200_pileup1_t, ents);
    DBUF(int32_t, clip); DBUF(int64_t, next); DBUF(int32_t, cig_x); DBUF(int32_t, cig_y);
    DBUF(double, baq_f); DBUF(int32_t, baq_idx); DBUF(uint8_t, ref_codes); DBUF(uint16_t, ent); DBUF(uint16_t, ent2); DBUF(uint32_t, x_off); DBUF(char, x_dat); DBUF(int32_t, ov_pairs);
    DBUF(float, gl_out); DBUF(int32_t, gl_n); DBUF(uint32_t, gl_flag);
    void *d_acc = nullptr;
    unsigned long long *d_misc = nullptr;
    double *d_beta = nullptr, *d_fk = nullptr, *d_lhet = nullptr;   // errmod tables
    double fk_depcorr = 0;                                             // dependency coefficient d_fk was built for
    double *d_q2p = nullptr, *d_qthr = nullptr;                      // BAQ tables

    // batch state
    bool staged = false, has_ref = false, has_prev = false, has_rbits = false, has_clip = false, maxdrop_applied = false;
    int64_t n = 0; int32_t n_files = 0, tid = 0; int64_t tid_len = 0;
    std::string name;
    b200_stage_conf_t sconf;
    int64_t win_base = 0, ref_beg = 0, ref_n = 0, ref_len = 0;
    int64_t ncols_cov = 0, ncols_all = 0; int32_t ncols_max = 0, n_groups = 0;
    int64_t acc_n_kept = 0; int32_t max_rend = 0;
    unsigned long long sum_rlen = 0, sum_indel_text = 0, sum_rlen_gen = 0;
    size_t last_out_len = 0;
    uint64_t gl_rng_draws = 0;   // hts_drand48 draws consumed so far by errmod's ks_shuffle
    std::vector<int64_t> h_file_start;
    std::vector<int32_t> h_clip_tmp;

    void free_all()
    {
        void *ps[] = { qual0, mapq0, pos, flag, mapq, l_qseq, n_cigar, cigar_off, qual_off, mtid, mpos, isize, prev, rbits, cigar, seq4, qual,
                       ref, dname, file_start, state, rlen, desc, endv, pmax, glo, ghi, status, out, bed_beg, bed_end, col_n,
                       col_off, col_state, tile_total, ovf_cnt, ovf_off, ovf_idx, ss_diff, ss_nplp, ss_fail, ss_extra, status2, ents, clip, next, cig_x, cig_y, baq_f, baq_idx, ref_codes, ent, ent2, x_off, x_dat, ov_pairs, gl_out, gl_n, gl_flag, d_beta, d_fk, d_lhet, d_q2p, d_qthr };
        for (void *p : ps) if (p) cudaFree(p);
    }
};

namespace plp { struct RawSoA; }
using plp::RawSoA;
int build_ranges(b200_engine *e, int *max_range);
int launch_baq(b200_engine *e, const RawSoA &r, const b200_stage_conf_t &cf);
int launch_overlap(b200_engine *e, const RawSoA &r);
int launch_depth_clip(b200_engine *e, const RawSoA &r);
