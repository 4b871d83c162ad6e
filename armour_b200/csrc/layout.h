// Device-side data layout of a batch of planning problems (HBM, structure of arrays).
//
// All arrays are problem-major; inside a problem the time interval is the slow index because every
// kernel assigns a CTA to one (problem, time interval) or one (problem, block of TB intervals), so
// each CTA streams one contiguous chunk.
#pragma once
#include <cstdint>

#include "robot_constants.h"

namespace armour {

#ifndef ARMOUR_TB
#define ARMOUR_TB 8
#endif
constexpr int TB = ARMOUR_TB;      // time intervals per CTA ("chunk") in the constraint kernels
constexpr int HP_CAP = 32;         // most candidate half-spaces stored for one (link, interval, obstacle) row
constexpr int HP_OVERFLOW = 255;   // row count marker: no stored list, evaluate the row from the generators
constexpr double K_DOMAIN = 1.0 + 1e-6;        // the candidate lists are exact for |k_j| <= K_DOMAIN
constexpr double HP_RHO_SCALE = 1.0 + 3e-5;    // >= K_DOMAIN^21 (largest total degree of a link monomial)

struct Batch {
    int nprob;     // problems in flight
    int T;         // time intervals
    int NJ;        // links
    int O;         // obstacles per problem (same for the whole batch)
    int capL;      // stored k-only monomials per link reach set
    int capU;      // stored k-only monomials per torque reach set
    int epoch;     // ordinal of the build that filled the tables (> 0); status[] and the unit flags are stamped with it
    // inputs
    const double* q0;         // [p][NF]
    const double* qd0;        // [p][NF]
    const double* qdd0;       // [p][NF]
    const double* obstacles;  // [p][O][12]
    // ARMTD comparison planner only (nullptr otherwise): cos / sin models of the joint reachable set handed in instead of
    // derived from the Bezier trajectory, [p][t][NF][6] = cos centre, k-coefficient, error coefficient, then the same for sin
    const double* jrs_ext;
    // reach sets written by the build kernel (or armour_import_reachsets)
    int* link_n;              // [p][t][NJ]
    double* link_c;           // [p][t][NJ][3]
    uint16_t* link_key;       // [p][t][NJ][capL]   2 bits per k_j (reference degree hash, k-only part)
    double* link_g;           // [p][t][NJ][capL][3]
    int* u_n;                 // [p][t][NF]
    double* u_c;              // [p][t][NF]
    double* u_r;              // [p][t][NF]         radius of the reduced nominal torque PZ
    uint16_t* u_key;          // [p][t][NF][capU]
    double* u_g;              // [p][t][NF][capU]
    double* torque_radius;    // [p][j*T + t]
    double* link_gens;        // [p][t][NJ][18]     column-major 3x6
    double* link_r;           // [p][t][NJ][3]      diag of the radius block of link_gens (all an evaluation needs)
    // collision half-space candidates: the number of candidates per row [p][t/TB][l][t%TB][o] (HP_OVERFLOW: no list), and per
    // problem the number of rows without a list.  The records themselves live in the evaluation image (img below).
    unsigned char* hp_cnt;
    int* hp_slow;
    // evaluation images, one fixed slot of img_chunk() bytes per chunk [p][t/TB]: everything k_constraints reads for one
    // (problem, TB intervals), packed at the end of every build so that the kernel reads only the bytes it uses.
    //   header   int2 [TB][NJ] link tables (first double of the table in the image, monomials)
    //            int4 [TB][NF] torque tables (first coefficient in doubles, first key in uint16 units, monomials, 0)
    //            double [TB][NJ][3] link centres, [TB][NJ][3] link radii, [TB][NF] torque centres, [TB][NF] torque radii
    //            uint32 [ngrp] stored candidates of the rows before row 32 g; uint8 [rows] candidate counts (hp_cnt)
    //   img_hdr()  candidate records (s*Cx, s*Cy, s*Cz, b) row after row in scan order (CSR: rows in the chunk's x order)
    //   then     link tables back to back, one 32-byte record (3 coefficients, key in the low 16 bits of the fourth double)
    //            per monomial; torque coefficients of all tables back to back, then their keys
    // During the build k_hyperplanes writes each row's candidates into a fixed run of HP_CAP records at img_hdr(); the pack
    // kernel compacts them in place (a record never moves up) and appends the tables.
    unsigned char* img;
    // outputs of the last evaluation
    double* link_sliced;      // [t][NJ][3] of problem 0 (armtd_NLP::link_sliced_center)
    int* status;              // [p] epoch * 8 + failure code of a build that overflowed a table (see failed()): evaluations
                              // of such a problem return fail-safe rows
    // optional indirection for launches over a subset of the problems (the batched solver's still-running list):
    // CTA row y works on problem plist[y]; nullptr = identity
    const int* plist;

    // byte offsets inside one evaluation image (see img)
    __host__ __device__ int img_rows() const { return NJ * TB * O; }
    __host__ __device__ size_t img_ut() const { return size_t(TB) * NJ * 8; }
    __host__ __device__ size_t img_lc() const { return img_ut() + size_t(TB) * NF * 16; }
    __host__ __device__ size_t img_lr() const { return img_lc() + size_t(TB) * NJ * 24; }
    __host__ __device__ size_t img_uc() const { return img_lr() + size_t(TB) * NJ * 24; }
    __host__ __device__ size_t img_ur() const { return img_uc() + size_t(TB) * NF * 8; }
    __host__ __device__ size_t img_grp() const { return img_ur() + size_t(TB) * NF * 8; }
    __host__ __device__ size_t img_cnt() const { return img_grp() + size_t(img_rows() + 31) / 32 * 4; }
    __host__ __device__ size_t img_hdr() const { return (img_cnt() + img_rows() + 127) / 128 * 128; }
    __host__ __device__ size_t img_chunk() const {
        const size_t tables = size_t(TB) * NJ * capL * 32 + size_t(TB) * NF * capU * 10;
        return (img_hdr() + size_t(img_rows()) * HP_CAP * 32 + tables + 127) / 128 * 128;
    }
    __host__ __device__ int m() const { return NF * T + NJ * T * O + 4 * NF; }
    // failure code of problem p in the CURRENT build (0: none); stamps of older builds do not count
    __device__ int failed(int p) const { return (status[p] >> 3) == epoch ? (status[p] & 7) : 0; }
};

}  // namespace armour
