// common.cuh -- shared scaffolding for the quasimodo_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/quasimodo_b200.h"

#define QM_WARP 32

struct qm_scratch {
    void  *ptr = nullptr;
    size_t cap = 0;
};

// stage timers (CUDA events on the launching stream; enabled by qm_profile_enable)
enum { QM_ST_SEED = 0, QM_ST_ADVANCE, QM_ST_EXTEND, QM_ST_PAIR, QM_ST_PILEUP, QM_ST_H2D, QM_ST_D2H, QM_ST_OTHER, QM_ST_RESCUE, QM_ST_N };
struct qm_prof_span { int stage; cudaEvent_t e0, e1; };

struct qm_ctx {
    int device = -1;
    int sm_count = 0;
    std::string err;
    // scratch arenas grown on demand (never shrunk); index = purpose.  32-36: the tuples of duplicate marking and the depth cap
    // (dedup.cu, depthcap.cu, sort.cu, sample.cu);
    // 37-39: BAM records in (bamin.cu: staged record stream, file-order rows and pairing state, pair layout)
    qm_scratch scratch[40];
    cudaStream_t own_stream = nullptr, copy_stream = nullptr;
    // side streams: the independent per-class extension kernels of one round run concurrently (fork/join by events)
    cudaStream_t side[12] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[12] = {};
    // host-entry hand-over to qm_align_se: the read batch arrives in se_n_parts pieces (reads [.., se_part_end[i]) are in
    // device memory once se_part_ev[i] has fired), so seeding can start on the first piece while the rest is still
    // being copied; consumed (reset to 0) by the next qm_align_se call
    int se_n_parts = 0;
    int64_t se_part_end[16] = {};
    cudaEvent_t se_part_ev[16] = {};
    // ... and when se_pk is set the pieces arrive PACKED (2 bits per base at se_pk, N flags at se_mk, row strides se_sp / se_sm):
    // qm_align_se expands reads [r0, r1) into the batch's code rows on the stream that is about to read them
    const uint8_t *se_pk = nullptr, *se_mk = nullptr;
    int se_sp = 0, se_sm = 0;
    int64_t text_bytes = 0;            // length of the text the last qm_mpileup_text left in scratch 17
    void *h_pinned = nullptr;          // 8 KB of page-locked host memory for the small per-round read-backs
    bool prof_on = false;
    std::vector<qm_prof_span> prof_spans;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[QM_ST_N] = {};
    long long prof_launches[QM_ST_N] = {};
};

// open / close a timed span on stream st (no-ops unless profiling is enabled)
int qm_prof_begin(qm_ctx *ctx, int stage, cudaStream_t st);
void qm_prof_end(qm_ctx *ctx, int stage, int span, cudaStream_t st, int launches);

// grow-only scratch; contents are NOT preserved across a growth
int qm_scratch_reserve(qm_ctx *ctx, int which, size_t bytes, void **out);
int qm_fail(qm_ctx *ctx, int code, const char *fmt, ...);

#define QM_CUDA(ctx, call)                                                                         \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return qm_fail((ctx), QM_ECUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,           \
                           cudaGetErrorString(e__));                                               \
    } while (0)

static __device__ __forceinline__ int qm_lane() { return threadIdx.x & 31; }
