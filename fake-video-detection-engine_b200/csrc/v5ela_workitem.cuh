// v5ela_workitem.cuh — the per-work-item band loop shared by the CUDA kernel and the CPU thread emulator (tests/emu).
//
// V5_FOR_THREADS(body) runs `body` for every thread of the CTA and ends with a CTA-wide barrier:
//   device : body executes once with tid = threadIdx.x, then __syncthreads()
//   emu    : body executes NT times in a loop (one pass per emulated thread) — the barrier is the loop end.
// Per-thread state that must survive a barrier lives in `acc` (a register struct on the device, an array in the emulator).
#pragma once
#include "v5ela_device.cuh"

namespace V5_NS {

// V5_FOR_WARP(body): same, but the ordering point is only warp-wide (device: __syncwarp()).
// V5_BLOCK_TASK / V5_GET_TASK: the block-stage task of a thread is computed once per round on the device and once per
// sub-stage loop in the emulator.
#ifdef __CUDA_ARCH__
#define V5_BLOCK_TASK(t) const BlockTask t = block_task_of<FAST>((int)threadIdx.x, S, p, g, r, want_y, round);
#define V5_GET_TASK(t) (void)0
#define V5_FOR_WARP(...)                     \
    {                                        \
        const int tid = (int)threadIdx.x;    \
        ThreadAcc &acc = acc_store[0];       \
        (void)acc;                           \
        __VA_ARGS__;                         \
    }                                        \
    __syncwarp();
#define V5_FOR_THREADS(...)                  \
    {                                        \
        const int tid = (int)threadIdx.x;    \
        ThreadAcc &acc = acc_store[0];       \
        (void)acc;                           \
        (void)tid;                           \
        __VA_ARGS__;                         \
    }                                        \
    __syncthreads();
#define V5_FOR_THREADS_NOSYNC(...)           \
    {                                        \
        const int tid = (int)threadIdx.x;    \
        ThreadAcc &acc = acc_store[0];       \
        (void)acc;                           \
        __VA_ARGS__;                         \
    }
// V5_FOR_EACH_WARP(body): warp-collective work (the tensor-core block stage). Device: every thread runs `body`; emulator: `body`
// runs once per warp with tid = 32 * warp and does the whole warp's work. Ends with a CTA barrier.
#define V5_FOR_EACH_WARP(...)                \
    {                                        \
        const int tid = (int)threadIdx.x;    \
        __VA_ARGS__;                         \
    }                                        \
    __syncthreads();
#else
// V5_EMU_REVERSE: the emulated threads of a phase run last to first — any order must give the same result, and the two orders
// together catch a buffer that one thread of a phase overwrites while another still reads it, whichever of them has the lower index.
#if defined(V5_EMU_REVERSE) && V5_EMU_REVERSE
#define V5_EMU_TID_LOOP(step) for (int tid = NT - (step); tid >= 0; tid -= (step))
#else
#define V5_EMU_TID_LOOP(step) for (int tid = 0; tid < NT; tid += (step))
#endif
#define V5_FOR_EACH_WARP(...)                        \
    V5_EMU_TID_LOOP(32) {                            \
        __VA_ARGS__;                                 \
    }
#define V5_FOR_THREADS_NOSYNC(...) V5_FOR_THREADS(__VA_ARGS__)
#define V5_BLOCK_TASK(t)
#define V5_GET_TASK(t) const BlockTask t = block_task_of<FAST>(tid, S, p, g, r, want_y, round)
#define V5_FOR_WARP(...)                     \
    V5_EMU_TID_LOOP(1) {                     \
        ThreadAcc &acc = acc_store[tid];     \
        (void)acc;                           \
        __VA_ARGS__;                         \
    }
#define V5_FOR_THREADS(...)                  \
    V5_EMU_TID_LOOP(1) {                     \
        ThreadAcc &acc = acc_store[tid];     \
        (void)acc;                           \
        __VA_ARGS__;                         \
    }
#endif

// End of a work item: per-thread texture partials -> shared memory, then shared memory -> the frame's record with
// global atomics (<= 768 + 3 per CTA per work item). tex_maxabs is a uint16 field; while the fused kernel runs, the
// aligned 32-bit word that starts at it (its upper half, ela_max[0..1], is still zero) is the atomicMax target — the
// finalize kernel writes ela_max afterwards.
#ifdef __CUDA_ARCH__
V5_DEV void flush_partials(int tid, Smem &S, ThreadAcc &acc)
{
    unsigned long long sq = acc.tex_sumsq, sa = acc.tex_sumabs;
    uint32_t mx = acc.tex_maxabs;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        sa += __shfl_xor_sync(0xffffffffu, sa, o);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((tid & 31) == 0) {
        atomicAdd(&S.tex_sumsq, sq);
        atomicAdd(&S.tex_sumabs, sa);
        atomicMax(&S.tex_maxabs, mx);
    }
}
V5_DEV void flush_global(int tid, Smem &S, v5ela_record *rec, uint32_t *tex_hist)
{
    for (int i = tid; i < 3 * 256; i += NT) {
        const uint32_t c = (&S.hist[0][0])[i];
        if (c) atomicAdd(&rec->ela_hist[0][0] + i, c);
    }
    if (tex_hist)
        for (int i = tid; i < 256; i += NT) {
            const uint32_t c = S.tex_hist[i];
            if (c) atomicAdd(tex_hist + i, c);
        }
    if (tid == 0) {
        atomicAdd(reinterpret_cast<unsigned long long *>(&rec->tex_sumabs), S.tex_sumabs);
        atomicAdd(reinterpret_cast<unsigned long long *>(&rec->tex_sumsq), S.tex_sumsq);
        atomicMax(reinterpret_cast<uint32_t *>(&rec->tex_maxabs), S.tex_maxabs);
    }
}
#else
inline void flush_partials(int, Smem &S, ThreadAcc &acc)
{
    S.tex_sumsq += acc.tex_sumsq;
    S.tex_sumabs += acc.tex_sumabs;
    if (acc.tex_maxabs > S.tex_maxabs) S.tex_maxabs = acc.tex_maxabs;
}
inline void flush_global(int tid, Smem &S, v5ela_record *rec, uint32_t *tex_hist)
{
    for (int i = tid; i < 3 * 256; i += NT) (&rec->ela_hist[0][0])[i] += (&S.hist[0][0])[i];
    if (tex_hist)
        for (int i = tid; i < 256; i += NT) tex_hist[i] += S.tex_hist[i];
    if (tid == 0) {
        rec->tex_sumabs += S.tex_sumabs;
        rec->tex_sumsq += S.tex_sumsq;
        if (S.tex_maxabs > rec->tex_maxabs) rec->tex_maxabs = (uint16_t)S.tex_maxabs;
    }
}
#endif

// The ghost cells of MCU row R of the work item's strip -> the entry's map (plain stores: each MCU belongs to one work item), and
// zeroed for MCU row R + 2.
V5_DEV void flush_ghost_row(int tid, Smem &S, const Geo &g, uint32_t *ghost, int R)
{
    for (int c = tid; c < g.m1 - g.m0; c += NT) {
        ghost[(int64_t)R * g.mw + g.m0 + c] = S.ghost[R & 1][c];
        S.ghost[R & 1][c] = 0;
    }
}

// RAGGED: every frame has its own size and pointers (KParams::frames); only with the general instantiation.
// SWEEP (with RAGGED; the sweep kernel): every entry also has its own quantisation tables and, optionally, a JPEG-ghost map
// (sweep_entries). The residual stage of iteration r completes MCU row r - 1, the loop's end the segment's last one.
template <bool FAST, bool TEXHIST, bool RAGGED = false, bool SWEEP = false>
V5_DEV void process_work_item(Smem &S, const KParams &p, int work, ThreadAcc *acc_store)
{
    static_assert(!RAGGED || (!FAST && !TEXHIST), "ragged batches take the general instantiation");
    static_assert(!SWEEP || RAGGED, "a sweep is a ragged batch");
    Geo g;
    int frame;
    make_geo<RAGGED>(p, work, g, frame);
    const SweepEntry *const entry = SWEEP ? sweep_entries(p.frames, p.n) + frame : nullptr;
    const QuantTab *const sweep_q = SWEEP ? sweep_quant(p.frames, p.n) + 2 * entry->slot : nullptr;
    uint32_t *const ghost = SWEEP ? entry->ghost : nullptr;

    V5_FOR_THREADS({
        for (int i = tid; i < 3 * 256; i += NT) (&S.hist[0][0])[i] = 0;
        if (TEXHIST)
            for (int i = tid; i < 256; i += NT) S.tex_hist[i] = 0;
        if (SWEEP)
            for (int i = tid; i < 2 * TW_MAX; i += NT) (&S.ghost[0][0])[i] = 0;
        for (int i = tid; i < 2 * 64; i += NT) {
            const QuantTab &q = SWEEP ? sweep_q[i >> 6] : p.q[i >> 6];
            const int k = i & 63;
#if V5_MMA_BLOCKS
            S.qtab[i >> 6][mma::qswz_pos(k)] = mma::qswz_entry(q.recip[k], q.bias[k], q.t[k], q.unbias[k]);
#else
            S.qtab[i >> 6][k] = QEntry{q.recip[k], q.bias[k], q.t[k], q.unbias[k]};
#endif
        }
#if V5_MMA_BLOCKS
#ifdef __CUDA_ARCH__
        for (int i = tid; i < 32 * 8; i += NT) S.lane[i & 7][i >> 3] = reinterpret_cast<const U4 *>(p.lane_consts)[i];   // word i & 7 of lane i >> 3
#else
        for (int i = tid; i < 32 * (int)(sizeof(mma::LaneConsts) / 16); i += NT)
            reinterpret_cast<U4 *>(S.lane)[i] = reinterpret_cast<const U4 *>(p.lane_consts)[i];
#endif
#endif
        if (tid == 0) {
            S.tex_sumabs = 0;
            S.tex_sumsq = 0;
            S.tex_maxabs = 0;
        }
        acc.tex_sumabs = 0;
        acc.tex_sumsq = 0;
        acc.tex_maxabs = 0;
    })

    // Bands r0-1 and r1 only contribute decoded chroma / original luma to the rows next to them.
    const int r_first = g.r0 > 0 ? g.r0 - 1 : 0;
    // FAST: 16-byte aligned frames whose strips are whole multiples of 48 bytes — the bulk copies cover every band completely
    const bool bulk = FAST || use_bulk(p, g);
    const bool rest = !FAST && load_rest_needed(p, g, bulk);
    V5_FOR_THREADS(if (bulk) stage_prefetch(tid, S, p, g, r_first))
    // Split barrier between the residual stage of one band and the conversion of the next (stage_convert): arrive there,
    // wait in front of the first store here. Only in the bulk-copy-only instantiation with two RGB buffers. Measured 3 %
    // SLOWER than the plain CTA barrier (profiles/r01/variants.txt) and therefore off: a compile-time variant.
#ifndef V5_SPLIT_BARRIER
#define V5_SPLIT_BARRIER 0
#endif
    constexpr bool SPLIT = FAST && RGB_BUFS == 2 && V5_SPLIT_BARRIER;
#ifndef V5_PAIR_ROWS
#define V5_PAIR_ROWS 1
#endif
    constexpr bool PAIRS = FAST && V5_PAIR_ROWS;             // two rows per residual unit (stage_residual_pairs)
    constexpr bool FUSE = FAST && FUSE2_OK;                  // two-phase band loop (v5ela_device.cuh)
    static_assert(!FUSE || (PAIRS && NT >= RGB_PITCH / 16 + 2 * (Y_PITCH / 16)), "two-phase band loop: pairs, and one thread per carried 16 bytes");
    if (FUSE) {
        // phase 1: residual stage of the band before (`pend`) + conversion of band r; phase 2: carries, request for band r+1 (its
        // buffer was last read by the residual stage just finished) and the block stage of band r.
        int pend = -1;
        for (int r = r_first; r <= g.r1; r++) {
            const bool has_band = r < g.mh;
            const bool want_y = r >= g.r0 && r < g.r1;
            const bool next_band = r + 1 <= g.r1 && r + 1 < g.mh;
            if (!has_band && 16 * r - 1 >= g.h) break;      // nothing left below the image
            V5_FOR_THREADS({
                if (pend >= 0) stage_residual_pairs<TEXHIST>(tid, S, p, g, acc, pend);
                if (has_band) {
                    mbar_wait(reinterpret_cast<uint64_t *>(&S.full_bar[rb(r)]), (acc.phase >> rb(r)) & 1u);
                    acc.phase ^= 1u << rb(r);
                    stage_convert(tid, S, p, g, r, acc, false, false, false);
                }
            })
            pend = r;
            V5_FOR_THREADS_NOSYNC({
                if (next_band) stage_prefetch(tid, S, p, g, r + 1);
                stage_carries(tid, S, r, has_band);
            })
            if (has_band) {
#if V5_MMA_BLOCKS
                V5_FOR_EACH_WARP(stage_blocks_mma<FAST>(tid, S, p, g, r, want_y))
#else
                const int rounds = (blocks_in_band(g, want_y) + NT / 4 - 1) / (NT / 4);
                for (int round = 0; round < rounds; round++) {
                    V5_BLOCK_TASK(t)
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_rows_fwd(tid, S, t))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_cols(tid, S, t, acc.col))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_cols_store(tid, S, t, acc.col))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_rows_inv(tid, S, t))
                }
                V5_FOR_THREADS((void)0)
#endif
            } else {
                V5_FOR_THREADS((void)0)
            }
        }
        if (pend >= 0) {
            V5_FOR_THREADS(stage_residual_pairs<TEXHIST>(tid, S, p, g, acc, pend))
        }
    } else {
        bool pending = false;                                   // an arrive on done_bar that nobody has waited for yet
        for (int r = r_first; r <= g.r1; r++) {
            const bool has_band = r < g.mh;
            const bool want_y = r >= g.r0 && r < g.r1;
            const bool next_band = r + 1 <= g.r1 && r + 1 < g.mh;
            if (!has_band && 16 * r - 1 >= g.h) break;          // nothing left below the image
            if (has_band) {
                // Band r was requested one iteration ago; request band r+1 into the other buffer (free since the residual
                // stage of iteration r-1), fetch what the bulk copy does not cover, then wait for band r.
                if (rest) {                                     // ragged right edge / unaligned frames only
                    V5_FOR_THREADS(stage_load_rest(tid, S, p, g, r, bulk))
                }
                // every thread waits for the bulk copy itself, so no CTA barrier is needed before the conversion
                V5_FOR_THREADS({
                    const bool defer = SPLIT && pending;         // the other RGB buffer may still be read: prefetch after the wait
                    if (!defer && RGB_BUFS == 2 && bulk && next_band) stage_prefetch(tid, S, p, g, r + 1);
                    if (bulk) {
                        mbar_wait(reinterpret_cast<uint64_t *>(&S.full_bar[rb(r)]), (acc.phase >> rb(r)) & 1u);
                        acc.phase ^= 1u << rb(r);
                    }
                    stage_convert(tid, S, p, g, r, acc, defer, defer && bulk && next_band);
                })
                pending = false;
                // single staging buffer: band r has been consumed by every warp (barrier above), fetch band r+1 over it now
                if (RGB_BUFS == 1 && bulk && next_band) {
                    V5_FOR_WARP(stage_prefetch(tid, S, p, g, r + 1))
                }
#if V5_MMA_BLOCKS
                V5_FOR_EACH_WARP(stage_blocks_mma<FAST>(tid, S, p, g, r, want_y))
#else
                const int rounds = (blocks_in_band(g, want_y) + NT / 4 - 1) / (NT / 4);
                for (int round = 0; round < rounds; round++) {
                    V5_BLOCK_TASK(t)
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_rows_fwd(tid, S, t))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_cols(tid, S, t, acc.col))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_cols_store(tid, S, t, acc.col))
                    V5_FOR_WARP(V5_GET_TASK(t); blocks_rows_inv(tid, S, t))
                }
                V5_FOR_THREADS((void)0)
#endif
            }
            if (SPLIT && next_band) {
                V5_FOR_THREADS_NOSYNC({
                    if (PAIRS) stage_residual_pairs<TEXHIST>(tid, S, p, g, acc, r);
                    else stage_residual<FAST, TEXHIST>(tid, S, p, g, acc, r);
                    mbar_arrive(reinterpret_cast<uint64_t *>(&S.done_bar));
                })
                pending = true;
            } else {
                V5_FOR_THREADS(if (PAIRS) stage_residual_pairs<TEXHIST>(tid, S, p, g, acc, r); else stage_residual<FAST, TEXHIST, SWEEP>(tid, S, p, g, acc, r, ghost != nullptr))
            }
            if (SWEEP && ghost && r - 1 >= g.r0 && r < g.r1) {
                V5_FOR_THREADS(flush_ghost_row(tid, S, g, ghost, r - 1))
            }
        }
    }

    V5_FOR_THREADS(flush_partials(tid, S, acc); if (SWEEP && ghost) flush_ghost_row(tid, S, g, ghost, g.r1 - 1))
    V5_FOR_THREADS(flush_global(tid, S, p.records + frame, TEXHIST ? p.tex_hist + (int64_t)frame * 256 : nullptr))
}

}  // namespace V5_NS
