// engine.cu -- C ABI (include/ra_engine.h) of the B200 batched multi-Raft engine.
//
// Host side: owns the HBM Struct-of-Arrays, stages host buffers, launches per step
//   raft_step_kernel     -- the hot path: one thread per member row, steady-state fast paths
//   raft_general_kernel  -- the rows that left the fast paths, one thread per stalled row
// (device logic: raft_step.cuh, row helpers: raft_row.cuh) and, around ra_engine_step,
//   ingest / pack + scan + gather -- flat host batch <-> per-row slots
// There is no CPU fallback: without a CUDA device ra_engine_create fails with
// RA_E_NODEVICE and nothing else works.
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>

#include "raft_step.cuh"
#include "raft_row.cuh"


// ------------------------------------------------------------------------------------------
// the hot kernel
// ------------------------------------------------------------------------------------------
#ifndef NST
#define NST 3                               // shared-memory stages per warp: NST record tiles (1 or 2 KB) in flight
#endif
#ifndef MINB
#define MINB 5                              // CTAs per SM the register allocation is held to: 20 warps,
                                            // <= 96 registers (no spills), 5 x 39 KB of shared memory
#endif
#ifndef MINB_NARROW
#define MINB_NARROW 5                       // the narrow pass (32-bit index arithmetic) needs ~84 registers: measured
#endif                                      // 0.0796 ms at 5 CTAs/SM (no spill), 0.0816 at 6 (80 regs, 24 B), 0.0865 at 7 (72, 68 B)
#define TILE_BYTES (RT * 64)
#define RA_BAR_WORDS 64                       // barrier flag words behind mbox_cnt[b] (one per source shard)
#define WARPS (CTA_T / 32)
// Cols::counters: [0..7] ra_counters' aggregate fields, [8..135] stall histogram (role x type),
// [136..142] the reference's per-path counters in the order of Member::c_ref (CR_*)
#define RA_N_COUNTERS (8 + 8 * 16 + 8)
#define RA_CNT_REF 136

// ---- TMA (cp.async.bulk) + mbarrier, sm_90+/sm_100a --------------------------------------
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64* bar, u32 count)
{ asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_fence_init()
{ asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async()
{ asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes)
{ asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity)
{
    // bounded: a TMA that never lands must fail the launch loudly, not hang the GPU
#pragma unroll 1
    for (u32 spins = 0; spins < (1u << 24); spins++) {
        u32 done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return;
    }
    __trap();
}
// one bulk copy global -> shared, completion counted in bytes on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_tile(void* dst_smem, const void* src_gmem, u32 bytes, u64* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Shared memory of one CTA = 4 independent warps x 32 member rows:
//   stage[warp][NST][4][32] x 16 B   record tiles staged by TMA, chunk-major (conflict-free LDS.128)
//   bars[warp][NST]                  one mbarrier per stage
//   peers[3][8][128] x 8 B           per-thread peer columns (next, match, commit_index_sent), lazy
// (narrow pass, NARROW = true: the peer cells are 8 + 4 bytes instead of 16 + 8)
template <int MM, bool NARROW = false>
struct StepSmem {
    ulonglong2 stage[WARPS][NST][4 * RT];
    ulonglong2 peers_nm[PSTR * CTA_T / (NARROW ? 2 : 1)];   // [s][thread] {next_index, match_index}
    // [s][thread] commit_index_sent, directly behind peers_nm (narrow: 4-byte cells, no column for the own slot)
    u64 peers_cs[NARROW ? (PSTR > 1 ? PSTR - 1 : 1) * CTA_T / 2 : PSTR * CTA_T];
    u64 bars[WARPS][NST];
};

// ---- the two kernels of a step ---------------------------------------------------------------
// raft_step_kernel     every row, steady-state fast paths only.  A row whose next event is not
//                      covered STALLS: it stops, saves its step context (64 B) to a compact list
//                      and writes its state back as far as it got.
// raft_general_kernel  one thread per stalled row (dense, so a rare event does not idle 31
//                      other lanes): resumes at the stalled event with the general path
//                      (process_event), runs the row's end-of-step.
// Both run the same end-of-step code; together they evaluate every event exactly once, in order.

__device__ __forceinline__ void flush_counters(const Cols& C, u32 lane, u32 k_events, u32 k_commits, u32 k_applied,
                                               u32 k_msgs, u32 k_dropped, u32 k_elect, u32 k_fatal)
{
    // per-launch device counters: one REDUX per counter, one atomic per warp and counter that moved
    if (__any_sync(0xffffffffu, (k_events | k_fatal | k_dropped | k_msgs) != 0)) {
        k_events = __reduce_add_sync(0xffffffffu, k_events); k_commits = __reduce_add_sync(0xffffffffu, k_commits);
        k_applied = __reduce_add_sync(0xffffffffu, k_applied); k_msgs = __reduce_add_sync(0xffffffffu, k_msgs);
        k_dropped = __reduce_add_sync(0xffffffffu, k_dropped); k_elect = __reduce_add_sync(0xffffffffu, k_elect);
        k_fatal = __reduce_add_sync(0xffffffffu, k_fatal);
        if (lane == 0) {
            if (k_events)  atomicAdd(&C.counters[0], (u64)k_events);
            if (k_commits) atomicAdd(&C.counters[1], (u64)k_commits);
            if (k_applied) atomicAdd(&C.counters[2], (u64)k_applied);
            if (k_msgs)    atomicAdd(&C.counters[3], (u64)k_msgs);
            if (k_dropped) atomicAdd(&C.counters[4], (u64)k_dropped);
            if (k_elect)   atomicAdd(&C.counters[5], (u64)k_elect);
            if (k_fatal)   atomicAdd(&C.counters[6], (u64)k_fatal);
        }
    }
}

// plane bit masks: 32 bits cover groups of up to 7 members, the generic kernel needs 36
template <bool SMALL> struct PlaneMask { typedef u32 type; };
template <> struct PlaneMask<false> { typedef u64 type; };
__device__ __forceinline__ u32 mask_ffs(u32 m) { return (u32)__ffs((int)m) - 1u; }
__device__ __forceinline__ u32 mask_ffs(u64 m) { return (u32)__ffsll((long long)m) - 1u; }
__device__ __forceinline__ u32 mask_or_warp(u32 m) { return __reduce_or_sync(0xffffffffu, m); }
__device__ __forceinline__ u64 mask_or_warp(u64 m)
{ return (u64)__reduce_or_sync(0xffffffffu, (u32)m) | ((u64)__reduce_or_sync(0xffffffffu, (u32)(m >> 32)) << 32); }

// the reference's counters: 7 byte-wide fields per row -> two 16-bit-field words per reduction
// (32 lanes x 255 < 65536), one atomic per warp and counter that moved
__device__ __forceinline__ void flush_ref_counters(const Cols& C, u32 lane, u64 c_ref)
{
    if (!__any_sync(0xffffffffu, c_ref != 0)) return;
    u32 w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u32 lo = (u32)(c_ref >> (16 * k)) & 0xffu, hi = (u32)(c_ref >> (16 * k + 8)) & 0xffu;
        w[k] = __reduce_add_sync(0xffffffffu, lo | (hi << 16));
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (w[k] & 0xffffu) atomicAdd(&C.counters[RA_CNT_REF + 2 * k], (u64)(w[k] & 0xffffu));
            if (2 * k + 1 < 7 && (w[k] >> 16)) atomicAdd(&C.counters[RA_CNT_REF + 2 * k + 1], (u64)(w[k] >> 16));
        }
    }
}

// Programmatic dependent launch (sm_90+).  A step is a chain of kernels on one stream (step kernel -> general kernel ->
// next step kernel ...), each reading what the one before wrote.  The two kernels of a step are launched with
// programmatic stream serialization: the next kernel's CTAs may be scheduled while this one's last CTAs still run
// (launch_dependents, at the start of every CTA), and grid_dep_wait -- the first statement of both kernels, before any
// memory access -- blocks until every earlier grid of the stream has completed and its writes are visible.  So the
// results are those of serial launches; what overlaps is the launch and the CTA ramp-up of the next kernel.
// (In a kernel launched without the attribute, or behind a copy, grid_dep_wait returns at once.)
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

#ifdef RA_WARP_TIMELINE
// Measurement build only (-DRA_WARP_TIMELINE, tools/warp_timeline.py): every warp of a hot-kernel launch that has
// work writes one record, indexed by its tile, read back through ra_debug_warp_timeline.  The default build has
// neither the buffer nor the export.
struct WarpTimeline {
    u64 t_entry, t_inputs, t_loop, t_exit;    // %globaltimer (ns): entry, per-row inputs landed, event loop done, exit
    u32 tile;
    u32 info;                                 // %smid | all lanes leaders << 16 | planes consumed << 24
    u32 pad[2];
};
#define RA_WTL_CAP (1u << 16)                 // warps recorded (tiles beyond are not)
__device__ WarpTimeline g_wtl[RA_WTL_CAP];
// the timestamp is taken after `dep` is available: a value the timed phase produced
__device__ __forceinline__ u64 wtl_now(u32 dep)
{ u64 t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) : "r"(dep) : "memory"); return t; }
__device__ __forceinline__ u32 wtl_smid() { u32 s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s; }
#endif

// the hot kernel, once per index width (raft_step.cuh): ra_wide::raft_step_kernel, ra_narrow::raft_step_kernel
namespace ra_wide {
#define RA_NARROW_PASS 0
#include "raft_step_kernel.cuh"
#undef RA_NARROW_PASS
}
#ifndef RA_NO_NARROW
namespace ra_narrow {
#define RA_NARROW_PASS 1
#include "raft_step_kernel.cuh"
#undef RA_NARROW_PASS
}
#endif

// general path for the stalled rows of this step (one thread per list entry)
__global__ void __launch_bounds__(CTA_T)
raft_general_kernel(const __grid_constant__ Cols C, const int cur, const FloodArgs F,
                    const StallCtx* __restrict__ stall_list, const u32* __restrict__ stall_count)
{
    constexpr int MM = MK_MM(0, TR_RUNTIME);
    __shared__ ulonglong2 s_peers[RA_MAX_MEMBERS * CTA_T + RA_MAX_MEMBERS * CTA_T / 2];   // nm[8][T] then cs[8][T]
    const u32 tid = threadIdx.x, lane = tid & 31u;
    grid_dep_wait();
    grid_dep_launch();
    if (*C.abort) return;
    const u32 n = *stall_count;
    for (u32 base = blockIdx.x * CTA_T; base < n; base += gridDim.x * CTA_T) {
        const u32 i = base + tid;
        u32 k_events = 0, k_commits = 0, k_applied = 0, k_msgs = 0, k_dropped = 0, k_elect = 0, k_fatal = 0;
        u64 k_ref = 0;
        if (i < n) {
            const ulonglong2* q = reinterpret_cast<const ulonglong2*>(&stall_list[i]);
            const ulonglong2 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
            const u32 r = (u32)q0.x, flags = (u32)(q0.x >> 32);
            u32 rem_mbox = (u32)q0.y, rem_loc = (u32)(q0.y >> 32);
            Member m;
            member_init(m, C, r, C.tc[r], C.lg[r], C.lw[r], C.ap[r], 0, cur, &s_peers[tid]);
            m.lrs_ok = 0;
            m.n_msgs = (u32)q1.x & 0xffffu; m.n_notes = ((u32)q1.x >> 16) & 0xffffu; m.status = (u32)(q1.x >> 32);
            m.sent_to = (u32)q1.y;
            { const u32 w = (u32)(q1.y >> 32); m.pn_type = w & 0xffu; m.pn_slot = (w >> 8) & 0xffu; m.wk = w >> 16; }
            m.pn_a = q2.x; m.pn_b = q2.y; m.pn_c = q3.x;
            u64 big = 0;                                        // see row_mark_wide
            if (flags & STALL_PENDING) {
                MT_SET(m.meta, 24, 1, 0);
                process_event<MM>(m, mk_rec(r, RA_EV_PIPELINE_RPCS, RA_NO_SLOT, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0));
                m.cold &= ~8u;
            }
#pragma unroll 1
            while (rem_mbox) {
                const u32 p = __ffs(rem_mbox) - 1; rem_mbox &= rem_mbox - 1;
                const Rec e = ld_rec_plane(C.mbox[cur], C.tiles, p, r);
                big |= rec_magnitude(e);
                if (MT_FATAL(m.meta)) m.c_pack += 1u;
                else if (flood_lost<MM>(F, C, m, r, e)) m.c_pack += 1u << 20;
                else if (!note_budget_ok(m)) budget_drop_record(m);
                else if (C.pure || !fast_event<MM>(m, e)) { process_event<MM>(m, e); m.cold &= ~8u; }
            }
#pragma unroll 1
            while (rem_loc) {
                const u32 p = __ffs(rem_loc) - 1; rem_loc &= rem_loc - 1;
                const Rec e = ld_rec_plane(C.loc, C.tiles, p, r);
                big |= rec_magnitude(e);
                if (MT_FATAL(m.meta)) m.c_pack += 1u;
                else if (!note_budget_ok(m)) budget_refuse_local(m);
                else if (C.pure || !fast_event<MM>(m, e)) { process_event<MM>(m, e); m.cold &= ~8u; }
            }
            peers_writeback<MM>(m);
            k_fatal = row_end_of_step<MM>(m, C, r, cur, F);
            member_writeback(m, C, r);
            row_mark_wide(C, r, m, big);
            k_events = m.c_pack & 0xffu; k_commits = m.c_commits; k_applied = m.c_applied;
            k_msgs = (m.c_pack >> 8) & 0xffu; k_dropped = m.c_pack >> 20; k_elect = (m.c_pack >> 16) & 15u;
            k_ref = m.c_ref;
        }
        flush_counters(C, lane, k_events, k_commits, k_applied, k_msgs, k_dropped, k_elect, k_fatal);
        flush_ref_counters(C, lane, k_ref);
    }
}

// ------------------------------------------------------------------------------------------
// plumbing kernels
// ------------------------------------------------------------------------------------------
__global__ void reset_empty_kernel(const Cols C)
{
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= C.rows) return;
    reset_row(C, r);
}

__global__ void load_rows_kernel(const Cols C, const ra_row_state* in, u32 n)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    load_row(C, in[i]);
}

__global__ void read_rows_kernel(const Cols C, ra_row_state* out, u32 n)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    read_row(C, out[i]);
}

__global__ void load_query_kernel(const Cols C, const ra_query_state* in, u32 n)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) load_query_row(C, in[i]);
}
__global__ void read_query_kernel(const Cols C, ra_query_state* out, u32 n)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) read_query_row(C, out[i]);
}

// flat host batch -> per-row local slots.  err[0]: 1 = ungrouped, 2 = too many for a row, 3 = bad row
__global__ void ingest_kernel(const Cols C, const ra_event* ev, u32 n, u32* err, const u32* sticky)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || *sticky) return;
    const u32 row = ev[i].row;
    if (row >= C.rows || ev[i].type > RA_EV_CONSISTENT_QUERY || ev[i].type == RA_EV_NONE) { atomicMax(err, 3u); return; }
    if (i > 0 && ev[i - 1].row == row) return;                 // not the head of its run
    u32 len = 1;
    while (i + len < n && ev[i + len].row == row && len <= RA_LOCAL_CAP) len++;
    if (len > RA_LOCAL_CAP) { atomicMax(err, 2u); return; }
    if (atomicCAS(&C.loc_n[row], 0u, len) != 0u) { atomicMax(err, 1u); return; }
    u32 tails = 0;
    for (u32 k = 0; k < len; k++)
        if (st_rec_plane(C.loc, C.tiles, k, row, ld_rec(&ev[i + k]))) tails |= 0x100u << k;
    if (tails) atomicOr(&C.loc_n[row], tails);
}

// the same for a batch of 32-byte host events: every record is a head (RS_PLAIN); err 3 also for an RPC type
__device__ __forceinline__ bool host_event_type_ok(u32 t)
{
    return t == RA_EV_WRITTEN || t == RA_EV_COMMAND || t == RA_EV_ELECTION_TIMEOUT || t == RA_EV_AWAIT_COND_TIMEOUT ||
           t == RA_EV_PIPELINE_RPCS || t == RA_EV_TICK || t == RA_EV_CONSISTENT_QUERY;
}
__global__ void ingest_host_kernel(const Cols C, const ra_host_event* ev, u32 n, u32* err, const u32* sticky)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || *sticky) return;
    const u32 row = ev[i].row;
    if (row >= C.rows || !host_event_type_ok(ev[i].type)) { atomicMax(err, 3u); return; }
    if (i > 0 && ev[i - 1].row == row) return;                 // not the head of its run
    u32 len = 1;
    while (i + len < n && ev[i + len].row == row && len <= RA_LOCAL_CAP) len++;
    if (len > RA_LOCAL_CAP) { atomicMax(err, 2u); return; }
    if (atomicCAS(&C.loc_n[row], 0u, len) != 0u) { atomicMax(err, 1u); return; }
    for (u32 k = 0; k < len; k++) {
        const ulonglong2* src = reinterpret_cast<const ulonglong2*>(&ev[i + k]);
        const ulonglong2 h = src[0], t = src[1];               // {row | type<<32 | flags<<40 | n<<48, term}, {a, b}
        ulonglong2* q = C.loc + rec_word(C.tiles, k, row, 0);
        const u64 type = (h.x >> 32) & 0xffull, flags = (h.x >> 40) & 0xffull, nn = (h.x >> 48) & 0xffffull;
        q[0] = make_ulonglong2(type | ((u64)RA_NO_SLOT << 8) | (flags << 16) | ((u64)RS_PLAIN << 24) | (nn << 32), h.y);
        q[RT] = t;
    }
}

// records that other shards sent to members of this engine -> mailbox planes of the next step.
// The slot is fixed by the record itself (sender slot, k-th record of that sender for this row),
// the receiver's count byte becomes max(k + 1).
__global__ void deliver_kernel(const Cols C, const int buf, const ra_event* inbox, const u32* counts, u32 cap)
{
    const u32 b = blockIdx.y;
    const u32 n = counts[b] < cap ? counts[b] : cap;
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        deliver_record(C, buf, ld_rec(&inbox[(size_t)b * cap + i]));
    }
}

__global__ void clear_loc_kernel(const Cols C)
{
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < C.rows) C.loc_n[r] = 0;
}

// ---- per-row output slots -> the caller's flat (row, seq)-ordered arrays ------------------------------
// offs = exclusive scan over the rows of out_n unpacked to msgs | notes << 32 (cub, through a transform
// iterator: no separate pass); offs[rows] = the totals.
struct PackCounts {
    __host__ __device__ __forceinline__ u64 operator()(const u32& v) const
    { return (u64)(v & 0xffffu) | ((u64)(v >> 16) << 32); }
};
typedef cub::TransformInputIterator<u64, PackCounts, const u32*> PackedIt;

// What the host reads when a call completes (pinned, mapped: written by gather_out_kernel itself, so a
// call needs no device->host copy whose size the host would first have to learn).
struct OutHdr { u64 n_msgs, n_notes; u32 status, n_ext; };    // status: ingest error 1..3 | 0x100 = outputs do not fit

// One warp per tile of 32 rows.  The warp's notes (and records) occupy one contiguous range of the output;
// a small table in shared memory maps every output position to (lane, k), then the range is written in
// 16-byte chunks, lane-consecutive: every store instruction of the warp is one contiguous 512-byte burst,
// which is what makes writing straight into HOST memory (PCIe posted writes) efficient.
// When the totals do not fit the caller's buffers (or the batch was rejected) nothing is written and the
// per-row slots are left alone, so that ra_engine_fetch_output can gather again.
__global__ void __launch_bounds__(128)
gather_out_kernel(const Cols C, const u64* __restrict__ offs, ulonglong2* __restrict__ msgs, const u64 msgs_cap,
                  ulonglong2* __restrict__ notes, const u64 notes_cap, OutHdr* hdr, const u32* err)
{
    __shared__ unsigned short tab[4][32 * (RA_NOTE_CAP > RA_MSG_CAP ? RA_NOTE_CAP : RA_MSG_CAP)];
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const u32 tile = blockIdx.x * 4 + warp;
    const u64 total = offs[C.rows];
    const u64 tm = total & 0xffffffffull, tn = total >> 32;
    const u32 bad = *err;
    const bool fits = tm <= msgs_cap && tn <= notes_cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        hdr->n_msgs = tm; hdr->n_notes = tn; hdr->n_ext = 0; hdr->status = bad | (fits ? 0u : 0x100u);
    }
    if (bad || !fits) return;
    const u32 r = tile * 32 + lane;
    const bool valid = r < C.rows;
    const u32 v = valid ? C.out_n[r] : 0u;
    if (!__any_sync(0xffffffffu, v != 0)) return;
    const u64 off = offs[valid ? r : C.rows];
    if (v) C.out_n[r] = 0;
    unsigned short* t = tab[warp];
    {   // notes: 2 chunks each
        const u32 nn = v >> 16;
        const u64 on = off >> 32;
        const u64 base = __shfl_sync(0xffffffffu, on, 0);
        const u32 cnt = (u32)(__shfl_sync(0xffffffffu, on + nn, 31) - base);
        for (u32 k = 0; k < nn; k++) t[(u32)(on - base) + k] = (unsigned short)((lane << 4) | k);
        __syncwarp();
        for (u32 c = lane; c < 2 * cnt; c += 32) {
            const u32 ent = t[c >> 1];
            const ulonglong2* src = reinterpret_cast<const ulonglong2*>(&C.onote[(size_t)(ent & 15u) * C.rows + tile * 32 + (ent >> 4)]);
            notes[(base << 1) + c] = src[c & 1u];
        }
        __syncwarp();
    }
    {   // RPC records: 4 chunks each
        const u32 nm = v & 0xffffu;
        const u64 om = off & 0xffffffffull;
        const u64 base = __shfl_sync(0xffffffffu, om, 0);
        const u32 cnt = (u32)(__shfl_sync(0xffffffffu, om + nm, 31) - base);
        if (cnt == 0) return;
        for (u32 k = 0; k < nm; k++) t[(u32)(om - base) + k] = (unsigned short)((lane << 4) | k);
        __syncwarp();
        for (u32 c = lane; c < 4 * cnt; c += 32) {
            const u32 ent = t[c >> 2];
            const ulonglong2* src = reinterpret_cast<const ulonglong2*>(&C.omsg[(size_t)(ent & 15u) * C.rows + tile * 32 + (ent >> 4)]);
            msgs[(base << 2) + c] = src[c & 3u];
        }
    }
}

// ---- compact note stream (ra_engine_set_note_format, include/ra_engine.h): one 16-byte unit per note ------------
// A note {row, type, slot, aux, a, b, c} becomes {row, type', n, aux, a} when slot = 0, 0 <= b - a < 256 and c is
// derivable: 0, or -- for WAL_APPEND -- the c of the row's previous WAL_APPEND note (bit 6 of type'), which the
// decoder remembers per row exactly as the engine does in Cols::wc.  Everything else gets bit 7, carries an index
// instead of a, and its {a, b, c} goes to the extension area behind the units.  In the steady-state flood every
// note is compact: half the device->host bytes.
__device__ __forceinline__ u32 note16_classify(const Cols& C, u32 r, u32 nn, u64& wc, u32& cmask)
{
    u32 extmask = 0;
    cmask = 0;
    for (u32 k = 0; k < nn; k++) {
        const ulonglong2* q = reinterpret_cast<const ulonglong2*>(&C.onote[(size_t)k * C.rows + r]);
        const ulonglong2 h = q[0], t = q[1];
        const u32 type = (u32)(h.x >> 32) & 0xffu, slot = (u32)(h.x >> 40) & 0xffu;
        const bool small = slot == 0 && t.x >= h.y && t.x - h.y < 256;
        bool cf = false;
        if (type == RA_NOTE_WAL_APPEND) { cf = t.y == wc; wc = t.y; }
        const bool compact = small && (type == RA_NOTE_WAL_APPEND ? cf : t.y == 0);
        if (!compact) extmask |= 1u << k;
        else if (cf) cmask |= 1u << k;
    }
    return extmask;
}

__global__ void note_ext_count_kernel(const Cols C, u32* __restrict__ next)
{
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > C.rows) return;
    if (r == C.rows) { next[r] = 0; return; }
    const u32 nn = C.out_n[r] >> 16;
    u32 cm; u64 wc = nn ? C.wc[r] : 0;
    next[r] = nn ? (u32)__popc(note16_classify(C, r, nn, wc, cm)) : 0u;
}

__global__ void __launch_bounds__(128)
gather_out16_kernel(const Cols C, const u64* __restrict__ offs, const u32* __restrict__ xoffs,
                    ulonglong2* __restrict__ msgs, const u64 msgs_cap, ulonglong2* __restrict__ units, const u64 units_cap,
                    OutHdr* hdr, const u32* err)
{
    __shared__ unsigned short tab[4][32 * (RA_NOTE_CAP > RA_MSG_CAP ? RA_NOTE_CAP : RA_MSG_CAP)];
    __shared__ u32 s_mask[4][32], s_xb[4][32];
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const u32 tile = blockIdx.x * 4 + warp;
    const u64 total = offs[C.rows];
    const u64 tm = total & 0xffffffffull, tn = total >> 32;
    const u64 tx = xoffs[C.rows];
    const u32 bad = *err;
    const bool fits = tm <= msgs_cap && tn + 2 * tx <= units_cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        hdr->n_msgs = tm; hdr->n_notes = tn; hdr->n_ext = (u32)tx; hdr->status = bad | (fits ? 0u : 0x100u);
    }
    if (bad || !fits) return;
    const u32 r = tile * 32 + lane;
    const bool valid = r < C.rows;
    const u32 v = valid ? C.out_n[r] : 0u;
    if (!__any_sync(0xffffffffu, v != 0)) return;
    const u64 off = offs[valid ? r : C.rows];
    if (v) C.out_n[r] = 0;
    unsigned short* t = tab[warp];
    {
        const u32 nn = v >> 16;
        const u64 on = off >> 32;
        const u64 base = __shfl_sync(0xffffffffu, on, 0);
        const u32 cnt = (u32)(__shfl_sync(0xffffffffu, on + nn, 31) - base);
        // the owner walks its row's notes in order (the WAL_APPEND rule depends on the one before)
        u32 extmask = 0, cmask = 0;
        const u32 xb = valid ? xoffs[r] : 0u;
        if (nn) {
            u64 wc = C.wc[r];
            extmask = note16_classify(C, r, nn, wc, cmask);
            C.wc[r] = wc;
            for (u32 k = 0; k < nn; k++) {
                t[(u32)(on - base) + k] = (unsigned short)((lane << 4) | k);
                if ((extmask >> k) & 1u) {                           // {a, b}, {c, 0} into the extension area
                    const ulonglong2* q = reinterpret_cast<const ulonglong2*>(&C.onote[(size_t)k * C.rows + r]);
                    const u64 idx = xb + (u32)__popc(extmask & ((1u << k) - 1u));
                    units[tn + 2 * idx] = make_ulonglong2(q[0].y, q[1].x);
                    units[tn + 2 * idx + 1] = make_ulonglong2(q[1].y, 0);
                }
            }
        }
        s_mask[warp][lane] = extmask | (cmask << 16);
        s_xb[warp][lane] = xb;
        __syncwarp();
        for (u32 j = lane; j < cnt; j += 32) {                       // one 16-byte unit per note, lane-consecutive
            const u32 ent = t[j], src_lane = ent >> 4, k = ent & 15u;
            const ulonglong2* q = reinterpret_cast<const ulonglong2*>(&C.onote[(size_t)k * C.rows + tile * 32 + src_lane]);
            const ulonglong2 h = q[0];
            const u32 m = s_mask[warp][src_lane];
            u64 w0 = h.x, w1 = h.y;
            if ((m >> k) & 1u) {
                w0 |= 0x80ull << 32;                                  // type' bit 7: extension; slot stays in place
                w1 = s_xb[warp][src_lane] + (u32)__popc(m & 0xffffu & ((1u << k) - 1u));
            } else {
                const u64 n = q[1].x - h.y;                           // b - a < 256 goes where the (zero) slot was
                w0 |= (n << 40) | (((m >> (16 + k)) & 1u) ? (0x40ull << 32) : 0ull);
            }
            units[base + j] = make_ulonglong2(w0, w1);
        }
        __syncwarp();
    }
    {   // RPC records: 4 chunks each (unchanged)
        const u32 nm = v & 0xffffu;
        const u64 om = off & 0xffffffffull;
        const u64 base = __shfl_sync(0xffffffffu, om, 0);
        const u32 cnt = (u32)(__shfl_sync(0xffffffffu, om + nm, 31) - base);
        if (cnt == 0) return;
        for (u32 k = 0; k < nm; k++) t[(u32)(om - base) + k] = (unsigned short)((lane << 4) | k);
        __syncwarp();
        for (u32 c = lane; c < 4 * cnt; c += 32) {
            const u32 ent = t[c >> 2];
            const ulonglong2* src = reinterpret_cast<const ulonglong2*>(&C.omsg[(size_t)(ent & 15u) * C.rows + tile * 32 + (ent >> 4)]);
            msgs[(base << 2) + c] = src[c & 3u];
        }
    }
}

// Step barrier of the peer transport without a collective: every shard release-stores the step's
// epoch into its flag word in every peer's HBM (the words behind mbox_cnt[0], reachable through the
// IPC mappings of the mailboxes) and acquire-spins until all peers' epochs have arrived in its own.
// One warp, one lane per peer.  Stream order makes the step kernels' peer stores happen-before the
// release; the acquire on the other side orders them before that shard's next step.
__global__ void peer_barrier_kernel(const Cols C, const u64 epoch, u32* err)
{
    const u32 k = threadIdx.x;
    if (k >= C.n_shards) return;
    u64* mine = C.mbox_cnt[0] + C.rows;                      // [source shard]
    u64* theirs = C.peer_cnt[0][k] + C.rows;                 // all shards have the same number of rows
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(theirs + C.shard), "l"(epoch) : "memory");
    u64 v = 0;
    for (u32 spins = 0; spins < (1u << 24); spins++) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine + k) : "memory");
        if (v >= epoch) return;
        __nanosleep(64);
    }
    atomicExch(err + 1, 1u);                                 // a peer never arrived: reported by the next call
}

// ------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------
// one host call in flight (ra_engine_submit .. ra_engine_collect); RA_IO_SLOTS of them per engine
#define RA_IO_SLOTS 2
struct IoSlot {
    int busy;
    void* d_ev; size_t d_ev_bytes;            // device copy of the call's events
    OutHdr* hdr;                              // pinned + mapped
    cudaEvent_t h2d_done, done;
    // gather_out_kernel compacts the outputs into the slot's device staging; the DMA to the caller's buffers is
    // enqueued right behind it with PREDICTED sizes (what the previous call produced, plus a margin), so the
    // call still has a single wait; collect tops up with a second copy in the rare step that produced more
    ra_event* user_msgs; ra_note* user_notes; size_t msgs_cap, notes_cap;
    ra_event* d_msgs; size_t d_msgs_cap; ra_note* d_notes; size_t d_notes_cap;
    size_t copied_msgs, copied_notes;         // (copied_notes counts 16-byte units in compact mode)
};

struct ra_engine {
    ra_engine_cfg cfg;
    Cols C;
    cudaStream_t stream; int own_stream;
    cudaStream_t copy_stream;                 // host -> device copies of submitted batches
    cudaEvent_t ev0, ev1;
    int cur;
    u64 step_no, steps;
    u64 bar_epoch;                            // peer transport: barriers passed since the last reset
    int flood_barrier;                        // peer transport: ra_engine_flood ends every step with the device barrier
    void* allocs[96]; int n_allocs;
    IoSlot io[RA_IO_SLOTS]; u32 io_head, io_tail;   // FIFO: submit fills io[io_head % SLOTS], collect drains io_tail
    // The hot kernel computes on 32-bit indexes where it can (ra_narrow::raft_step_kernel, exact for any input: rows
    // that do not fit stall to the 64-bit general kernel) -- unless most rows do not fit, where the 64-bit hot kernel
    // is the faster choice.  narrow_mode: 0 auto (bulk loads decide: ra_engine_load_rows), 1 always narrow
    // (RA_STEP_WIDE=0), 2 never (RA_STEP_WIDE=1).  A performance choice only; results do not depend on it.
    int narrow, narrow_mode;
    int out_pending;                          // the last collect ended in RA_E_CAPACITY: outputs wait in the row slots
    size_t pred_msgs, pred_notes, pred_ext;   // outputs of the last collected call (sizes the next DMA is enqueued with)
    int compact;                              // notes leave as 16-byte units (ra_engine_set_note_format)
    u32 *d_next, *d_xoffs; void* d_scan_tmp2; size_t scan_tmp2_bytes;   // compact stream: per-row extension counts + scan
    size_t last_ext;                          // extension entries of the last collected call
    int loc_dirty;                            // the flood host model may have left host events queued
    u64* d_offs; void* d_scan_tmp; size_t scan_tmp_bytes;
    u32* d_err;                               // [0] sticky ingest error (= Cols::abort), [1] peer barrier timeout
    StallCtx* d_stall; u32* d_stall_cnt;      // d_stall_cnt[2]: alternating per step
    ra_row_state* d_rows; size_t d_rows_cap;
    float last_ms; u32 last_launches;
    u32 general_grid;
    char err[256];
};

static int fail(ra_engine* e, cudaError_t ce, const char* what)
{
    if (e) snprintf(e->err, sizeof e->err, "%s: %s", what, cudaGetErrorString(ce));
    return RA_E_CUDA;
}
#define CK(call) do { cudaError_t ce_ = (call); if (ce_ != cudaSuccess) return fail(e, ce_, #call); } while (0)

template <typename T>
static int dalloc(ra_engine* e, T** p, size_t count)
{
    void* q = nullptr;
    cudaError_t ce = cudaMalloc(&q, count * sizeof(T) ? count * sizeof(T) : 16);
    if (ce != cudaSuccess) return fail(e, ce, "cudaMalloc");
    cudaMemsetAsync(q, 0, count * sizeof(T) ? count * sizeof(T) : 16, e->stream);
    e->allocs[e->n_allocs++] = q;
    *p = (T*)q;
    return RA_OK;
}

static inline u32 nblocks(u64 n, u32 t) { return (u32)((n + t - 1) / t); }

extern "C" const char* ra_engine_strerror(int st)
{
    switch (st) {
    case RA_OK: return "ok";
    case RA_E_INVAL: return "invalid argument";
    case RA_E_NOMEM: return "out of memory";
    case RA_E_CUDA: return "CUDA error (see ra_engine_last_cuda_error)";
    case RA_E_UNGROUPED: return "events of one row are not adjacent in the batch";
    case RA_E_CAPACITY: return "capacity exceeded (RA_LOCAL_CAP per row, or output buffers too small)";
    case RA_E_NODEVICE: return "no CUDA device: the engine has no CPU fallback";
    case RA_E_BUSY: return "a submitted batch has not been collected yet (or both submit slots are in flight)";
    default: return "unknown status";
    }
}

extern "C" const char* ra_engine_last_cuda_error(ra_engine* e) { return e ? e->err : ""; }

extern "C" void ra_engine_destroy(ra_engine* e)
{
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    for (int i = 0; i < e->n_allocs; i++) cudaFree(e->allocs[i]);
    cudaFree(e->d_rows); cudaFree(e->d_scan_tmp); cudaFree(e->d_scan_tmp2);
    for (int i = 0; i < RA_IO_SLOTS; i++) {
        IoSlot& q = e->io[i];
        cudaFree(q.d_ev); cudaFree(q.d_msgs); cudaFree(q.d_notes);
        if (q.hdr) cudaFreeHost(q.hdr);
        if (q.h2d_done) cudaEventDestroy(q.h2d_done);
        if (q.done) cudaEventDestroy(q.done);
    }
    cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->own_stream) cudaStreamDestroy(e->stream);
    free(e);
}

extern "C" int ra_engine_reset_empty(ra_engine* e)
{
    if (!e) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    reset_empty_kernel<<<nblocks(e->C.rows, 256), 256, 0, e->stream>>>(e->C);
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(e->C.counters, 0, RA_N_COUNTERS * sizeof(u64), e->stream));
    CK(cudaMemsetAsync(e->d_stall_cnt, 0, 4 * sizeof(u32), e->stream));
    e->cur = 0; e->step_no = 0; e->steps = 0; e->bar_epoch = 0;
    e->narrow = e->narrow_mode != 2;
    if (e->C.routed) CK(cudaMemsetAsync(e->C.mbox_cnt[0] + e->C.rows, 0, RA_BAR_WORDS * sizeof(u64), e->stream));
    CK(cudaMemsetAsync(e->d_err, 0, 4 * sizeof(u32), e->stream));
    CK(cudaMemsetAsync(e->C.q_used, 0, 4 * sizeof(u32), e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < RA_IO_SLOTS; i++) e->io[i].busy = 0;
    e->io_head = e->io_tail = 0; e->out_pending = 0; e->loc_dirty = 0; e->pred_msgs = e->pred_notes = e->pred_ext = 0; e->last_ext = 0;
    CK(cudaMemsetAsync(e->C.wc, 0, (size_t)e->C.rows * sizeof(u64), e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RA_OK;
}

extern "C" int ra_engine_create(const ra_engine_cfg* cfg, ra_engine** out)
{
    if (!cfg || !out || cfg->n_members < 1 || cfg->n_members > RA_MAX_MEMBERS || cfg->n_groups == 0) return RA_E_INVAL;
    if ((u64)cfg->n_groups * cfg->n_members > 0x7fffffffull) return RA_E_INVAL;
    if (cfg->n_shards > 1 && (!cfg->route_on_device || cfg->shard >= cfg->n_shards || cfg->n_shards > 64)) return RA_E_INVAL;
    if (cfg->note_cap && (cfg->note_cap < RA_NOTE_RESERVE + 2 || cfg->note_cap > RA_NOTE_CAP)) return RA_E_INVAL;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device >= ndev) return RA_E_NODEVICE;
    ra_engine* e = (ra_engine*)calloc(1, sizeof(ra_engine));
    if (!e) return RA_E_NOMEM;
    e->cfg = *cfg;
    { const char* w = getenv("RA_STEP_WIDE"); e->narrow_mode = !(w && *w) ? 0 : (*w == '0' ? 1 : 2); e->narrow = e->narrow_mode != 2; }
    if (e->cfg.max_pipeline_count == 0) e->cfg.max_pipeline_count = 4096;
    if (e->cfg.max_aer_batch == 0) e->cfg.max_aer_batch = 128;
    int rc = RA_OK;
    cudaError_t ce;
    if ((ce = cudaSetDevice(cfg->device)) != cudaSuccess) { rc = fail(e, ce, "cudaSetDevice"); goto bad; }
    if ((ce = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail(e, ce, "cudaStreamCreate"); goto bad; }
    e->own_stream = 1;
    if ((ce = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) { rc = fail(e, ce, "cudaStreamCreate"); goto bad; }
    cudaEventCreate(&e->ev0); cudaEventCreate(&e->ev1);
    for (int i = 0; i < RA_IO_SLOTS; i++) {
        IoSlot& q = e->io[i];
        if ((ce = cudaHostAlloc((void**)&q.hdr, sizeof(OutHdr), cudaHostAllocMapped | cudaHostAllocPortable)) != cudaSuccess) { rc = fail(e, ce, "cudaHostAlloc"); goto bad; }
        memset(q.hdr, 0, sizeof(OutHdr));
        cudaEventCreateWithFlags(&q.h2d_done, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&q.done, cudaEventDisableTiming);
    }
    {
        Cols& C = e->C;
        const size_t R = (size_t)cfg->n_groups * cfg->n_members, M = cfg->n_members;
        C.rows = (u32)R; C.groups = cfg->n_groups; C.members = cfg->n_members;
        C.groups_inv = cfg->n_groups > 1 ? (u32)(0x100000000ull / cfg->n_groups) : 0xFFFFFFFFu;
        C.max_pipeline = e->cfg.max_pipeline_count; C.max_batch = e->cfg.max_aer_batch;
        C.routed = cfg->route_on_device ? 1 : 0; C.pure = cfg->pure ? 1 : 0;
        C.note_cap = cfg->note_cap ? cfg->note_cap : RA_NOTE_CAP;
        C.n_shards = cfg->n_shards > 1 ? cfg->n_shards : 1; C.shard = cfg->n_shards > 1 ? cfg->shard : 0;
        C.outbox = nullptr; C.out_cnt = nullptr; C.out_cap = 0;
        C.peer_mode = 0;
        for (int b = 0; b < 2; b++) for (int k = 0; k < 8; k++) { C.peer_mbox[b][k] = nullptr; C.peer_cnt[b][k] = nullptr; }
#define DA(p, n) if ((rc = dalloc(e, &(p), (n))) != RA_OK) goto bad
        DA(C.tc, R); DA(C.lg, R); DA(C.lw, R); DA(C.ap, R); DA(C.sn, R); DA(C.tk, R); DA(C.fm, R);
        DA(C.cd, 2 * R); DA(C.pnm, M * R); DA(C.pcs, M * R); DA(C.run, RA_MAX_RUNS * R); DA(C.lrs, R);
        DA(C.qi, R); DA(C.qa, R); DA(C.pqi, M * R); DA(C.q_used, 4); DA(C.wc, R); DA(C.wf, R);
        C.tiles = (u32)((R + RT - 1) / RT);
        const size_t PW = (size_t)C.tiles * 4 * RT;             // 16-byte words per tiled plane
        DA(C.loc, (size_t)RA_LOCAL_CAP * PW); DA(C.loc_n, R);
        DA(C.onote, (size_t)RA_NOTE_CAP * R); DA(C.out_n, R + 1); DA(C.counters, RA_N_COUNTERS);   // out_n[R] stays 0: the scan's total
        if (C.routed) {
            // + RA_BAR_WORDS: the peer transport's step barrier flags live behind the counts of buffer 0,
            // so they are covered by the IPC mapping the peers already have
            for (int b = 0; b < 2; b++) { DA(C.mbox[b], M * RA_MBOX_DEPTH * PW); DA(C.mbox_cnt[b], R + RA_BAR_WORDS); }
            DA(C.omsg, (size_t)RA_MSG_CAP * (C.pure ? R : 1));
        } else {
            C.mbox[0] = C.mbox[1] = nullptr; C.mbox_cnt[0] = C.mbox_cnt[1] = nullptr;
            DA(C.omsg, (size_t)RA_MSG_CAP * R);
        }
        DA(e->d_offs, R + 1); DA(e->d_err, 4); DA(e->d_next, R + 1); DA(e->d_xoffs, R + 1);
        DA(e->d_stall, R); DA(e->d_stall_cnt, 4);
#undef DA
        C.abort = e->d_err;
        e->scan_tmp_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, e->scan_tmp_bytes, PackedIt(C.out_n, PackCounts()), e->d_offs, (int)(R + 1), e->stream);
        if ((ce = cudaMalloc(&e->d_scan_tmp, e->scan_tmp_bytes ? e->scan_tmp_bytes : 16)) != cudaSuccess) { rc = fail(e, ce, "cudaMalloc scan"); goto bad; }
        e->scan_tmp2_bytes = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, e->scan_tmp2_bytes, e->d_next, e->d_xoffs, (int)(R + 1), e->stream);
        if ((ce = cudaMalloc(&e->d_scan_tmp2, e->scan_tmp2_bytes ? e->scan_tmp2_bytes : 16)) != cudaSuccess) { rc = fail(e, ce, "cudaMalloc scan"); goto bad; }
    }
#define SMEM_ATTR_NS(NS, NARROW, MEMB, TRN, FLT) \
    if ((ce = cudaFuncSetAttribute(NS::raft_step_kernel<MK_MM(MEMB, TRN), FLT>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)sizeof(StepSmem<MK_MM(MEMB, TRN), NARROW>))) != cudaSuccess) { rc = fail(e, ce, "cudaFuncSetAttribute"); goto bad; }
#define SMEM_ATTR(MEMB, TRN, FLT) SMEM_ATTR_NS(ra_wide, false, MEMB, TRN, FLT)
#ifndef RA_NO_NARROW
    SMEM_ATTR_NS(ra_narrow, true, 5, TR_LOCAL, false) SMEM_ATTR_NS(ra_narrow, true, 5, TR_PEER, false) SMEM_ATTR_NS(ra_narrow, true, 5, TR_HOST, false)
    SMEM_ATTR_NS(ra_narrow, true, 3, TR_LOCAL, false) SMEM_ATTR_NS(ra_narrow, true, 7, TR_LOCAL, false)
#endif
    SMEM_ATTR(0, TR_RUNTIME, true) SMEM_ATTR(0, TR_RUNTIME, false)
    SMEM_ATTR(5, TR_LOCAL, false) SMEM_ATTR(5, TR_PEER, false) SMEM_ATTR(5, TR_BUCKET, false) SMEM_ATTR(5, TR_HOST, false)
    SMEM_ATTR(3, TR_LOCAL, false) SMEM_ATTR(7, TR_LOCAL, false) SMEM_ATTR(5, TR_LOCAL, true) SMEM_ATTR(7, TR_LOCAL, true)
#undef SMEM_ATTR
#undef SMEM_ATTR_NS
    {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        e->general_grid = (u32)sms * 2;
    }
    if ((rc = ra_engine_reset_empty(e)) != RA_OK) goto bad;
    *out = e;
    return RA_OK;
bad:
    ra_engine_destroy(e);
    return rc;
}

template <typename T>
static int ensure(ra_engine* e, T** p, size_t* cap, size_t need)
{
    if (*cap >= need && *p) return RA_OK;
    if (*p) cudaFree(*p);
    size_t nc = need < 1024 ? 1024 : need + need / 4;
    void* q = nullptr;
    cudaError_t ce = cudaMalloc(&q, nc * sizeof(T));
    if (ce != cudaSuccess) { *p = nullptr; *cap = 0; return fail(e, ce, "cudaMalloc staging"); }
    *p = (T*)q; *cap = nc;
    return RA_OK;
}

extern "C" int ra_engine_load_rows(ra_engine* e, const ra_row_state* rows, size_t n)
{
    if (!e || (!rows && n)) return RA_E_INVAL;
    if (n == 0) return RA_OK;
    for (size_t i = 0; i < n; i++)
        if (rows[i].row >= e->C.rows || rows[i].n_members != e->C.members || !ra_row_state_valid(&rows[i])) return RA_E_INVAL;
    if (e->narrow_mode == 0 && n * 2 >= e->C.rows) {            // a bulk load: which hot kernel suits this engine?
        size_t wide = 0;
        for (size_t i = 0; i < n; i++) wide += row_state_is_wide(rows[i], e->C.members) ? 1 : 0;
        e->narrow = wide * 2 < n;
    }
    CK(cudaSetDevice(e->cfg.device));
    int rc = ensure(e, &e->d_rows, &e->d_rows_cap, n); if (rc) return rc;
    CK(cudaMemcpyAsync(e->d_rows, rows, n * sizeof(ra_row_state), cudaMemcpyHostToDevice, e->stream));
    load_rows_kernel<<<nblocks(n, 128), 128, 0, e->stream>>>(e->C, e->d_rows, (u32)n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    return RA_OK;
}

extern "C" int ra_engine_read_rows(ra_engine* e, ra_row_state* rows, size_t n)
{
    if (!e || (!rows && n)) return RA_E_INVAL;
    if (n == 0) return RA_OK;
    for (size_t i = 0; i < n; i++) if (rows[i].row >= e->C.rows) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    int rc = ensure(e, &e->d_rows, &e->d_rows_cap, n); if (rc) return rc;
    CK(cudaMemcpyAsync(e->d_rows, rows, n * sizeof(ra_row_state), cudaMemcpyHostToDevice, e->stream));
    read_rows_kernel<<<nblocks(n, 128), 128, 0, e->stream>>>(e->C, e->d_rows, (u32)n);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(rows, e->d_rows, n * sizeof(ra_row_state), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RA_OK;
}

static int query_io(ra_engine* e, ra_query_state* q, size_t n, bool load)
{
    if (!e || (!q && n)) return RA_E_INVAL;
    if (n == 0) return RA_OK;
    for (size_t i = 0; i < n; i++) if (q[i].row >= e->C.rows) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    ra_query_state* d = nullptr;
    CK(cudaMalloc(&d, n * sizeof(ra_query_state)));
    cudaError_t ce = cudaMemcpyAsync(d, q, n * sizeof(ra_query_state), cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) {
        if (load) load_query_kernel<<<nblocks(n, 128), 128, 0, e->stream>>>(e->C, d, (u32)n);
        else {
            read_query_kernel<<<nblocks(n, 128), 128, 0, e->stream>>>(e->C, d, (u32)n);
            ce = cudaMemcpyAsync(q, d, n * sizeof(ra_query_state), cudaMemcpyDeviceToHost, e->stream);
        }
    }
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    cudaFree(d);
    return ce == cudaSuccess ? RA_OK : fail(e, ce, "query state");
}
extern "C" int ra_engine_load_query_state(ra_engine* e, const ra_query_state* q, size_t n)
{ return query_io(e, const_cast<ra_query_state*>(q), n, true); }
extern "C" int ra_engine_read_query_state(ra_engine* e, ra_query_state* q, size_t n)
{ return query_io(e, q, n, false); }

// launch with programmatic stream serialization (see grid_dep_wait): CTA_T threads, `smem` bytes of dynamic shared memory
template <typename... P, typename... A>
static cudaError_t launch_chained(void (*k)(P...), u32 grid, size_t smem, cudaStream_t s, A... a)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(CTA_T); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k, a...);
}

static int launch_step(ra_engine* e, const FloodArgs& F)
{
    if (e->C.n_shards > 1) {
        if (!e->C.peer_mode) {
            if (!e->C.outbox) return RA_E_INVAL;                // ra_engine_set_outbox / peer_set first
            cudaError_t c0 = cudaMemsetAsync(e->C.out_cnt, 0, e->C.n_shards * sizeof(u32), e->stream);
            if (c0 != cudaSuccess) return fail(e, c0, "cudaMemsetAsync out_cnt");
        }
    }
#ifdef RA_INTERLEAVE
    const u32 grid = (((e->C.tiles + WARPS - 1) / WARPS + e->C.members - 1) / e->C.members) * e->C.members;
#else
    const u32 grid = (e->C.tiles + WARPS - 1) / WARPS;
#endif
    u32* cnt = e->d_stall_cnt + (e->steps & 1), *cnt_next = e->d_stall_cnt + ((e->steps + 1) & 1);
    // one specialisation of the hot kernel per (member count, transport): see MK_MM
    const int tr = !e->C.routed ? TR_HOST : (e->C.n_shards > 1 ? (e->C.peer_mode ? TR_PEER : TR_BUCKET) : TR_LOCAL);
    cudaError_t ce = cudaSuccess;
#define LAUNCH_NS(NS, NARROW, MEMB, TRN, FLT) ce = launch_chained(NS::raft_step_kernel<MK_MM(MEMB, TRN), FLT>, grid, \
        sizeof(StepSmem<MK_MM(MEMB, TRN), NARROW>), e->stream, e->C, e->cur, F, e->d_stall, cnt, cnt_next)
#define LAUNCH(MEMB, TRN, FLT) LAUNCH_NS(ra_wide, false, MEMB, TRN, FLT)
#ifndef RA_NO_NARROW
    // 32-bit index arithmetic for the specialisations that carry the load (exact: rows or records that do not fit
    // stall to the 64-bit general kernel); RA_STEP_WIDE=1 in the environment keeps the 64-bit hot kernel
#define LAUNCH_N(MEMB, TRN, FLT) do { if (e->narrow) LAUNCH_NS(ra_narrow, true, MEMB, TRN, FLT); else LAUNCH_NS(ra_wide, false, MEMB, TRN, FLT); } while (0)
#else
#define LAUNCH_N(MEMB, TRN, FLT) LAUNCH_NS(ra_wide, false, MEMB, TRN, FLT)
#endif
    const bool faults = (F.drop | F.withhold | F.part) != 0;     // fault injection: its own specialisations
    if (faults) {
        if (e->C.members == 5 && tr == TR_LOCAL) LAUNCH(5, TR_LOCAL, true);
        else if (e->C.members == 7 && tr == TR_LOCAL) LAUNCH(7, TR_LOCAL, true);
        else LAUNCH(0, TR_RUNTIME, true);
    } else if (e->C.members == 5) {
        switch (tr) {
        case TR_LOCAL:  LAUNCH_N(5, TR_LOCAL, false); break;
        case TR_PEER:   LAUNCH_N(5, TR_PEER, false); break;
        case TR_BUCKET: LAUNCH(5, TR_BUCKET, false); break;
        default:        LAUNCH_N(5, TR_HOST, false); break;
        }
    } else if (e->C.members == 3 && tr == TR_LOCAL) {
        LAUNCH_N(3, TR_LOCAL, false);
    } else if (e->C.members == 7 && tr == TR_LOCAL) {
        LAUNCH_N(7, TR_LOCAL, false);
    } else {
        LAUNCH(0, TR_RUNTIME, false);
    }
#undef LAUNCH
#undef LAUNCH_N
#undef LAUNCH_NS
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ce, "raft_step_kernel");
    ce = launch_chained(raft_general_kernel, e->general_grid, 0, e->stream, e->C, e->cur, F,
                        (const StallCtx*)e->d_stall, (const u32*)cnt);
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ce, "raft_general_kernel");
    if (e->C.routed) e->cur ^= 1;
    e->steps++;
    return RA_OK;
}

// ---- one batch through the engine: submit (everything enqueued, nothing waited for) .. collect ---------
// stream order of one call:   [copy stream] H2D events  ->  [engine stream] ingest -> raft_step -> raft_general
//   -> scan of the per-row output counts -> gather_out (writes records, notes and the totals into HOST memory)
// There is no synchronisation inside a call and no device->host copy issued by the host: the one wait is
// ra_engine_collect's on the call's `done` event.
static bool host_ptr_mapped(const void* p, void** dev)
{
    cudaPointerAttributes a;
    if (!p || cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost || !a.devicePointer) return false;
    *dev = a.devicePointer;
    return true;
}

static int enqueue_gather(ra_engine* e, IoSlot& q)
{
    int rc;
    if ((rc = ensure(e, &q.d_msgs, &q.d_msgs_cap, q.msgs_cap ? q.msgs_cap : 1))) return rc;
    if ((rc = ensure(e, &q.d_notes, &q.d_notes_cap, q.notes_cap ? q.notes_cap : 1))) return rc;
    void* dh = nullptr;
    host_ptr_mapped(q.hdr, &dh);
    const u32 R = e->C.rows;
    CK(cub::DeviceScan::ExclusiveSum(e->d_scan_tmp, e->scan_tmp_bytes, PackedIt(e->C.out_n, PackCounts()), e->d_offs,
                                     (int)(R + 1), e->stream));
    if (e->compact) {
        note_ext_count_kernel<<<nblocks((u64)R + 1, 256), 256, 0, e->stream>>>(e->C, e->d_next);
        CK(cub::DeviceScan::ExclusiveSum(e->d_scan_tmp2, e->scan_tmp2_bytes, e->d_next, e->d_xoffs, (int)(R + 1), e->stream));
        gather_out16_kernel<<<nblocks(e->C.tiles, 4), 128, 0, e->stream>>>(
            e->C, e->d_offs, e->d_xoffs, (ulonglong2*)q.d_msgs, (u64)q.msgs_cap, (ulonglong2*)q.d_notes, (u64)q.notes_cap,
            (OutHdr*)dh, e->d_err);
    } else
    gather_out_kernel<<<nblocks(e->C.tiles, 4), 128, 0, e->stream>>>(
        e->C, e->d_offs, (ulonglong2*)q.d_msgs, (u64)q.msgs_cap, (ulonglong2*)q.d_notes, (u64)q.notes_cap, (OutHdr*)dh, e->d_err);
    CK(cudaGetLastError());
    // the outputs follow by DMA, sized by what the previous call produced (+ 1/16): steady streams of batches
    // produce steady amounts of output.  (A pinned destination -- ra_engine_alloc_host / ra_engine_register_host --
    // makes it a true asynchronous copy; a pageable one is staged by the driver.)
    const size_t unit = e->compact ? 16 : sizeof(ra_note);
    const size_t pn = e->compact ? e->pred_notes + 2 * e->pred_ext : e->pred_notes;   // compact: units, extensions behind
    q.copied_msgs = e->pred_msgs + e->pred_msgs / 16 + (e->pred_msgs ? 16 : 0);
    q.copied_notes = pn + pn / 16 + (pn ? 64 : 0);
    if (q.copied_msgs > q.msgs_cap) q.copied_msgs = q.msgs_cap;
    if (q.copied_notes > q.notes_cap) q.copied_notes = q.notes_cap;
    if (q.copied_msgs) CK(cudaMemcpyAsync(q.user_msgs, q.d_msgs, q.copied_msgs * sizeof(ra_event), cudaMemcpyDeviceToHost, e->stream));
    if (q.copied_notes) CK(cudaMemcpyAsync(q.user_notes, q.d_notes, q.copied_notes * unit, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaEventRecord(q.done, e->stream));
    return RA_OK;
}

// a batch handed over in pieces (one per producer thread): copied back to back into one device array
struct EvSeg { const void* p; size_t n; };

static int submit_impl(ra_engine* e, const EvSeg* segs, size_t n_segs, bool host32,
                       ra_event* msgs, size_t msgs_cap, ra_note* notes, size_t notes_cap)
{
    if (!e || (!segs && n_segs) || (!msgs && msgs_cap) || (!notes && notes_cap)) return RA_E_INVAL;
    size_t n_ev = 0;
    for (size_t k = 0; k < n_segs; k++) { if (!segs[k].p && segs[k].n) return RA_E_INVAL; n_ev += segs[k].n; }
    if (n_ev > 0x7fffffffull) return RA_E_INVAL;
    if (e->out_pending) return RA_E_CAPACITY;                     // ra_engine_fetch_output first
    IoSlot& q = e->io[e->io_head % RA_IO_SLOTS];
    if (e->io_head - e->io_tail >= RA_IO_SLOTS || q.busy) return RA_E_BUSY;
    CK(cudaSetDevice(e->cfg.device));
    const u32 R = e->C.rows;
    const size_t rec = host32 ? sizeof(ra_host_event) : sizeof(ra_event);
    const size_t bytes = n_ev * rec;
    if (n_ev) {
        if (q.d_ev_bytes < bytes) {
            cudaFree(q.d_ev); q.d_ev = nullptr; q.d_ev_bytes = 0;
            const size_t nb = bytes + bytes / 4 + 4096;
            CK(cudaMalloc(&q.d_ev, nb));
            q.d_ev_bytes = nb;
        }
        // a pinned source makes this a true asynchronous DMA; a pageable one is staged by the driver
        size_t off = 0;
        for (size_t k = 0; k < n_segs; k++) {
            if (!segs[k].n) continue;
            CK(cudaMemcpyAsync((char*)q.d_ev + off, segs[k].p, segs[k].n * rec, cudaMemcpyHostToDevice, e->copy_stream));
            off += segs[k].n * rec;
        }
        CK(cudaEventRecord(q.h2d_done, e->copy_stream));
        CK(cudaStreamWaitEvent(e->stream, q.h2d_done, 0));
    }
    if (e->loc_dirty) {     // a step after flood() must not see the flood host model's queued host events
        clear_loc_kernel<<<nblocks(R, 256), 256, 0, e->stream>>>(e->C);
        e->loc_dirty = 0;
    }
    if (n_ev) {
        if (host32) ingest_host_kernel<<<nblocks(n_ev, 256), 256, 0, e->stream>>>(
                        e->C, reinterpret_cast<const ra_host_event*>(q.d_ev), (u32)n_ev, e->d_err, e->d_err);
        else ingest_kernel<<<nblocks(n_ev, 256), 256, 0, e->stream>>>(e->C, reinterpret_cast<const ra_event*>(q.d_ev),
                                                                        (u32)n_ev, e->d_err, e->d_err);
        CK(cudaGetLastError());
    }
    FloodArgs F; memset(&F, 0, sizeof F);
    int rc;
    if ((rc = launch_step(e, F))) return rc;
    q.user_msgs = msgs; q.user_notes = notes; q.msgs_cap = msgs_cap; q.notes_cap = notes_cap;
    if ((rc = enqueue_gather(e, q))) return rc;
    q.busy = 1;
    e->io_head++;
    return RA_OK;
}

static int finish_slot(ra_engine* e, IoSlot& q, size_t* n_msgs, size_t* n_notes, bool was_step)
{
    CK(cudaEventSynchronize(q.done));
    const OutHdr h = *q.hdr;
    if (n_msgs) *n_msgs = (size_t)h.n_msgs;
    if (n_notes) *n_notes = (size_t)h.n_notes;
    const u32 bad = h.status & 0xffu;
    if (bad) {
        // the batch was rejected by ingest: the step kernels of this call (and of any call submitted behind it)
        // did nothing.  Undo this call's buffer flip; once the last such call is collected, clean up.
        if (was_step) { if (e->C.routed) e->cur ^= 1; e->steps--; }
        if (e->io_head == e->io_tail) {
            CK(cudaStreamSynchronize(e->stream));
            clear_loc_kernel<<<nblocks(e->C.rows, 256), 256, 0, e->stream>>>(e->C);
            CK(cudaMemsetAsync(e->d_err, 0, sizeof(u32), e->stream));
            CK(cudaStreamSynchronize(e->stream));
        }
        return bad == 1 ? RA_E_UNGROUPED : (bad == 2 ? RA_E_CAPACITY : RA_E_INVAL);
    }
    if (h.status & 0x100u) { e->out_pending = 1; return RA_E_CAPACITY; }   // nothing lost: ra_engine_fetch_output
    // top up what the predicted-size copies did not cover (first call, a burst)
    bool more = false;
    if (h.n_msgs > q.copied_msgs) {
        CK(cudaMemcpyAsync(q.user_msgs + q.copied_msgs, q.d_msgs + q.copied_msgs, (size_t)(h.n_msgs - q.copied_msgs) * sizeof(ra_event),
                           cudaMemcpyDeviceToHost, e->copy_stream));
        more = true;
    }
    {
        const size_t unit = e->compact ? 16 : sizeof(ra_note);
        const size_t have = e->compact ? (size_t)h.n_notes + 2 * (size_t)h.n_ext : (size_t)h.n_notes;
        if (have > q.copied_notes) {
            CK(cudaMemcpyAsync((char*)q.user_notes + q.copied_notes * unit, (const char*)q.d_notes + q.copied_notes * unit,
                               (have - q.copied_notes) * unit, cudaMemcpyDeviceToHost, e->copy_stream));
            more = true;
        }
    }
    if (more) CK(cudaStreamSynchronize(e->copy_stream));
    e->pred_msgs = (size_t)h.n_msgs; e->pred_notes = (size_t)h.n_notes; e->pred_ext = (size_t)h.n_ext; e->last_ext = (size_t)h.n_ext;
    return RA_OK;
}

extern "C" int ra_engine_collect(ra_engine* e, size_t* n_msgs, size_t* n_notes)
{
    if (!e) return RA_E_INVAL;
    if (e->io_head == e->io_tail) return RA_E_INVAL;              // nothing submitted
    CK(cudaSetDevice(e->cfg.device));
    IoSlot& q = e->io[e->io_tail % RA_IO_SLOTS];
    e->io_tail++;
    q.busy = 0;
    return finish_slot(e, q, n_msgs, n_notes, true);
}

extern "C" int ra_engine_submit(ra_engine* e, const ra_event* ev, size_t n_ev,
                                ra_event* msgs, size_t msgs_cap, ra_note* notes, size_t notes_cap)
{ if (!ev && n_ev) return RA_E_INVAL; EvSeg s = { ev, n_ev }; return submit_impl(e, &s, 1, false, msgs, msgs_cap, notes, notes_cap); }

extern "C" int ra_engine_submit_host(ra_engine* e, const ra_host_event* ev, size_t n_ev,
                                     ra_event* msgs, size_t msgs_cap, ra_note* notes, size_t notes_cap)
{ if (!ev && n_ev) return RA_E_INVAL; EvSeg s = { ev, n_ev }; return submit_impl(e, &s, 1, true, msgs, msgs_cap, notes, notes_cap); }

extern "C" int ra_engine_submit_host_segs(ra_engine* e, const ra_host_event_seg* segs, size_t n_segs,
                                          ra_event* msgs, size_t msgs_cap, ra_note* notes, size_t notes_cap)
{
    if (n_segs > 256 || (!segs && n_segs)) return RA_E_INVAL;
    EvSeg s[256];
    for (size_t k = 0; k < n_segs; k++) { s[k].p = segs[k].ev; s[k].n = segs[k].n; }
    return submit_impl(e, s, n_segs, true, msgs, msgs_cap, notes, notes_cap);
}

// outputs that did not fit the buffers of the call that produced them (RA_E_CAPACITY): how many, and again
extern "C" int ra_engine_pending_output(ra_engine* e, size_t* n_msgs, size_t* n_notes)
{
    if (!e) return RA_E_INVAL;
    const IoSlot& q = e->io[(e->io_tail + RA_IO_SLOTS - 1) % RA_IO_SLOTS];
    if (n_msgs) *n_msgs = e->out_pending ? (size_t)q.hdr->n_msgs : 0;
    if (n_notes) *n_notes = e->out_pending ? (size_t)q.hdr->n_notes : 0;
    return RA_OK;
}

extern "C" int ra_engine_fetch_output(ra_engine* e, ra_event* msgs, size_t msgs_cap, size_t* n_msgs,
                                      ra_note* notes, size_t notes_cap, size_t* n_notes)
{
    if (!e || (!msgs && msgs_cap) || (!notes && notes_cap)) return RA_E_INVAL;
    if (!e->out_pending) { if (n_msgs) *n_msgs = 0; if (n_notes) *n_notes = 0; return RA_OK; }
    if (e->io_head != e->io_tail) return RA_E_BUSY;
    CK(cudaSetDevice(e->cfg.device));
    IoSlot& q = e->io[(e->io_tail + RA_IO_SLOTS - 1) % RA_IO_SLOTS];
    q.user_msgs = msgs; q.user_notes = notes; q.msgs_cap = msgs_cap; q.notes_cap = notes_cap;
    int rc = enqueue_gather(e, q);
    if (rc) return rc;
    e->out_pending = 0;
    return finish_slot(e, q, n_msgs, n_notes, false);
}

static int step_impl(ra_engine* e, const void* ev, size_t n_ev, bool host32,
                     ra_event* msgs, size_t msgs_cap, size_t* n_msgs,
                     ra_note* notes, size_t notes_cap, size_t* n_notes)
{
    if (e && e->io_head != e->io_tail) return RA_E_BUSY;          // collect what was submitted first
    if (!ev && n_ev) return RA_E_INVAL;
    EvSeg sg = { ev, n_ev };
    int rc = submit_impl(e, &sg, 1, host32, msgs, msgs_cap, notes, notes_cap);
    if (rc) return rc;
    return ra_engine_collect(e, n_msgs, n_notes);
}

extern "C" int ra_engine_step(ra_engine* e, const ra_event* ev, size_t n_ev,
                              ra_event* msgs, size_t msgs_cap, size_t* n_msgs,
                              ra_note*  notes, size_t notes_cap, size_t* n_notes)
{ return step_impl(e, ev, n_ev, false, msgs, msgs_cap, n_msgs, notes, notes_cap, n_notes); }

extern "C" int ra_engine_step_host(ra_engine* e, const ra_host_event* ev, size_t n_ev,
                                   ra_event* msgs, size_t msgs_cap, size_t* n_msgs,
                                   ra_note* notes, size_t notes_cap, size_t* n_notes)
{ return step_impl(e, ev, n_ev, true, msgs, msgs_cap, n_msgs, notes, notes_cap, n_notes); }

// notes as 16-byte units (include/ra_engine.h: ra_note16); switch only while no call is in flight
extern "C" int ra_engine_set_note_format(ra_engine* e, int compact)
{
    if (!e) return RA_E_INVAL;
    if (e->io_head != e->io_tail || e->out_pending) return RA_E_BUSY;
    CK(cudaSetDevice(e->cfg.device));
    e->compact = compact ? 1 : 0;
    e->pred_notes = e->pred_ext = 0;
    CK(cudaMemsetAsync(e->C.wc, 0, (size_t)e->C.rows * sizeof(u64), e->stream));   // the decoder starts from zero too
    CK(cudaStreamSynchronize(e->stream));
    return RA_OK;
}
extern "C" size_t ra_engine_last_ext_count(ra_engine* e) { return e ? e->last_ext : 0; }

// caller-owned host buffers (a NIF's resource binaries ...) pinned and mapped once, so that batches built in
// them are copied by DMA and outputs are written into them directly
extern "C" int ra_engine_register_host(void* p, size_t bytes)
{
    if (!p || !bytes) return RA_E_INVAL;
    return cudaHostRegister(p, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable) == cudaSuccess ? RA_OK : RA_E_CUDA;
}
extern "C" int ra_engine_unregister_host(void* p)
{
    if (!p) return RA_E_INVAL;
    return cudaHostUnregister(p) == cudaSuccess ? RA_OK : RA_E_CUDA;
}

extern "C" int ra_engine_flood(ra_engine* e, uint32_t n_steps, uint32_t cmds_per_step,
                               uint32_t election_permille, uint64_t seed)
{ return ra_engine_flood_faults(e, n_steps, cmds_per_step, election_permille, seed, nullptr); }

extern "C" int ra_engine_flood_faults(ra_engine* e, uint32_t n_steps, uint32_t cmds_per_step,
                                      uint32_t election_permille, uint64_t seed, const ra_flood_faults* ff)
{
    if (!e || !e->C.routed) return RA_E_INVAL;
    if (ff && ff->partition_permille && !ff->partition_steps) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaEventRecord(e->ev0, e->stream));
    for (u32 t = 0; t < n_steps; t++) {
        FloodArgs F; memset(&F, 0, sizeof F);
        F.on = 1; F.cmds = cmds_per_step; F.permille = election_permille;
        if (ff) { F.drop = ff->drop_permille; F.withhold = ff->withhold_permille; F.part = ff->partition_permille; F.part_len = ff->partition_steps; }
        F.seed = seed; F.step = e->step_no + t;
        int rc = launch_step(e, F);
        if (rc) return rc;
        if (e->flood_barrier && e->C.peer_mode) {               // lock step with the other shards, no host in the loop
            e->bar_epoch++;
            peer_barrier_kernel<<<1, 32, 0, e->stream>>>(e->C, e->bar_epoch, e->d_err);
        }
    }
    CK(cudaEventRecord(e->ev1, e->stream));
    e->step_no += n_steps;
    e->loc_dirty = 1;
    e->last_launches = 2 * n_steps;
    return RA_OK;
}

extern "C" int ra_engine_stall_histogram(ra_engine* e, uint64_t* out128)
{
    if (!e || !out128) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpyAsync(out128, e->C.counters + 8, 128 * sizeof(u64), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RA_OK;
}

#ifdef RA_WARP_TIMELINE
// Measurement build only: copies the warp records of the hot-kernel launches since the last clear (48 bytes each,
// struct WarpTimeline; a warp that had no work writes none) for the first min(tiles, cap) tiles into out, then
// clears them when `clear` is set.  *n = the number of records copied.  Not part of include/ra_engine.h.
extern "C" int ra_debug_warp_timeline(ra_engine* e, void* out, size_t cap, size_t* n, int clear)
{
    if (!e || !n) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    size_t k = e->C.tiles < RA_WTL_CAP ? e->C.tiles : RA_WTL_CAP;
    if (k > cap) k = cap;
    if (out && k) CK(cudaMemcpyFromSymbol(out, g_wtl, k * sizeof(WarpTimeline)));
    if (clear) {
        void* p = nullptr;
        CK(cudaGetSymbolAddress(&p, g_wtl));
        CK(cudaMemset(p, 0, sizeof(WarpTimeline) * RA_WTL_CAP));
    }
    CK(cudaDeviceSynchronize());
    *n = k;
    return RA_OK;
}
#endif

extern "C" int ra_engine_set_stream(ra_engine* e, void* cuda_stream)
{
    if (!e) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    if (e->own_stream) cudaStreamDestroy(e->stream);
    e->stream = (cudaStream_t)cuda_stream;
    e->own_stream = 0;
    return RA_OK;
}

extern "C" int ra_engine_set_outbox(ra_engine* e, void* outbox, uint32_t* counts, uint32_t cap)
{
    if (!e || e->C.n_shards < 2 || !outbox || !counts || !cap) return RA_E_INVAL;
    e->C.outbox = (ra_event*)outbox; e->C.out_cnt = counts; e->C.out_cap = cap;
    return RA_OK;
}

extern "C" int ra_engine_deliver(ra_engine* e, const void* inbox, const uint32_t* counts, uint32_t cap)
{
    if (!e || e->C.n_shards < 2 || !inbox || !counts || !cap) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    // e->cur is the buffer the next step reads: the one the last step's senders wrote into
    dim3 grid(nblocks(cap, 256) < 512 ? nblocks(cap, 256) : 512, e->C.n_shards);
    deliver_kernel<<<grid, 256, 0, e->stream>>>(e->C, e->cur, (const ra_event*)inbox, counts, cap);
    CK(cudaGetLastError());
    return RA_OK;
}

extern "C" int ra_engine_peer_get(ra_engine* e, ra_peer_ptrs* out)
{
    if (!e || !out || !e->C.routed) return RA_E_INVAL;
    for (int b = 0; b < 2; b++) { out->mbox[b] = e->C.mbox[b]; out->mbox_cnt[b] = e->C.mbox_cnt[b]; }
    return RA_OK;
}

extern "C" int ra_engine_peer_set(ra_engine* e, uint32_t shard, const ra_peer_ptrs* p)
{
    if (!e || !p || e->C.n_shards < 2 || e->C.n_shards > 8 || shard >= e->C.n_shards) return RA_E_INVAL;
    Cols& C = e->C;
    for (int b = 0; b < 2; b++) { C.peer_mbox[b][shard] = (ulonglong2*)p->mbox[b]; C.peer_cnt[b][shard] = (u64*)p->mbox_cnt[b]; }
    for (int b = 0; b < 2; b++) { C.peer_mbox[b][C.shard] = C.mbox[b]; C.peer_cnt[b][C.shard] = C.mbox_cnt[b]; }
    bool all = true;
    for (u32 k = 0; k < C.n_shards; k++) all = all && C.peer_mbox[0][k] && C.peer_mbox[1][k] && C.peer_cnt[0][k] && C.peer_cnt[1][k];
    C.peer_mode = all ? 1 : 0;
    return RA_OK;
}

extern "C" int ra_engine_peer_barrier(ra_engine* e)
{
    if (!e || !e->C.peer_mode) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    e->bar_epoch++;
    peer_barrier_kernel<<<1, 32, 0, e->stream>>>(e->C, e->bar_epoch, e->d_err);
    CK(cudaGetLastError());
    return RA_OK;
}

extern "C" int ra_engine_set_flood_barrier(ra_engine* e, int on)
{
    if (!e) return RA_E_INVAL;
    e->flood_barrier = on ? 1 : 0;
    return RA_OK;
}

extern "C" int ra_engine_ipc_export(ra_engine* e, ra_ipc_handles* out)
{
    if (!e || !out || !e->C.routed) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->h[0], e->C.mbox[0]));
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->h[1], e->C.mbox[1]));
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->h[2], e->C.mbox_cnt[0]));
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)out->h[3], e->C.mbox_cnt[1]));
    return RA_OK;
}

extern "C" int ra_engine_ipc_import(ra_engine* e, uint32_t shard, const ra_ipc_handles* h)
{
    if (!e || !h) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    ra_peer_ptrs p;
    void* q[4];
    for (int i = 0; i < 4; i++) {
        cudaIpcMemHandle_t hh; memcpy(&hh, h->h[i], sizeof hh);
        CK(cudaIpcOpenMemHandle(&q[i], hh, cudaIpcMemLazyEnablePeerAccess));
    }
    p.mbox[0] = q[0]; p.mbox[1] = q[1]; p.mbox_cnt[0] = q[2]; p.mbox_cnt[1] = q[3];
    return ra_engine_peer_set(e, shard, &p);
}

extern "C" int ra_engine_get_cfg(ra_engine* e, ra_engine_cfg* out)
{
    if (!e || !out) return RA_E_INVAL;
    *out = e->cfg;
    return RA_OK;
}

extern "C" int ra_engine_sync(ra_engine* e)
{
    if (!e) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    if (e->bar_epoch) {                                       // did a peer barrier give up waiting?
        u32 h = 0;
        CK(cudaMemcpyAsync(&h, e->d_err + 1, sizeof h, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        if (h) { snprintf(e->err, sizeof e->err, "peer barrier timed out (epoch %llu)", (unsigned long long)e->bar_epoch); return RA_E_CUDA; }
    }
    return RA_OK;
}

extern "C" int ra_engine_last_kernel_ms(ra_engine* e, float* ms, uint32_t* launches)
{
    if (!e) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaEventSynchronize(e->ev1));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, e->ev0, e->ev1));
    if (ms) *ms = t;
    if (launches) *launches = e->last_launches;
    return RA_OK;
}

extern "C" int ra_engine_counters(ra_engine* e, ra_counters* out)
{
    if (!e || !out) return RA_E_INVAL;
    CK(cudaSetDevice(e->cfg.device));
    u64 h[RA_N_COUNTERS];
    CK(cudaMemcpyAsync(h, e->C.counters, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    out->aer_received_follower = h[RA_CNT_REF + 0]; out->aer_received_follower_empty = h[RA_CNT_REF + 1];
    out->aer_replies_success = h[RA_CNT_REF + 2]; out->aer_replies_failed = h[RA_CNT_REF + 3];
    out->elections = h[RA_CNT_REF + 4]; out->pre_vote_elections = h[RA_CNT_REF + 5];
    out->term_and_voted_for_updates = h[RA_CNT_REF + 6];
    out->events = h[0]; out->commits = h[1]; out->applied = h[2]; out->msgs_out = h[3];
    out->msgs_dropped = h[4]; out->elections_won = h[5]; out->fatal_rows = h[6]; out->steps = e->steps;
    return RA_OK;
}
