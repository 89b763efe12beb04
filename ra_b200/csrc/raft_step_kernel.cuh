// raft_step_kernel -- the hot kernel of a step (see engine.cu for the frame it lives in: StepSmem, the TMA / mbarrier
// helpers, the counter flushes).  Included by engine.cu inside namespace ra_wide and inside namespace ra_narrow.
#if RA_NARROW_PASS
#define RA_STEP_MINB MINB_NARROW
#else
#define RA_STEP_MINB MINB
#endif
template <int MM, bool FAULTS>
__global__ void __launch_bounds__(CTA_T, RA_STEP_MINB)
raft_step_kernel(const __grid_constant__ Cols C, const int cur, const FloodArgs F,
                 StallCtx* __restrict__ stall_list, u32* __restrict__ stall_count, u32* __restrict__ stall_count_next)
{
    grid_dep_wait();                                            // the step's inputs are the previous kernels' outputs
    grid_dep_launch();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef StepSmem<MM, RA_NARROW_PASS != 0> Smem;
    Smem& S = *reinterpret_cast<Smem*>(smem_raw);
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
#ifdef RA_INTERLEAVE
    // CTAs are handed their tiles slot-interleaved: consecutive CTAs work on different slots' row ranges, so that
    // the long-running warps of one kind of row (a slot full of leaders) are spread over the whole launch
    // instead of filling its first wave.  (grid = per * members CTAs, see launch_step)
    u32 wtile;
    {
        const u32 k = C.members, per = gridDim.x / k;
        wtile = ((blockIdx.x % k) * per + blockIdx.x / k) * WARPS + warp;
    }
#else
    const u32 wtile = blockIdx.x * WARPS + warp;                 // this warp's record tile
#endif
    const u32 r = wtile * RT + lane;
#ifdef RA_WARP_TIMELINE
    const u64 wtl_t0 = wtl_now(r);
#endif
    const bool valid = r < C.rows;
    u32 k_events = 0, k_commits = 0, k_applied = 0, k_msgs = 0, k_dropped = 0, k_elect = 0, k_fatal = 0;
    u64 k_ref = 0;
    if (blockIdx.x == 0 && tid == 0) *stall_count_next = 0;    // the list of the step after this one

    // ---- what does this row have to do? ---------------------------------------------------
    // every per-row input of the step is requested up front, in one round trip to HBM
    const ulonglong2 z2 = make_ulonglong2(0, 0);
    ulonglong2 ap = z2, tc = z2, lg = z2, lw = z2;
    u64 cntw = 0, lrs = 0; u32 nloc = 0;
#if RA_NARROW_PASS
    u32 wfb = 0;                                                // the row's sticky `wide` byte (Cols::wf)
#endif
    if (valid) {
        ap = C.ap[r];
        nloc = C.loc_n[r];
#if RA_NARROW_PASS
        wfb = C.wf[r];
#endif
        if (C.routed) cntw = C.mbox_cnt[cur][r];
        tc = C.tc[r]; lg = C.lg[r]; lw = C.lw[r]; lrs = C.lrs[r];
    }
    if (*C.abort) return;                                       // a host batch was rejected: nothing may change
    const bool fatal0 = MT_FATAL(ap.y) != 0;
    const bool pending = valid && MT_PIPE_PEND(ap.y) != 0;
    // planes of this row: mailbox plane (sender s, depth k) = bit s * DEPTH + k, host slot k = bit NPM + k
    constexpr u32 NPM = (MMEM ? MMEM : RA_MAX_MEMBERS) * RA_MBOX_DEPTH;
    typedef typename PlaneMask<(NPM + RA_LOCAL_CAP <= 32)>::type mask_t;
    mask_t mine = 0;
    u32 my_tail = 0;                                            // senders (bits 0..7) / host slots (8..)
    if (valid && !fatal0) {                                     // whose records carry a 32-byte tail
        u32 mb = 0;
        for (u32 s = 0; s < NMEM(C); s++) {
            const u32 c = (u32)(cntw >> (8 * s)) & 0xffu;
            mb |= ((1u << (c & 7u)) - 1u) << (RA_MBOX_DEPTH * s);
            my_tail |= ((c >> 3) & 1u) << s;
        }
        mine = (mask_t)mb | ((mask_t)((1u << (nloc & 7u)) - 1u) << NPM);
        my_tail |= nloc & 0xff00u;
    }
    const bool work = valid && (F.on || nloc || cntw || pending);
    // everything below is per warp: no CTA-wide barrier anywhere in this kernel
    mask_t todo = mask_or_warp(mine);                           // planes still to consume
    const u32 w_tail = __reduce_or_sync(0xffffffffu, my_tail);
    if (!__any_sync(0xffffffffu, work)) return;                 // whole warp idle
#ifdef RA_WARP_TIMELINE
    const u64 wtl_t1 = wtl_now(w_tail ^ (u32)ap.y);
    const bool wtl_leaders = __all_sync(0xffffffffu, valid && MT_ROLE(ap.y) == RA_LEADER);
#endif
    u64* bars = &S.bars[warp][0];
    if (lane == 0) {
        for (int i = 0; i < NST; i++) mbar_init(&bars[i], 1);
        mbar_fence_init();
    }
    __syncwarp();

    Member m;
#if RA_NARROW_PASS
    member_init(m, C, valid ? r : 0, tc, lg, lw, ap, lrs, cur, reinterpret_cast<ulonglong2*>(reinterpret_cast<uint2*>(S.peers_nm) + tid));
#else
    member_init(m, C, valid ? r : 0, tc, lg, lw, ap, lrs, cur, &S.peers_nm[tid]);
#endif
    m.row = r;
#if RA_NARROW_PASS
    const bool wide_row = wfb != 0;     // some value of this row does not fit 32-bit arithmetic: the general kernel's
#else
    const bool wide_row = false;
#endif
    if (work && !fatal0 && !wide_row && MT_ROLE(ap.y) == RA_LEADER) peers_prefetch<MM>(m);

    bool stalled = false;
    u32 stall_flags = 0;

    // ---- inputs: TMA stages this warp's record tiles through a ring of NST 2 KB slots, in ------
    // evaluation order: deferred pipeline pass, mailbox planes by sender slot then depth, then
    // the host-event planes.  A slot is refilled as soon as the warp has consumed it.
    mask_t rem = 0;                                             // a stalled row's planes not yet evaluated
    if (work && ((!fatal0 && pending) || wide_row)) {           // pipeline_rpcs is not a fast path
        stalled = true; stall_flags = (!fatal0 && pending) ? STALL_PENDING : 0u; rem = mine;
    }
    mask_t toissue = todo;                                      // planes still to request
    u32 n_issued = 0, n_done = 0, st_issue = 0, st = 0, par = 0; // ring positions = counters mod NST, phase parity
#pragma unroll 1
    while (todo) {
        if (lane == 0) {
#pragma unroll 1
            while (toissue && n_issued < n_done + NST) {
                const u32 q = mask_ffs(toissue); toissue &= toissue - 1;
                // (the tile address is rebuilt per issue -- a handful of integer ops in one lane -- instead of
                // holding two 64-bit plane bases in registers through the whole event loop)
                const size_t plane_words = (size_t)C.tiles * (4 * RT);      // 16-byte words per plane
                const ulonglong2* src = (q < NPM ? C.mbox[cur] + (size_t)q * plane_words
                                                 : C.loc + (size_t)(q - NPM) * plane_words) + (size_t)wtile * (4 * RT);
                const u32 tbit = q < NPM ? q / RA_MBOX_DEPTH : 8u + q - NPM;
                const u32 bytes = ((w_tail >> tbit) & 1u) ? TILE_BYTES : TILE_BYTES / 2;
                fence_proxy_async();                            // the slot was read through the generic proxy
                mbar_expect_tx(&bars[st_issue], bytes);
                tma_load_tile(&S.stage[warp][st_issue][0], src, bytes, &bars[st_issue]);
                n_issued++; st_issue = st_issue + 1 == NST ? 0 : st_issue + 1;
            }
        }
        const u32 p = mask_ffs(todo); todo &= todo - 1;
        const bool my = !stalled && ((mine >> p) & 1u);
        mbar_wait(&bars[st], par);
        if (my) {
            const ulonglong2* sp = &S.stage[warp][st][0];
            const ulonglong2 c0 = sp[lane], c1 = sp[RT + lane];
            ulonglong2 t2 = make_ulonglong2(0, 0), t3 = t2;
            if (rec_has_tail(c0)) { t2 = sp[2 * RT + lane]; t3 = sp[3 * RT + lane]; }
            Rec e;
            const bool fits = rec_decode(c0, c1, t2, t3, r, e);  // (narrow pass: every field below 2^30)
            if (MT_FATAL(m.meta)) m.c_pack += 1u;
            else if (FAULTS && p < NPM && flood_lost<MM>(F, C, m, r, e)) m.c_pack += 1u << 20;   // fault injection: lost in transit
            else if (!fits || !note_budget_ok(m) || C.pure || !fast_event<MM>(m, e)) {
                stalled = true;                                 // planes are consumed in bit order:
                rem = mine & ~(((mask_t)1 << p) - 1);           // p and up are left for the general kernel
                atomicAdd(&C.counters[8 + (m_role(m) & 7u) * 16 + (R_type(e) & 15u)], 1ull);   // diagnostics
            }
        }
        n_done++;
        if (++st == NST) { st = 0; par ^= 1u; }
        __syncwarp();                                           // every lane is done with the slot
    }
#ifdef RA_WARP_TIMELINE
    const u64 wtl_t2 = wtl_now(n_done);
#endif
    const u32 rem_mbox = (u32)(rem & (((mask_t)1 << (NPM - 1) << 1) - 1)), rem_loc = (u32)(rem >> (NPM - 1) >> 1);

    if (work) {
        if (cntw && !fatal0) C.mbox_cnt[cur][r] = 0;
        if (nloc) C.loc_n[r] = 0;
        if ((m.pstate & 3u) == 2u) asm volatile("cp.async.wait_all;" ::: "memory");   // prefetch never consumed
        peers_writeback<MM>(m);
        if (!stalled) k_fatal = row_end_of_step<MM, FAULTS>(m, C, r, cur, F);
        if (!wide_row) member_writeback(m, C, r);               // (a wide row's registers were never valid here)
        k_events = m.c_pack & 0xffu; k_commits = m.c_commits; k_applied = m.c_applied;
        k_msgs = (m.c_pack >> 8) & 0xffu; k_dropped = m.c_pack >> 20; k_elect = (m.c_pack >> 16) & 15u;
        k_ref = m.c_ref;
    }
    // stalled rows: hand the rest of the step to raft_general_kernel
    const u32 sm = __ballot_sync(0xffffffffu, stalled);
    if (sm) {
        u32 base = 0;
        if (lane == 0) base = atomicAdd(stall_count, (u32)__popc(sm));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (stalled) {
            ulonglong2* q = reinterpret_cast<ulonglong2*>(&stall_list[base + __popc(sm & ((1u << lane) - 1u))]);
            q[0] = make_ulonglong2((u64)r | ((u64)stall_flags << 32), (u64)rem_mbox | ((u64)rem_loc << 32));
            q[1] = make_ulonglong2((u64)(m.n_msgs | (m.n_notes << 16)) | ((u64)m.status << 32),
                                   (u64)m.sent_to | ((u64)(m.pn_type | (m.pn_slot << 8) | (m.wk << 16)) << 32));
            q[2] = make_ulonglong2(W(m.pn_a), W(m.pn_b));
            q[3] = make_ulonglong2(W(m.pn_c), 0);
        }
    }
    flush_counters(C, lane, k_events, k_commits, k_applied, k_msgs, k_dropped, k_elect, k_fatal);
    flush_ref_counters(C, lane, k_ref);
#ifdef RA_WARP_TIMELINE
    const u64 wtl_t3 = wtl_now(lane);
    if (lane == 0 && wtile < RA_WTL_CAP) {
        WarpTimeline& w = g_wtl[wtile];
        w.t_entry = wtl_t0; w.t_inputs = wtl_t1; w.t_loop = wtl_t2; w.t_exit = wtl_t3;
        w.tile = wtile; w.info = (wtl_smid() & 0xffffu) | ((wtl_leaders ? 1u : 0u) << 16) | ((n_done & 0xffu) << 24);
    }
#endif
}

#undef RA_STEP_MINB
