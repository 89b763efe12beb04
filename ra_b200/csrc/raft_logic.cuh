// raft_logic.cuh -- the member-level Raft logic (records, the per-thread member view, the log view, notes, emit_msg,
// quorum, the leader's RPC passes, elections, the general clauses of ra_server:handle_<state>/2 and the steady-state
// fast paths; reference lines are cited at each function, the map is at the top of raft_common.cuh).
// NO include guard: raft_step.cuh includes this file once per index width, inside namespace ra_wide (RA_NARROW_PASS 0)
// and inside namespace ra_narrow (RA_NARROW_PASS 1; the general clauses are left out there).
//
// ---- index width of this pass (raft_step.cuh) ---------------------------------------------------------
// narrow pass: every index / term lives in ONE 32-bit register.  It is exact because the hot kernel runs a row's
// events through it only while (a) the row's sticky `wide` byte (Cols::wf) is clear -- which, by induction over
// everything that ever writes the row (load_rows, both kernels), means that every value of its state is below 2^30
// plus what one step can add -- and (b) every field of the record at hand is below 2^30 (rec_decode says so);
// anything else stalls to raft_general_kernel, which computes on the ABI's 64 bits.  Memory formats are the same
// in both passes (64-bit cells, 64-byte records): W() widens on the way out, N() narrows on the way in.
#if RA_NARROW_PASS
typedef u32 ix_t;
typedef int sx_t;
#else
typedef u64 ix_t;
typedef i64 sx_t;
#endif
static constexpr ix_t IX_UNDEF = (ix_t)~(ix_t)0;            // == RA_UNDEF in the wide pass
#define RA_NARROW_LIMIT 0x40000000ull                        /* 2^30 */
struct ixpair { ix_t x, y; };
#if RA_NARROW_PASS && defined(RA_HOST_EMU)
// host emulation: a value that leaves or enters the 32-bit pass out of range is a bug in the guards above
extern "C" void ra_emu_narrow_violation(const char* what, unsigned long long v);
__device__ __forceinline__ u64 W(ix_t v) { if (v >= 0x80000000u) ra_emu_narrow_violation("W", v); return (u64)v; }
__device__ __forceinline__ ix_t N(u64 v) { if (v >= 0x80000000ull) ra_emu_narrow_violation("N", v); return (ix_t)v; }
#else
__device__ __forceinline__ u64 W(ix_t v) { return (u64)v; }
__device__ __forceinline__ ix_t N(u64 v) { return (ix_t)v; }
#endif
#if RA_NARROW_PASS
__device__ __forceinline__ u32 lo32(ix_t v) { return v; }
__device__ __forceinline__ u32 hi32(ix_t) { return 0u; }
#else
__device__ __forceinline__ u32 lo32(ix_t v) { return (u32)(v & 0xffffffffull); }
__device__ __forceinline__ u32 hi32(ix_t v) { return (u32)(v >> 32); }
#endif

#if !RA_NARROW_PASS
// 64-byte record as four 16-byte words
struct Rec { ulonglong2 w0, w1, w2, w3; };
__device__ __forceinline__ Rec ld_rec(const ra_event* p)
{
    const ulonglong2* q = reinterpret_cast<const ulonglong2*>(p);
    Rec r; r.w0 = q[0]; r.w1 = q[1]; r.w2 = q[2]; r.w3 = q[3];
    return r;
}
__device__ __forceinline__ void st_rec(ra_event* p, const Rec& r)
{
    ulonglong2* q = reinterpret_cast<ulonglong2*>(p);
    q[0] = r.w0; q[1] = r.w1; q[2] = r.w2; q[3] = r.w3;
}
// ---- record planes: 32-byte head + optional 32-byte tail ---------------------------------------
// Inside the engine (mailbox and host-event planes) a record is stored as
//   chunk 0 {H, term}   chunk 1 {x, y}   [chunk 2 {c, d}   chunk 3 {e, -}]
//   H = type | from << 8 | flags << 16 | shape << 24 | dbit << 31 | n << 32 | n1 << 48
// The shape says how a..e are rebuilt -- a lossless re-encoding that does not depend on the type:
//   RS_LONG   a = x, b = y, c d e from the tail
//   RS_PLAIN  a = x, b = y, c = d = e = 0                       written, command, vote requests ...
//   RS_REPLY  a = x, b = y, c = term, d = dbit, e = 0           append_entries_reply in steady state
//   RS_AER    a = x, b = term, c = y, d = dbit ? term : 0, e = 0  append_entries_rpc in steady state
// Chunks 0 and 1 of a tile are contiguous (1 KB), so a tile none of whose records has a tail costs
// half the bytes to write and to fetch; whether a tail exists travels with the record counts
// (bit 3 of the per-sender count nibble / bits 8.. of loc_n).
enum { RS_LONG = 0, RS_PLAIN = 1, RS_REPLY = 2, RS_AER = 3 };
__device__ __forceinline__ bool st_rec_plane(ulonglong2* base, u32 tiles, u32 plane, u32 row, const Rec& r)
{
    const u64 term = r.w1.x, a = r.w1.y, b = r.w2.x, c = r.w2.y, d = r.w3.x, e = r.w3.y;
    u32 shape = RS_LONG, dbit = 0;
    u64 y = b;
    if (e == 0) {
        if ((c | d) == 0) shape = RS_PLAIN;
        else if (c == term && d <= 1) { shape = RS_REPLY; dbit = (u32)d; }
        else if (b == term && (d == 0 || d == term)) { shape = RS_AER; y = c; dbit = d != 0; }
    }
    const u64 H = ((r.w0.x >> 32) & 0x00FFFFFFull) | ((u64)shape << 24) | ((u64)dbit << 31) | (r.w0.y << 32);
    ulonglong2* q = base + rec_word(tiles, plane, row, 0);
    q[0] = make_ulonglong2(H, term); q[RT] = make_ulonglong2(a, y);
    if (shape != RS_LONG) return false;
    q[2 * RT] = make_ulonglong2(c, d); q[3 * RT] = make_ulonglong2(e, 0);
    return true;
}
__device__ __forceinline__ bool rec_has_tail(const ulonglong2& c0) { return ((u32)(c0.x >> 24) & 3u) == RS_LONG; }
__device__ __forceinline__ Rec rec_decode(const ulonglong2& c0, const ulonglong2& c1, const ulonglong2& t2, const ulonglong2& t3, u32 row)
{
    const u64 H = c0.x, term = c0.y;
    const u32 shape = (u32)(H >> 24) & 3u;
    const u64 dbit = (H >> 31) & 1ull;
    Rec r;
    r.w0.x = (u64)row | ((H & 0x00FFFFFFull) << 32);
    r.w0.y = H >> 32;
    r.w1.x = term; r.w1.y = c1.x;
    r.w2.x = shape == RS_AER ? term : c1.y;
    r.w2.y = shape == RS_LONG ? t2.x : shape == RS_REPLY ? term : shape == RS_AER ? c1.y : 0ull;
    r.w3.x = shape == RS_LONG ? t2.y : shape == RS_REPLY ? dbit : shape == RS_AER ? (dbit ? term : 0ull) : 0ull;
    r.w3.y = shape == RS_LONG ? t3.x : 0ull;
    return r;
}
__device__ __forceinline__ bool rec_decode(const ulonglong2& c0, const ulonglong2& c1, const ulonglong2& t2, const ulonglong2& t3,
                                           u32 row, Rec& r)
{ r = rec_decode(c0, c1, t2, t3, row); return true; }         // (the narrow pass can refuse a record)
__device__ __forceinline__ Rec ld_rec_plane(const ulonglong2* base, u32 tiles, u32 plane, u32 row)
{
    const ulonglong2* q = base + rec_word(tiles, plane, row, 0);
    const ulonglong2 c0 = q[0], c1 = q[RT];
    ulonglong2 t2 = make_ulonglong2(0, 0), t3 = t2;
    if (rec_has_tail(c0)) { t2 = q[2 * RT]; t3 = q[3 * RT]; }
    return rec_decode(c0, c1, t2, t3, row);
}
// header word: row | type<<32 | from<<40 | flags<<48 | pad<<56 ; second: n | n1<<16 | seq<<32
__device__ __forceinline__ u32 R_row(const Rec& r)   { return (u32)r.w0.x; }
__device__ __forceinline__ u32 R_type(const Rec& r)  { return (u32)(r.w0.x >> 32) & 0xff; }
__device__ __forceinline__ u32 R_from(const Rec& r)  { return (u32)(r.w0.x >> 40) & 0xff; }
__device__ __forceinline__ u32 R_flags(const Rec& r) { return (u32)(r.w0.x >> 48) & 0xff; }
__device__ __forceinline__ u32 R_n(const Rec& r)     { return (u32)r.w0.y & 0xffff; }
__device__ __forceinline__ u32 R_n1(const Rec& r)    { return (u32)(r.w0.y >> 16) & 0xffff; }
__device__ __forceinline__ u64 R_term(const Rec& r)  { return r.w1.x; }
__device__ __forceinline__ u64 R_a(const Rec& r)     { return r.w1.y; }
__device__ __forceinline__ u64 R_b(const Rec& r)     { return r.w2.x; }
__device__ __forceinline__ u64 R_c(const Rec& r)     { return r.w2.y; }
__device__ __forceinline__ u64 R_d(const Rec& r)     { return r.w3.x; }
__device__ __forceinline__ u64 R_e(const Rec& r)     { return r.w3.y; }

__device__ __forceinline__ Rec mk_rec(u32 row, u32 type, u32 from, u32 flags, u32 n, u32 n1, u32 seq,
                                      u64 term, u64 a, u64 b, u64 c, u64 d, u64 e)
{
    Rec r;
    r.w0.x = (u64)row | ((u64)(type & 0xff) << 32) | ((u64)(from & 0xff) << 40) | ((u64)(flags & 0xff) << 48);
    r.w0.y = (u64)(n & 0xffff) | ((u64)(n1 & 0xffff) << 16) | ((u64)seq << 32);
    r.w1.x = term; r.w1.y = a; r.w2.x = b; r.w2.y = c; r.w3.x = d; r.w3.y = e;
    return r;
}
__device__ __forceinline__ void R_set_row_seq(Rec& r, u32 row, u32 seq)
{
    r.w0.x = (r.w0.x & 0xFFFFFFFF00000000ull) | row;
    r.w0.y = (r.w0.y & 0x00000000FFFFFFFFull) | ((u64)seq << 32);
}
__device__ __forceinline__ void R_set_from(Rec& r, u32 from)
{
    r.w0.x = (r.w0.x & ~(0xffull << 40)) | ((u64)(from & 0xff) << 40);
}
__device__ __forceinline__ void R_or_flags(Rec& r, u32 f)
{
    r.w0.x |= ((u64)(f & 0xff) << 48);
}
__device__ __forceinline__ void R_clear_pad(Rec& r) { r.w0.x &= ~(0xffull << 56); }

#else   // ---- narrow pass: the same record in ten 32-bit registers ----------------------------------------
// hdr = type | from << 8 | flags << 16 | pad << 24 (the upper half of the ABI header word), nn = n | n1 << 16
struct Rec { u32 row, hdr, nn, seq; ix_t term, a, b, c, d, e; };
__device__ __forceinline__ void st_rec(ra_event* p, const Rec& r)
{
    ulonglong2* q = reinterpret_cast<ulonglong2*>(p);
    q[0] = make_ulonglong2((u64)r.row | ((u64)r.hdr << 32), (u64)r.nn | ((u64)r.seq << 32));
    q[1] = make_ulonglong2(W(r.term), W(r.a)); q[2] = make_ulonglong2(W(r.b), W(r.c)); q[3] = make_ulonglong2(W(r.d), W(r.e));
}
enum { RS_LONG = 0, RS_PLAIN = 1, RS_REPLY = 2, RS_AER = 3 };
__device__ __forceinline__ bool st_rec_plane(ulonglong2* base, u32 tiles, u32 plane, u32 row, const Rec& r)
{
    const ix_t term = r.term, a = r.a, b = r.b, c = r.c, d = r.d, e = r.e;
    u32 shape = RS_LONG, dbit = 0;
    ix_t y = b;
    if (e == 0) {
        if ((c | d) == 0) shape = RS_PLAIN;
        else if (c == term && d <= 1) { shape = RS_REPLY; dbit = (u32)d; }
        else if (b == term && (d == 0 || d == term)) { shape = RS_AER; y = c; dbit = d != 0; }
    }
    const u64 H = (u64)((r.hdr & 0x00FFFFFFu) | (shape << 24) | (dbit << 31)) | ((u64)r.nn << 32);
    ulonglong2* q = base + rec_word(tiles, plane, row, 0);
    q[0] = make_ulonglong2(H, W(term)); q[RT] = make_ulonglong2(W(a), W(y));
    if (shape != RS_LONG) return false;
    q[2 * RT] = make_ulonglong2(W(c), W(d)); q[3 * RT] = make_ulonglong2(W(e), 0);
    return true;
}
__device__ __forceinline__ bool rec_has_tail(const ulonglong2& c0) { return ((u32)(c0.x >> 24) & 3u) == RS_LONG; }
// false: some field does not fit the narrow pass (the event stalls to the general kernel, undecoded)
__device__ __forceinline__ bool rec_decode(const ulonglong2& c0, const ulonglong2& c1, const ulonglong2& t2, const ulonglong2& t3,
                                           u32 row, Rec& r)
{
    const u32 Hlo = (u32)c0.x, shape = (Hlo >> 24) & 3u, dbit = Hlo >> 31;
    const u32 term = (u32)c0.y, x = (u32)c1.x, y = (u32)c1.y;
    u32 big = (u32)(c0.y >> 32) | (u32)(c1.x >> 32) | (u32)(c1.y >> 32) | ((term | x | y) >> 30);
    r.row = row; r.hdr = Hlo & 0x00FFFFFFu; r.nn = (u32)(c0.x >> 32); r.seq = 0;
    r.term = term; r.a = x;
    if (shape == RS_LONG) {
        big |= (u32)(t2.x >> 32) | (u32)(t2.y >> 32) | (u32)(t3.x >> 32) | (((u32)t2.x | (u32)t2.y | (u32)t3.x) >> 30);
        r.b = y; r.c = (u32)t2.x; r.d = (u32)t2.y; r.e = (u32)t3.x;
    } else {
        r.b = shape == RS_AER ? term : y;
        r.c = shape == RS_REPLY ? term : shape == RS_AER ? y : 0u;
        r.d = shape == RS_REPLY ? dbit : shape == RS_AER ? (dbit ? term : 0u) : 0u;
        r.e = 0;
    }
    return big == 0;
}
__device__ __forceinline__ u32 R_row(const Rec& r)   { return r.row; }
__device__ __forceinline__ u32 R_type(const Rec& r)  { return r.hdr & 0xff; }
__device__ __forceinline__ u32 R_from(const Rec& r)  { return (r.hdr >> 8) & 0xff; }
__device__ __forceinline__ u32 R_flags(const Rec& r) { return (r.hdr >> 16) & 0xff; }
__device__ __forceinline__ u32 R_n(const Rec& r)     { return r.nn & 0xffff; }
__device__ __forceinline__ u32 R_n1(const Rec& r)    { return r.nn >> 16; }
__device__ __forceinline__ ix_t R_term(const Rec& r) { return r.term; }
__device__ __forceinline__ ix_t R_a(const Rec& r)    { return r.a; }
__device__ __forceinline__ ix_t R_b(const Rec& r)    { return r.b; }
__device__ __forceinline__ ix_t R_c(const Rec& r)    { return r.c; }
__device__ __forceinline__ ix_t R_d(const Rec& r)    { return r.d; }
__device__ __forceinline__ ix_t R_e(const Rec& r)    { return r.e; }
__device__ __forceinline__ Rec mk_rec(u32 row, u32 type, u32 from, u32 flags, u32 n, u32 n1, u32 seq,
                                      ix_t term, ix_t a, ix_t b, ix_t c, ix_t d, ix_t e)
{
    Rec r;
    r.row = row; r.hdr = (type & 0xff) | ((from & 0xff) << 8) | ((flags & 0xff) << 16);
    r.nn = (n & 0xffff) | ((n1 & 0xffff) << 16); r.seq = seq;
    r.term = term; r.a = a; r.b = b; r.c = c; r.d = d; r.e = e;
    return r;
}
__device__ __forceinline__ void R_set_row_seq(Rec& r, u32 row, u32 seq) { r.row = row; r.seq = seq; }
__device__ __forceinline__ void R_set_from(Rec& r, u32 from) { r.hdr = (r.hdr & ~(0xffu << 8)) | ((from & 0xff) << 8); }
__device__ __forceinline__ void R_or_flags(Rec& r, u32 f) { r.hdr |= (f & 0xff) << 16; }
__device__ __forceinline__ void R_clear_pad(Rec& r) { r.hdr &= 0x00FFFFFFu; }
#endif

// ------------------------------------------------------------------------------------
// per-thread view of one member
// ------------------------------------------------------------------------------------
struct Member {
    const Cols* C;
    u32 row, slot, group;
    // scalars (registers)
    ix_t term, commit, last_idx, last_term, lw_idx, lw_term, applied;
    u64 meta;
    // outputs
    u32 n_msgs, n_notes;
    u32 status;                 // RA_ST_* (bits 0-15) | role at the start of the step << 16 | fatal code << 20 | host events not consumed << 28
    u32 wk;                     // WAL_APPEND notes of this step: count (0..2) | index of the last << 4 | of the one before << 8
    u32 sent_to;                // 4 bits per peer slot: records put in (me -> slot) this step
    // one note kept back so that a continuing WAL_APPEND / APPLY can merge into it
    u32 pn_type, pn_slot; ix_t pn_a, pn_b, pn_c;
    // flood host model: the last two finalised WAL_APPEND notes
    // counters
    u32 c_pack;                 // events | msgs << 8 | elections << 16 | dropped << 20
    u64 c_ref;                  // the reference's counters of this path, 8 bits each (CR_*)
    u32 c_commits, c_applied;   // per row and step: far below 2^32
    int nb;                     // mailbox buffer written this step
    // per-peer columns staged in shared memory on first use: sp[(f*8 + s) * CTA_T], f = 0 next,
    // 1 match, 2 commit_index_sent (this thread's column: consecutive lanes, no bank conflicts)
    ix_t lrs;                   // start index of the last term run (valid when n_runs > 0 and lrs_ok)
    u32 lrs_ok;
    // bit2: the last run changed, Cols::lrs has to be rewritten; bit3: evaluate_quorum ran in this
    // step and none of its inputs (last_written, match indexes, log tail) moved since
    u32 cold;
    // exact shortcut for make_pipelined_rpc_effects: set when a pass found every normal peer with
    // next_index >= next_log_index and commit_index_sent >= commit_index; stays true while only
    // success replies (next/match can only grow) arrive and neither the log nor commit_index move
    u32 pipe_clean;             // cleared wherever last_index or commit_index move
#ifdef RA_HOST_EMU
    ulonglong2* sp;             // &nm[0][thread] of the per-thread peer columns (host emulation: plain memory)
#else
    u32 sp;                     // shared-window address of &nm[0][thread]: one register, and every access is an LDS / STS
#endif
    u32 pstate;                 // bit0 loaded, bits 8..15 {next,match} dirty, bits 16..23 commit_sent dirty
};

__device__ __forceinline__ u32 m_role(const Member& m) { return MT_ROLE(m.meta); }
__device__ __forceinline__ u32 m_nruns(const Member& m) { return MT_NRUNS(m.meta); }
// a member's log view is non-empty iff it holds at least one term run (first_index = start of
// run 0 then, last_index + 1 otherwise: load_rows enforces it, every mutation keeps it)
__device__ __forceinline__ bool log_nonempty(const Member& m) { return MT_NRUNS(m.meta) != 0; }
// COLD row fields -- snapshot index/term, pre-vote token and counter, first_index, machine
// versions -- are not kept in registers at all: the few clauses that need one read it from
// its column (and write it straight back), which keeps ~12 registers out of the hot kernel.
__device__ __forceinline__ ix_t snap_idx(const Member& m)  { return N(m.C->sn[m.row].x); }
__device__ __forceinline__ ix_t snap_term(const Member& m) { return N(m.C->sn[m.row].y); }
__device__ __forceinline__ ix_t tok(const Member& m)       { return N(m.C->tk[m.row].x); }
__device__ __forceinline__ ix_t tok_ctr(const Member& m)   { return N(m.C->tk[m.row].y); }
__device__ __forceinline__ void tok_set(const Member& m, ix_t token, ix_t ctr) { st2(&m.C->tk[m.row], W(token), W(ctr)); }
__device__ __forceinline__ ix_t first_idx(const Member& m) { return N(m.C->fm[m.row].x); }
__device__ __forceinline__ u64 macver(const Member& m)    { return m.C->fm[m.row].y; }   // two packed 32-bit versions
__device__ __forceinline__ void first_idx_set(const Member& m, ix_t v) { m.C->fm[m.row].x = W(v); }
// consistent-query indexes: same treatment (cold; read and written in place)
__device__ __forceinline__ u64& q_index(const Member& m)  { return m.C->qi[m.row]; }
__device__ __forceinline__ u64& q_agreed(const Member& m) { return m.C->qa[m.row]; }
__device__ __forceinline__ u64& q_peer(const Member& m, u32 s) { return m.C->pqi[(size_t)s * m.C->rows + m.row]; }
// reset_query_index/1 :3743-3747 (out of line: reached from the hot kernel only on a term / vote change)
__device__ __noinline__ void reset_query_indexes(u64* pqi, u32 rows, u32 row, u32 members)
{
    for (u32 s = 0; s < members; s++) pqi[(size_t)s * rows + row] = 0;
}

__device__ __forceinline__ ixpair run_get(const Member& m, u32 k)
{ const ulonglong2 v = m.C->run[(size_t)k * m.C->rows + m.row]; ixpair r; r.x = N(v.x); r.y = N(v.y); return r; }
__device__ __forceinline__ void run_set(const Member& m, u32 k, ix_t start, ix_t term)
{ st2(&m.C->run[(size_t)k * m.C->rows + m.row], W(start), W(term)); }
__device__ __forceinline__ void lrs_writeback(const Member& m)
{
    if (!(m.cold & 4u)) return;
    const u32 nr = MT_NRUNS(m.meta);
    m.C->lrs[m.row] = nr ? W(m.lrs_ok ? m.lrs : run_get(m, nr - 1).x) : 0ull;
}

#if !RA_NARROW_PASS
// Per-thread peer columns in shared memory (dynamic peer index without local memory):
//   nm[s][thread] 16 B {next_index, match_index},  cs[s][thread] 8 B commit_index_sent.
// m.sp points at nm[0][thread].
template <int MM>
#ifdef RA_HOST_EMU
__device__ __forceinline__ ulonglong2* peer_nm_p(const Member& m, u32 s) { return m.sp + s * CTA_T; }
#else
__device__ __forceinline__ ulonglong2* peer_nm_p(const Member& m, u32 s)
{ return reinterpret_cast<ulonglong2*>(__cvta_shared_to_generic(m.sp + s * (CTA_T * 16u))); }
#endif
template <int MM>
__device__ __forceinline__ u64* peer_cs_p(const Member& m, u32 s)
{
#ifdef RA_HOST_EMU
    return reinterpret_cast<u64*>(m.sp + PSTR * CTA_T) - threadIdx.x + s * CTA_T;
#else
    // cs[s][thread] sits directly behind nm[PSTR][CTA_T]: nm base of thread 0 + PSTR * CTA_T * 16, then 8-byte cells
    return reinterpret_cast<u64*>(__cvta_shared_to_generic(m.sp - threadIdx.x * 16u + PSTR * (CTA_T * 16u) + (s * CTA_T + threadIdx.x) * 8u));
#endif
}

// asynchronous global -> shared copies of the row's peer cells (LDGSTS): issued as soon as the
// role is known, waited for at the first use, so the DRAM latency hides behind the record tiles
template <int MM>
__device__ __forceinline__ void peers_prefetch(Member& m)
{
#ifndef RA_HOST_EMU
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::
                     "r"((u32)__cvta_generic_to_shared(peer_nm_p<MM>(m, s))), "l"(&C.pnm[(size_t)s * C.rows + m.row]) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::
                     "r"((u32)__cvta_generic_to_shared(peer_cs_p<MM>(m, s))), "l"(&C.pcs[(size_t)s * C.rows + m.row]) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    m.pstate |= 2u;
#else
    (void)m;                                    // host emulation (tests/emu): peers_ensure loads on first use
#endif
}
template <int MM>
__device__ __forceinline__ void peers_ensure(Member& m)
{
    if (m.pstate & 1u) return;
#ifndef RA_HOST_EMU
    if (m.pstate & 2u) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        m.pstate |= 1u;
        return;
    }
#endif
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        *peer_nm_p<MM>(m, s) = C.pnm[(size_t)s * C.rows + m.row];
        *peer_cs_p<MM>(m, s) = C.pcs[(size_t)s * C.rows + m.row];
    }
    m.pstate |= 1u;
}
template <int MM>
__device__ __forceinline__ ixpair peer_nm(Member& m, u32 s)
{ const ulonglong2 v = *peer_nm_p<MM>(m, s); ixpair r; r.x = v.x; r.y = v.y; return r; }
template <int MM>
__device__ __forceinline__ ix_t peer_match(Member& m, u32 s) { return peer_nm_p<MM>(m, s)->y; }
template <int MM>
__device__ __forceinline__ void peer_nm_set(Member& m, u32 s, u64 next, u64 match)
{ *peer_nm_p<MM>(m, s) = make_ulonglong2(next, match); m.pstate |= 1u << (8 + s); }
template <int MM>
__device__ __forceinline__ u64 peer_cs(Member& m, u32 s) { return *peer_cs_p<MM>(m, s); }
template <int MM>
__device__ __forceinline__ void peer_cs_set(Member& m, u32 s, u64 v)
{ *peer_cs_p<MM>(m, s) = v; m.pstate |= 1u << (16 + s); }
template <int MM>
__device__ __forceinline__ void peers_writeback(Member& m)
{
    if (!(m.pstate >> 8)) return;
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        if (m.pstate & (1u << (8 + s))) { ulonglong2 v = *peer_nm_p<MM>(m, s); st2(&C.pnm[(size_t)s * C.rows + m.row], v.x, v.y); }
        if (m.pstate & (1u << (16 + s))) C.pcs[(size_t)s * C.rows + m.row] = *peer_cs_p<MM>(m, s);
    }
}

#else
// Narrow pass: the same per-thread columns hold 32-bit values -- nm[s][thread] 8 B {next_index, match_index},
// cs[c][thread] 4 B commit_index_sent, c = s without the member's own slot (a member is not its own peer; the 512 bytes
// are what lets a seventh CTA fit an SM) -- less than half the shared memory of the 64-bit columns -- filled from the low words of
// the 64-bit cells in HBM (the high words are zero for a row this pass may touch) and written back zero-extended.
// m.sp = shared-window address of nm[0][thread] (host emulation: pointer to this thread's scratch, same layout).
#ifdef RA_HOST_EMU
template <int MM> __device__ __forceinline__ u32* peer_nm_q(const Member& m, u32 s)
{ return reinterpret_cast<u32*>(m.sp) + 2 * (s * CTA_T); }
template <int MM> __device__ __forceinline__ u32* peer_cs_q(const Member& m, u32 s)
{ return reinterpret_cast<u32*>(m.sp) + 2 * (PSTR * CTA_T) + (s - (s > m.slot ? 1u : 0u)) * CTA_T; }
#else
template <int MM> __device__ __forceinline__ u32 peer_nm_a(const Member& m, u32 s) { return m.sp + s * (CTA_T * 8u); }
template <int MM> __device__ __forceinline__ u32 peer_cs_a(const Member& m, u32 s)
{ return m.sp - threadIdx.x * 8u + PSTR * (CTA_T * 8u) + ((s - (s > m.slot ? 1u : 0u)) * CTA_T + threadIdx.x) * 4u; }
template <int MM> __device__ __forceinline__ u32* peer_nm_q(const Member& m, u32 s)
{ return reinterpret_cast<u32*>(__cvta_shared_to_generic(peer_nm_a<MM>(m, s))); }
template <int MM> __device__ __forceinline__ u32* peer_cs_q(const Member& m, u32 s)
{ return reinterpret_cast<u32*>(__cvta_shared_to_generic(peer_cs_a<MM>(m, s))); }
#endif
template <int MM> __device__ __forceinline__ ixpair peer_nm(Member& m, u32 s)
{ const uint2 v = *reinterpret_cast<const uint2*>(peer_nm_q<MM>(m, s)); ixpair r; r.x = v.x; r.y = v.y; return r; }
template <int MM> __device__ __forceinline__ ix_t peer_match(Member& m, u32 s) { return peer_nm_q<MM>(m, s)[1]; }
template <int MM> __device__ __forceinline__ void peer_nm_put(Member& m, u32 s, ix_t next, ix_t match)
{ *reinterpret_cast<uint2*>(peer_nm_q<MM>(m, s)) = make_uint2(next, match); }
template <int MM> __device__ __forceinline__ ix_t peer_cs(Member& m, u32 s) { return *peer_cs_q<MM>(m, s); }
template <int MM> __device__ __forceinline__ void peer_cs_put(Member& m, u32 s, ix_t v) { *peer_cs_q<MM>(m, s) = v; }
template <int MM>
__device__ __forceinline__ void peers_prefetch(Member& m)
{
#ifndef RA_HOST_EMU
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        const ulonglong2* g = &C.pnm[(size_t)s * C.rows + m.row];
        const u32 a = peer_nm_a<MM>(m, s);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(a), "l"(&g->x) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(a + 4u), "l"(&g->y) : "memory");
        if (s != m.slot)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(peer_cs_a<MM>(m, s)), "l"(&C.pcs[(size_t)s * C.rows + m.row]) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    m.pstate |= 2u;
#else
    (void)m;
#endif
}
template <int MM>
__device__ __forceinline__ void peers_ensure(Member& m)
{
    if (m.pstate & 1u) return;
#ifndef RA_HOST_EMU
    if (m.pstate & 2u) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        m.pstate |= 1u;
        return;
    }
#endif
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        const ulonglong2 v = C.pnm[(size_t)s * C.rows + m.row];
        peer_nm_put<MM>(m, s, N(v.x), N(v.y));
        if (s != m.slot) peer_cs_put<MM>(m, s, N(C.pcs[(size_t)s * C.rows + m.row]));
    }
    m.pstate |= 1u;
}
template <int MM>
__device__ __forceinline__ void peer_nm_set(Member& m, u32 s, ix_t next, ix_t match)
{ peer_nm_put<MM>(m, s, next, match); m.pstate |= 1u << (8 + s); }
template <int MM>
__device__ __forceinline__ void peer_cs_set(Member& m, u32 s, ix_t v)
{ if (s == m.slot) return; peer_cs_put<MM>(m, s, v); m.pstate |= 1u << (16 + s); }    // (no column for the own slot)
template <int MM>
__device__ __forceinline__ void peers_writeback(Member& m)
{
    if (!(m.pstate >> 8)) return;
    const Cols& C = *m.C;
    for (u32 s = 0; s < NMEM(C); s++) {
        if (m.pstate & (1u << (8 + s))) { const ixpair v = peer_nm<MM>(m, s); st2(&C.pnm[(size_t)s * C.rows + m.row], W(v.x), W(v.y)); }
        if (m.pstate & (1u << (16 + s))) C.pcs[(size_t)s * C.rows + m.row] = W(peer_cs<MM>(m, s));
    }
}
#endif

// ---- log view -----------------------------------------------------------------------

// run that holds idx (idx <= last_index, log non-empty); returns k, fills start/term/end.
// term = RA_UNDEF when idx lies below the first run, i.e. below first_index.
__device__ __forceinline__ u32 run_find(const Member& m, ix_t idx, ix_t& start, ix_t& term, ix_t& end)
{
    u32 nr = m_nruns(m);
    ix_t e = m.last_idx;
    for (u32 k = nr; k-- > 0;) {
        ixpair r = run_get(m, k);
        if (r.x <= idx) { start = r.x; term = r.y; end = e; return k; }
        e = r.x - 1;
    }
    start = idx; term = IX_UNDEF; end = e;
    return 0;
}

// ra_log:fetch_term/2 (ra_log.erl:1140-1152)
__device__ __forceinline__ ix_t log_fetch_term(const Member& m, sx_t idx)
{
    if (idx < 0) return IX_UNDEF;
    ix_t i = (ix_t)idx;
    if (!log_nonempty(m) || i > m.last_idx) return IX_UNDEF;
    if (i == m.last_idx || (m.lrs_ok && i >= m.lrs)) return m.last_term;     // inside the last run
    ix_t s, t, e; run_find(m, i, s, t, e);
    return t;
}

// ra_server:fetch_term/2 (:3158-3169): falls back on the snapshot
__device__ __forceinline__ ix_t srv_fetch_term(Member& m, sx_t idx)
{
    ix_t t = log_fetch_term(m, idx);
    if (t != IX_UNDEF) return t;
    if (idx >= 0 && MT_HAS_SNAP(m.meta)) {
        if (snap_idx(m) == (ix_t)idx) return snap_term(m);
    }
    return IX_UNDEF;
}

// append n entries of one term at last_index+1 .. (ra_log:append/2, tail of write/2)
__device__ __forceinline__ void log_append(Member& m, ix_t n, ix_t term)
{
    if (n == 0) return;
    u32 nr = m_nruns(m);
    ix_t idx = m.last_idx + 1;
    bool empty = !log_nonempty(m);
    if (empty) { first_idx_set(m, idx); nr = 0; }
    if (empty || nr == 0 || term != m.last_term) {
        if (nr == RA_MAX_RUNS) {
            // contract: forget the oldest run (horizon of RA_MAX_RUNS term runs)
            for (u32 k = 0; k + 1 < RA_MAX_RUNS; k++) { ixpair r = run_get(m, k + 1); run_set(m, k, r.x, r.y); }
            nr = RA_MAX_RUNS - 1;
            first_idx_set(m, run_get(m, 0).x);
        }
        run_set(m, nr, idx, term);
        nr++;
        m.lrs = idx; m.lrs_ok = 1; m.cold |= 4u;
    }
    MT_SET(m.meta, 19, 4, nr);
    m.last_idx = idx + n - 1;
    m.last_term = term;
    m.pipe_clean = 0;                          // next_log_index moved
    m.cold &= ~8u;                             // apply_to may reach further now
}

#if !RA_NARROW_PASS       // truncation, set_last_index, the general written walk: raft_general_kernel only
// drop everything above idx; `fallback_term` is used when idx is no longer inside the log
__device__ __forceinline__ void log_truncate(Member& m, u64 idx, u64 fallback_term)
{
    u32 nr = m_nruns(m);
    m.lrs_ok = 0; m.cold = (m.cold | 4u) & ~8u;
    while (nr > 0 && run_get(m, nr - 1).x > idx) nr--;
    if (!log_nonempty(m) || idx < first_idx(m)) {
        nr = 0;
        first_idx_set(m, idx + 1);
        m.last_term = fallback_term;
    } else {
        m.last_term = run_get(m, nr - 1).y;
    }
    m.last_idx = idx;
    MT_SET(m.meta, 19, 4, nr);
}

// ra_log:set_last_index/2 (ra_log.erl:800-845); false = {not_found,_}
__device__ __forceinline__ bool log_set_last_index(Member& m, u64 idx)
{
    u64 t = log_fetch_term(m, (i64)idx);
    bool has = MT_HAS_SNAP(m.meta) != 0;
    bool at_snap = has && snap_idx(m) == idx;
    if (t == RA_UNDEF && !at_snap) return false;
    if (at_snap) {
        log_truncate(m, idx, snap_term(m));
        m.last_term = snap_term(m);
        m.lw_idx = snap_idx(m); m.lw_term = snap_term(m);
        return true;
    }
    u64 lwidx = idx < m.lw_idx ? idx : m.lw_idx;
    u64 lwterm = (has && snap_idx(m) == lwidx) ? snap_term(m) : log_fetch_term(m, (i64)lwidx);
    log_truncate(m, idx, t);
    m.last_term = t;
    m.lw_idx = lwidx; m.lw_term = lwterm;
    return true;
}

// ra_log:handle_event({written,Term,[{From,To}]}) (ra_log.erl:849-896): the reference walks
// the range down one index at a time; with runs the same answer is found run by run.
__device__ __forceinline__ void log_handle_written(Member& m, u64 term, u64 from, u64 to)
{
    u64 cur = to;
    bool has = MT_HAS_SNAP(m.meta) != 0;
    for (int guard = 0; guard < 2 * RA_MAX_RUNS + 4; guard++) {
        bool in = log_nonempty(m) && cur >= first_idx(m) && cur <= m.last_idx;
        if (in) {
            u64 s, t, e; run_find(m, cur, s, t, e);
            if (t == term) { m.lw_idx = cur; m.lw_term = term; return; }
            u64 lo = s > first_idx(m) ? s : first_idx(m);      // every index in [lo,cur] mismatches
            if (from > lo) return;                            // the walk ends inside the run
            if (lo == 0 || lo - 1 < from) return;
            cur = lo - 1;
            continue;
        }
        if (has && cur <= snap_idx(m)) return;                 // :871-881
        if (cur > m.last_idx) {
            // undefined above the log: the walk either meets the snapshot clause first ...
            u64 stop = cur < snap_idx(m) ? cur : snap_idx(m);
            if (has && snap_idx(m) > m.last_idx && stop >= from) return;
            // ... or reaches last_index
            if (m.last_idx < from) return;
            cur = m.last_idx;
            if (!(log_nonempty(m))) return;                   // below/outside: nothing can match
            continue;
        }
        return;                                               // below the log: no effect either way
    }
}

#endif

// ---- outputs ---------------------------------------------------------------------------

__device__ __forceinline__ void set_fatal(Member& m, u32 code)
{
    if (!(m.status & RA_ST_FATAL)) m.status |= RA_ST_FATAL | ((code & 0xffu) << 20);
    MT_SET(m.meta, 26, 1, 1);
}

// inlined: a leader writes ~3 notes a step, and the out-of-line call (argument moves, CALL / RET) measured slower
// than the larger code (B200: 0.0798 -> 0.0793 ms per flood step, profiles/r03_ab_explore.txt)
__device__ __forceinline__ void note_store_raw(ra_note* slot_ptr, u32 row, u32 type, u32 slot, u32 aux, u64 a, u64 b, u64 c)
{
    ulonglong2* q = reinterpret_cast<ulonglong2*>(slot_ptr);
    q[0] = make_ulonglong2((u64)row | ((u64)(type & 0xff) << 32) | ((u64)(slot & 0xff) << 40) | ((u64)(aux & 0xffff) << 48), a);
    q[1] = make_ulonglong2(b, c);
}
__device__ __forceinline__ void note_store(Member& m, u32 k, u32 type, u32 slot, u32 aux, u64 a, u64 b, u64 c)
{
    note_store_raw(&m.C->onote[(size_t)k * m.C->rows + m.row], m.row, type, slot, aux, a, b, c);
}

// a host ("local") event record into tiled plane k; inlined for the same reason
__device__ __forceinline__ void put_local(ulonglong2* loc, u32 tiles, u32 k, u32 row, u32 type, u32 n, u64 term, u64 a, u64 b)
{
    ulonglong2* q = loc + rec_word(tiles, k, row, 0);               // RS_PLAIN: head only
    q[0] = make_ulonglong2((u64)type | ((u64)RA_NO_SLOT << 8) | ((u64)RS_PLAIN << 24) | ((u64)(n & 0xffff) << 32), term);
    q[RT] = make_ulonglong2(a, b);
}

// `aux`: the row's step flags when this is the last note of the step and no STATUS note follows
__device__ __forceinline__ void note_flush(Member& m, u32 aux = 0)
{
    if (m.pn_type == RA_NOTE_NONE) return;
    note_store(m, m.n_notes - 1, m.pn_type, m.pn_slot, aux, W(m.pn_a), W(m.pn_b), W(m.pn_c));
    if (m.pn_type == RA_NOTE_WAL_APPEND) {          // the flood host model reads the last two back (row_end_of_step)
        const u32 n = m.wk & 3u;
        m.wk = (n < 2 ? n + 1 : 2u) | ((m.n_notes - 1) << 4) | ((m.wk & 0xf0u) << 4);
    }
    m.pn_type = RA_NOTE_NONE;
}

__device__ __forceinline__ void note(Member& m, u32 type, u32 slot, ix_t a, ix_t b, ix_t c)
{
    if (m.pn_type == type && type == RA_NOTE_WAL_APPEND && m.pn_c == c && m.pn_b + 1 == a) { m.pn_b = b; return; }
    if (m.pn_type == type && type == RA_NOTE_APPLY && m.pn_b + 1 == a) { m.pn_b = b; return; }
    if (m.n_notes >= m.C->note_cap - 1) {
        // Cannot happen while an event stays within RA_NOTE_RESERVE notes (note_budget_ok is checked before every
        // event); a burst of per-peer notes can exceed it.  Never lose a note silently: the row stops like a
        // crashed server (the host reloads it from what it persisted).
        m.status |= RA_ST_NOTE_OVERFLOW; set_fatal(m, RA_FATAL_NOTE_OVERFLOW); return;
    }
    note_flush(m);
    m.n_notes++;
    m.pn_type = type; m.pn_slot = slot; m.pn_a = a; m.pn_b = b; m.pn_c = c;
}

// Note budget (include/ra_engine.h, RA_NOTE_RESERVE): a row takes the next event of its step only while
// RA_NOTE_RESERVE slots + the STATUS slot are free.  Otherwise it stops for this step: mailbox records it has
// not reached are dropped and counted like a full transport (Raft tolerates loss, the tick path re-sends),
// host events are left unconsumed and reported (RA_ST_NOTE_OVERFLOW, STATUS.c bits 8..15).
#ifdef RA_NO_BUDGET
__device__ __forceinline__ bool note_budget_ok(const Member&) { return true; }
#else
__device__ __forceinline__ bool note_budget_ok(const Member& m) { return m.n_notes + RA_NOTE_RESERVE + 1u <= m.C->note_cap; }
#endif
__device__ __forceinline__ void budget_drop_record(Member& m)
{ m.status |= RA_ST_NOTE_OVERFLOW | RA_ST_MSG_DROPPED; m.c_pack += 1u << 20; }
__device__ __forceinline__ void budget_refuse_local(Member& m)
{ m.status |= RA_ST_NOTE_OVERFLOW; m.status += 1u << 28; }          // bits 28..31: host events not consumed

// send one RPC record to the member in `to` of my group
template <int MM>
__device__ __forceinline__ void emit_msg(Member& m, u32 to, Rec r)
{
    const Cols& C = *m.C;
    u32 dst = to * C.groups + m.group;                  // (an id outside the group is the host's business)
    const bool is_next = (R_flags(r) & RA_EVF_NEXT_EVENT) != 0;
    const bool routed = MTR == TR_RUNTIME ? (C.routed != 0) : (MTR != TR_HOST);
    if (routed && !is_next && to >= NMEM(C)) return;    // no mailbox for an unknown peer
    if (!is_next) R_set_from(r, m.slot);
    R_clear_pad(r);
    if (routed && !is_next) {
        u32 k = (m.sent_to >> (4 * to)) & 7u;        // bit 3 of the nibble: some record has a tail
        if (k >= RA_MBOX_DEPTH) { m.status |= RA_ST_MSG_DROPPED; m.c_pack += 1u << 20; return; }
        R_set_row_seq(r, dst, k);
        const bool sharded = MTR == TR_RUNTIME ? (C.n_shards > 1) : (MTR == TR_PEER || MTR == TR_BUCKET);
        if (sharded) {
            const u32 ds = (C.shard + to + 8u * C.n_shards - m.slot) % C.n_shards;
            const bool peer = MTR == TR_RUNTIME ? (C.peer_mode != 0) : (MTR == TR_PEER);
            if (peer) {
                // NVLink peer store into the destination GPU's mailbox plane (same local row index)
                if (st_rec_plane(C.peer_mbox[m.nb][ds], C.tiles, m.slot * RA_MBOX_DEPTH + k, dst, r)) m.sent_to |= 8u << (4 * to);
                m.sent_to += 1u << (4 * to);
                m.c_pack += 1u << 8;
                return;
            }
            if (ds != C.shard) {
                // bucket of the destination shard: one atomic per group of converged lanes
                const u32 act = __activemask();
                const u32 grp = __match_any_sync(act, ds);
                const u32 ldr = __ffs(grp) - 1;
                u32 base = 0;
                if ((threadIdx.x & 31u) == ldr) base = atomicAdd(&C.out_cnt[ds], (u32)__popc(grp));
                base = __shfl_sync(grp, base, ldr);
                const u32 pos = base + __popc(grp & ((1u << (threadIdx.x & 31u)) - 1u));
                if (pos >= C.out_cap) { m.status |= RA_ST_MSG_DROPPED; m.c_pack += 1u << 20; return; }
                st_rec(&C.outbox[(size_t)ds * C.out_cap + pos], r);
                m.sent_to += 1u << (4 * to);
                m.c_pack += 1u << 8;
                return;
            }
        }
        if (st_rec_plane(C.mbox[m.nb], C.tiles, m.slot * RA_MBOX_DEPTH + k, dst, r)) m.sent_to |= 8u << (4 * to);
        m.sent_to += 1u << (4 * to);
        m.c_pack += 1u << 8;
        return;
    }
    if (m.n_msgs >= RA_MSG_CAP) { m.status |= RA_ST_MSG_DROPPED; m.c_pack += 1u << 20; return; }
    R_set_row_seq(r, dst, m.n_msgs);
    st_rec(&C.omsg[(size_t)m.n_msgs * C.rows + m.row], r);
    m.n_msgs++;
    m.c_pack += 1u << 8;
}

// ---- next-event queue (gen_statem semantics: new next_events go to the front) ----------
// A {next_event,_} is never an arbitrary message on this path: it is the event being handled
// (re-dispatched under the new role) or one of four synthetic ones, so the queue holds 4-bit
// codes, not 64-byte records, and lives in one register.
enum { NX_REDISPATCH = 1, NX_PIPELINE = 2, NX_SELF_PRE_VOTE = 3, NX_SELF_VOTE = 4, NX_NOOP = 5, NX_TICK = 6 };
struct NextQ { u32 codes; u32 n; };
__device__ __forceinline__ void nq_push(NextQ& q, u32 code) { q.codes |= code << (4 * q.n); q.n++; }

// ---- term / vote --------------------------------------------------------------------

// shifts of the reference's per-path counters inside Member::c_ref (ra.hrl:324-343)
enum { CR_AER_RX = 0, CR_AER_RX_EMPTY = 8, CR_REPLY_OK = 16, CR_REPLY_FAIL = 24, CR_ELECTIONS = 32, CR_PRE_VOTE_ELECTIONS = 40,
       CR_TERM_VOTE = 48 };
#ifdef RA_NO_REF_COUNTERS
#define CR_INC(m, f) ((void)0)
#else
#define CR_INC(m, f) ((m).c_ref += 1ull << (f))
#endif

// update_term_and_voted_for/3 :3014-3031
__device__ __forceinline__ void update_term_and_voted_for(Member& m, ix_t term, u32 voted)
{
    if (term == m.term && voted == MT_VOTED(m.meta)) return;
    CR_INC(m, CR_TERM_VOTE);                                            // :3026
    // reset_query_index/1 :3029.  Every peer query_index of the engine is zero until a heartbeat reply or
    // ra_engine_load_query_state writes one -- both raise q_used first -- so until then there is nothing to reset
    if (*m.C->q_used) reset_query_indexes(m.C->pqi, m.C->rows, m.row, m.C->members);
    m.term = term;
    MT_SET(m.meta, 7, 4, voted);
    m.status |= RA_ST_TERM_VOTE_CHANGED;
}
// update_term/2 :3033-3037
__device__ __forceinline__ void update_term(Member& m, ix_t term)
{
    if (term > m.term) update_term_and_voted_for(m, term, SLOT_NONE);
}
// is_candidate_log_up_to_date/3 :3132-3139
__device__ __forceinline__ bool log_up_to_date(ix_t idx, ix_t term, ix_t last_idx, ix_t last_term)
{
    return term > last_term || (term == last_term && idx >= last_idx);
}
// required_quorum/1 :3969-3972
template <int MM>
__device__ __forceinline__ u32 required_quorum(const Member& m)
{
    u32 mask = (u32)(m.meta >> 56) & ((1u << NMEM(*m.C)) - 1u);
    return (u32)__popc(mask) / 2 + 1;
}

// append_entries_reply/3 :3597-3604
__device__ __forceinline__ Rec aer_reply(const Member& m, ix_t term, bool success)
{
    return mk_rec(0, RA_EV_AER_REPLY, 0, 0, 0, 0, 0, term, m.last_idx + 1, m.lw_idx, m.lw_term, success ? 1 : 0, 0);
}
template <int MM>
__device__ __forceinline__ void reply_vote(Member& m, u32 to, u32 type, ix_t term, ix_t token, bool granted)
{
    emit_msg<MM>(m, to, mk_rec(0, type, 0, 0, 0, 0, 0, term, 0, 0, token, granted ? 1 : 0, 0));
}

// ---- apply / quorum -----------------------------------------------------------------

// apply_to/3 :3217-3255 for '$usr' / same-version noop entries
__device__ __forceinline__ void apply_to(Member& m, ix_t upto)
{
    if (!(upto > m.applied)) return;
    if (!MT_MV_OK(m.meta)) return;
    ix_t from = m.applied + 1;
    ix_t to = m.last_idx < upto ? m.last_idx : upto;
    if (to < from) return;
    note(m, RA_NOTE_APPLY, 0, from, to, 0);
    m.c_applied += (u32)(to - from + 1);
    m.applied = to;
}

// evaluate_quorum/2 :3606-3619 with match_indexes/1 :3644-3655 and agreed_commit/1
// :3657-3661.  The reference sorts [LastWritten | voter match indexes] descending and takes
// element trunc(N/2)+1.  Here one value per member slot sits in a register (the leader's own
// slot holds its last_written index, a non-voter contributes 0, which can never be ranked
// above a real candidate), an odd-even transposition network orders them, and the element is
// picked by rank: no array in local memory, no data-dependent loop.
template <typename T>
__device__ __forceinline__ void cex(T& a, T& b)              // a >= b afterwards
{
    const bool sw = a < b;
    const T t = sw ? b : a;
    b = sw ? a : b;
    a = t;
}
template <int MM>
__device__ __forceinline__ void evaluate_quorum(Member& m)
{
    const u32 M = NMEM(*m.C);
    constexpr int NV = MMEM ? MMEM : RA_MAX_MEMBERS;
    ix_t v[NV];
    u32 n = 1;
#pragma unroll
    for (int s = 0; s < NV; s++) {
        const bool in = (u32)s < M;
        const bool self = (u32)s == m.slot;
        const bool voter = in && !self && MT_VOTER(m.meta, s);
        v[s] = self ? m.lw_idx : (voter ? peer_match<MM>(m, s) : (ix_t)0);
        n += voter ? 1u : 0u;
    }
    const u32 nth = n / 2 + 1;                                  // 1-based rank, descending
    const ix_t ci0 = m.commit;
#ifndef RA_NO_QSHORT
    {
        // exact shortcut for the common outcome "nothing moves": the nth largest value IS commit_index exactly
        // when fewer than nth values exceed it and at least nth reach it; increment_commit_index/1 then leaves
        // commit_index alone whatever fetch_term says (8 of a steady-state leader's 9 evaluations per step)
        u32 gt = 0, ge = 0;
#pragma unroll
        for (int s = 0; s < NV; s++) { gt += v[s] > ci0 ? 1u : 0u; ge += v[s] >= ci0 ? 1u : 0u; }
        if (gt < nth && ge >= nth) { apply_to(m, m.commit); m.cold |= 8u; return; }
    }
#endif
#pragma unroll
    for (int pass = 0; pass < NV; pass++) {
#pragma unroll
        for (int i = pass & 1; i + 1 < NV; i += 2) cex(v[i], v[i + 1]);
    }
    ix_t best = v[0];
#pragma unroll
    for (int i = 1; i < NV; i++) best = (nth == (u32)(i + 1)) ? v[i] : best;
    if (srv_fetch_term(m, (sx_t)best) == m.term) m.commit = best;       // §5.4.2 gate :3625-3629
    if (m.commit != ci0) m.pipe_clean = 0;
    if (m.commit > ci0) {
        note(m, RA_NOTE_COMMIT, 0, ci0, m.commit, 0);
        m.c_commits += (u32)(m.commit - ci0);
    }
    apply_to(m, m.commit);
    m.cold |= 8u;
}

// evaluate_commit_index_follower/2 :2229-2263
__device__ __forceinline__ void evaluate_commit_index_follower(Member& m)
{
    if (MT_LEADER(m.meta) == SLOT_NONE) return;
    apply_to(m, m.last_idx < m.commit ? m.last_idx : m.commit);
}

// ---- leader RPC generation --------------------------------------------------------------

// make_append_entries_rpc/6 :2401-2418 -> new next index
template <int MM>
__device__ __forceinline__ ix_t make_aer(Member& m, u32 peer, sx_t prev_idx, ix_t prev_term, ix_t num)
{
    ix_t last = m.last_idx;
    ix_t from = (ix_t)(prev_idx + 1);
    ix_t to = (ix_t)prev_idx + num; if (last < to) to = last;
    u32 n = 0, n1 = 0; ix_t d = 0, e = 0;
    ix_t s = 0, t = IX_UNDEF, end = 0; u32 k = 0;
    if (to >= from && log_nonempty(m) && from <= m.last_idx) {
        if (m.lrs_ok && from >= m.lrs) { s = m.lrs; t = m.last_term; end = m.last_idx; k = m_nruns(m) - 1; }
        else k = run_find(m, from, s, t, end);
    }
    if (t != IX_UNDEF) {                                   // `from` is inside the log
        d = t;
        if (end < to) {                                   // second run; contract: cut after it
            n1 = (u32)(end - from + 1);
            ixpair r2 = run_get(m, k + 1);
            e = r2.y;
            ix_t end2 = (k + 2 < m_nruns(m)) ? run_get(m, k + 2).x - 1 : m.last_idx;
            if (end2 < to) to = end2;
        }
        n = (u32)(to - from + 1);
    } else {
        to = from - 1; if (last < to) to = last;
    }
    emit_msg<MM>(m, peer, mk_rec(0, RA_EV_AER, 0, 0, n, n1, 0, m.term, (ix_t)prev_idx, prev_term, m.commit, d, e));
    return to + 1;
}

// make_rpc_effect/5 :2365-2399
template <int MM>
__device__ __forceinline__ ix_t make_rpc_effect(Member& m, u32 peer, ix_t next, ix_t max_batch, bool& snapshot)
{
    sx_t prev = (sx_t)next - 1;
    snapshot = false;
    ix_t pt = log_fetch_term(m, prev);
    if (pt != IX_UNDEF) return make_aer<MM>(m, peer, prev, pt, max_batch);
    if (!MT_HAS_SNAP(m.meta)) { set_fatal(m, RA_FATAL_NO_SNAPSHOT); return next; }
    if (prev >= 0 && snap_idx(m) == (ix_t)prev) return make_aer<MM>(m, peer, prev, snap_term(m), max_batch);
    if (!(prev < (sx_t)snap_idx(m))) { set_fatal(m, RA_FATAL_ASSERT); return next; }
    snapshot = true;
    note(m, RA_NOTE_SEND_SNAPSHOT, peer, peer, snap_idx(m), 0);
    return snap_idx(m);
}

#if !RA_NARROW_PASS
// ---- consistent queries: the heartbeat round, :3700-3825 (general path only) ------------------
// heartbeat_reply/2 :3700-3702, cast to the rpc's leader_id
template <int MM>
__device__ __forceinline__ void send_heartbeat_reply(Member& m, u32 to, u64 term, u64 query_index)
{
    emit_msg<MM>(m, to, mk_rec(0, RA_EV_HEARTBEAT_REPLY, 0, 0, 0, 0, 0, term, query_index, 0, 0, 0, 0));
}
// heartbeat_rpc_effects/4 :3749-3771: normal peers whose query_index lags
template <int MM>
__device__ __forceinline__ void heartbeat_rpc_effects(Member& m, u64 query_index)
{
    for (u32 s = 0; s < NMEM(*m.C); s++) {
        if (s == m.slot) continue;
        if (MT_PSTATUS(m.meta, s) != RA_PEER_NORMAL) continue;
        if (!(q_peer(m, s) < query_index)) continue;
        emit_msg<MM>(m, s, mk_rec(0, RA_EV_HEARTBEAT_RPC, 0, 0, 0, 0, 0, m.term, query_index, 0, 0, 0, 0));
    }
}
// get_current_query_quorum/1 :3796-3797 = agreed_commit(query_indexes/1 :3632-3642): own index and the
// voter peers', same rank select as evaluate_quorum
template <int MM>
__device__ __forceinline__ u64 query_quorum(Member& m)
{
    const u32 M = NMEM(*m.C);
    constexpr int NV = MMEM ? MMEM : RA_MAX_MEMBERS;
    u64 v[NV];
    u32 n = 1;
#pragma unroll
    for (int s = 0; s < NV; s++) {
        const bool in = (u32)s < M;
        const bool self = (u32)s == m.slot;
        const bool voter = in && !self && MT_VOTER(m.meta, s);
        v[s] = self ? q_index(m) : (voter ? q_peer(m, s) : 0ull);
        n += voter ? 1u : 0u;
    }
#pragma unroll
    for (int pass = 0; pass < NV; pass++) {
#pragma unroll
        for (int i = pass & 1; i + 1 < NV; i += 2) cex(v[i], v[i + 1]);
    }
    const u32 nth = n / 2 + 1;
    u64 best = v[0];
#pragma unroll
    for (int i = 1; i < NV; i++) best = (nth == (u32)(i + 1)) ? v[i] : best;
    return best;
}
// what the waiting queries learn: every one with an index <= agreed is applied by the host
__device__ __forceinline__ void query_agreed(Member& m, u64 agreed)
{
    if (agreed > q_agreed(m)) {
        q_agreed(m) = agreed;
        note(m, RA_NOTE_QUERY_AGREED, 0, agreed, 0, 0);
    }
}
// update_heartbeat_rpc_effects/1 :3704-3720 (tick, enforce leadership)
template <int MM>
__device__ __forceinline__ void update_heartbeat_rpc_effects(Member& m)
{
    if (NMEM(*m.C) <= 1) query_agreed(m, q_index(m));         // no peers: apply everything waiting
    else heartbeat_rpc_effects<MM>(m, q_index(m));
}

#endif

// The leader's three ways of walking its peers share one loop (one inlined copy of
// make_rpc_effect/5 in the hot kernel):
//   RP_PIPELINE  make_pipelined_rpc_effects/3 :2268-2329 -> More
//   RP_STALE     make_rpcs/1 over stale_peers/1 :2985-3003 (tick)       } batch 1, peers are
//   RP_ALL       make_all_rpcs/1 :2337-2350 (enforce leadership)        } not updated
enum { RP_PIPELINE = 0, RP_STALE = 1, RP_ALL = 2 };
template <int MM>
__device__ __forceinline__ bool rpc_pass(Member& m, u32 mode, bool force, const bool heartbeats = true)
{
    // (`heartbeats` = false in the hot kernel: its one RP_ALL call site has made sure that no consistent
    // query is in flight and that every peer is `normal`, so neither heartbeats nor backoff peers exist)
    const Cols& C = *m.C;
    if (mode == RP_PIPELINE && m.pipe_clean && !force) return false;
    ix_t next_log_idx = m.last_idx + 1;
#if RA_NARROW_PASS
    // (the configured limits are 32-bit unsigned; every quantity they are compared with or cut to is below 2^31 in
    // this pass -- in_flight, the distance to last_index -- so clamping them to 2^31 - 1 changes no outcome)
    sx_t max_pipe = (sx_t)(C.max_pipeline < 0x7fffffffu ? C.max_pipeline : 0x7fffffffu);
    sx_t max_batch = (sx_t)(C.max_batch < 0x7fffffffu ? C.max_batch : 0x7fffffffu);
#else
    sx_t max_pipe = C.max_pipeline, max_batch = C.max_batch;
#endif
    bool more = false, clean = true;
    if (heartbeats && mode == RP_ALL)          // make_all_rpcs/1: CancelEffects ++ EffectsAER ++ EffectsHR
        for (u32 s = 0; s < NMEM(C); s++)
            if (s != m.slot && MT_PSTATUS(m.meta, s) == RA_PEER_SNAPSHOT_BACKOFF)
                note(m, RA_NOTE_CANCEL_SNAPSHOT_RETRY, s, s, 0, 0);
    for (u32 s = 0; s < NMEM(C); s++) {
        if (s == m.slot) continue;
        if (MT_PSTATUS(m.meta, s) != RA_PEER_NORMAL &&
            !(heartbeats && mode == RP_ALL && MT_PSTATUS(m.meta, s) == RA_PEER_SNAPSHOT_BACKOFF)) continue;
        ixpair nm = peer_nm<MM>(m, s);
        ix_t cs = peer_cs<MM>(m, s);
        i64 bs = 1;                            // (64-bit in both passes: max_pipe - in_flight may pass 2^31)
        if (mode == RP_PIPELINE) {
            if (!(nm.x < next_log_idx || cs < m.commit)) continue;
            sx_t in_flight = (sx_t)nm.x - (sx_t)nm.y - 1;
            if (!(in_flight < max_pipe || force)) { clean = false; continue; }
            bs = (i64)max_pipe - (i64)in_flight; if ((i64)max_batch < bs) bs = max_batch; if (bs < 1) bs = 1;
        } else if (mode == RP_STALE) {
            bool stale = ((sx_t)nm.y < (sx_t)nm.x - 1) || (cs < m.commit);
            if (!stale) continue;
        }
        bool snap;
        ix_t nn = make_rpc_effect<MM>(m, s, nm.x, (ix_t)bs, snap);
        if (MT_FATAL(m.meta)) return false;
        if (mode != RP_PIPELINE) continue;
        if (!(nn >= nm.x)) { set_fatal(m, RA_FATAL_ASSERT); return false; }
        peer_nm_set<MM>(m, s, nn, nm.y);
        peer_cs_set<MM>(m, s, m.commit);
        if (snap && !C.pure) MT_SET(m.meta, 32 + 3 * s, 3, RA_PEER_SENDING_SNAPSHOT);
        sx_t nif = (sx_t)nn - (sx_t)nm.y - 1;
        if (nn < next_log_idx && nif < max_pipe) more = true;
        if (nn < next_log_idx) clean = false;
    }
    if (mode == RP_PIPELINE) m.pipe_clean = clean ? 1u : 0u;
#if !RA_NARROW_PASS
    else if (heartbeats) update_heartbeat_rpc_effects<MM>(m);  // make_rpcs / make_all_rpcs: EffectsAER ++ EffectsHR
#endif
    return more;
}
template <int MM>
__device__ __forceinline__ bool make_pipelined_rpcs(Member& m, bool force) { return rpc_pass<MM>(m, RP_PIPELINE, force); }
template <int MM>
__device__ __forceinline__ void make_rpcs(Member& m, bool all) { (void)rpc_pass<MM>(m, all ? RP_ALL : RP_STALE, false); }

#if !RA_NARROW_PASS
// initialise_peers/1 :3207-3215 (becoming leader: general path)
template <int MM>
__device__ __forceinline__ void initialise_peers(Member& m)
{
    ix_t next = m.last_idx + 1;
    m.pstate |= 1u;                         // every peer cell is overwritten: nothing to load
    m.pipe_clean = 0;
    for (u32 s = 0; s < NMEM(*m.C); s++) {
        peer_nm_set<MM>(m, s, next, 0);
        peer_cs_set<MM>(m, s, 0);
        q_peer(m, s) = 0;                   // new_peer/0 :2963-2968
        MT_SET(m.meta, 32 + 3 * s, 3, RA_PEER_NORMAL);
    }
}

#endif

// ---- elections --------------------------------------------------------------------------

// call_for_election/3 :2853-2897
template <int MM>
__device__ __forceinline__ u32 call_for_election(Member& m, u32 target, NextQ& nq)
{
    Rec req;
    if (target == RA_CANDIDATE) {
        ix_t nt = m.term + 1;
        CR_INC(m, CR_ELECTIONS);                                        // :2856
        req = mk_rec(0, RA_EV_REQUEST_VOTE, 0, 0, 0, 0, 0, nt, m.last_idx, m.last_term, 0, 0, 0);
        update_term_and_voted_for(m, nt, m.slot);
    } else {
        ix_t token = tok_ctr(m) + 1;                                // make_ref()
        CR_INC(m, CR_PRE_VOTE_ELECTIONS);                               // :2878
#if RA_NARROW_PASS
        // (fast_event let the row in only with machine version 0: version 1 | machine version << 32 fits)
        req = mk_rec(0, RA_EV_PRE_VOTE, 0, 0, 0, 0, 0, m.term, m.last_idx, m.last_term, token, 1u, 0);
#else
        u64 mv = macver(m) & 0xffffffffull;
        req = mk_rec(0, RA_EV_PRE_VOTE, 0, 0, 0, 0, 0, m.term, m.last_idx, m.last_term, token, 1ull | (mv << 32), 0);
#endif
        update_term_and_voted_for(m, m.term, m.slot);
        tok_set(m, token, token);
    }
    MT_SET(m.meta, 3, 4, SLOT_NONE);       // leader_id => undefined
    MT_SET(m.meta, 15, 4, 0);              // votes => 0
    nq_push(nq, target == RA_CANDIDATE ? NX_SELF_VOTE : NX_SELF_PRE_VOTE);   // {next_event, cast, VoteForSelf}
    for (u32 s = 0; s < NMEM(*m.C); s++)
        if (s != m.slot) emit_msg<MM>(m, s, req);
    return target;
}

// process_pre_vote/3 :2899-2956 (one reply site)
template <int MM>
__device__ __forceinline__ u32 process_pre_vote(Member& m, u32 fsm, const Rec& e)
{
    ix_t term = R_term(e), token = R_c(e);
    u32 version = lo32(R_d(e)), their = hi32(R_d(e));
    const u64 mvs = macver(m);
    u32 macver = (u32)(mvs & 0xffffffffull), eff = (u32)(mvs >> 32);
    bool send = true, granted = false, tmo = false;
    ix_t rterm = term;
    if (term >= m.term) {
        update_term(m, term);
        if (log_up_to_date(R_a(e), R_b(e), m.last_idx, m.last_term)) {
            if (version > 1) granted = false;                                   // :2914-2917
            else if (their == eff || (their >= eff && their <= macver)) granted = true;   // :2918-2928
            else { granted = false; tmo = true; }                               // :2929-2934
        } else if (fsm == RA_FOLLOWER) { send = false; tmo = true; }            // :2941-2942
        else granted = false;                                                   // :2943-2945
    } else {
        rterm = m.term;                                                         // :2948-2956
    }
    if (tmo) m.status |= RA_ST_START_ELECTION_TMO;
    if (send) reply_vote<MM>(m, R_from(e), RA_EV_PRE_VOTE_RES, rterm, token, granted);
    return fsm;
}

#if !RA_NARROW_PASS       // ---- the general clauses: raft_general_kernel (and the host emulation) only -----------------
// has_log_entry_or_snapshot/3 :3141-3156  (0 ok, 1 missing, 2 term_mismatch)
__device__ __forceinline__ u32 has_entry(const Member& m, u64 idx, u64 term)
{
    u64 t = log_fetch_term(m, (i64)idx);
    if (t == RA_UNDEF) {
        if (MT_HAS_SNAP(m.meta) && snap_idx(m) == idx) return snap_term(m) == term ? 0u : 2u;
        return 1u;
    }
    return t == term ? 0u : 2u;
}

__device__ __forceinline__ void remember_cond_reply(Member& m, u32 reason, const Rec& rp)
{
    const Cols& C = *m.C;
    MT_SET(m.meta, 13, 2, reason);
    MT_SET(m.meta, 25, 1, 1);
    st2(&C.cd[m.row], R_term(rp), R_a(rp));
    st2(&C.cd[(size_t)C.rows + m.row], R_b(rp), R_c(rp));
}

// ---- handle_follower/2 :1264-1641 -----------------------------------------------------------
template <int MM>
__device__ __forceinline__ u32 handle_follower(Member& m, const Rec& e, NextQ& nq)
{
    const u32 type = R_type(e);
    if (type == RA_EV_AER) {
        u64 term = R_term(e), cur = m.term;
        u32 leader = R_from(e);
        CR_INC(m, CR_AER_RX);                                              // :1278 and :1418
        if (term >= cur) {
            u64 pl_idx = R_a(e), pl_term = R_b(e), leader_commit = R_c(e);
            u32 n0 = R_n(e), n1 = R_n1(e);
            m.status |= RA_ST_LEADER_MSG;
            MT_SET(m.meta, 3, 4, leader);
            update_term(m, term);
            u32 r = has_entry(m, pl_idx, pl_term);
            if (r == 0) {
                // drop_existing/3 :3673-3681, run by run instead of entry by entry
                u64 idx = pl_idx + 1, stop = pl_idx + n0;
                while (idx <= stop) {
                    if (!log_nonempty(m) || idx > m.last_idx) break;
                    u64 s, t, end; run_find(m, idx, s, t, end);
                    if (t == RA_UNDEF) break;
                    bool first_piece = (n1 != 0) && (idx - (pl_idx + 1) < n1);
                    u64 et = (n1 == 0 || first_piece) ? R_d(e) : R_e(e);
                    u64 pe = first_piece ? pl_idx + n1 : stop;
                    if (t != et) break;
                    u64 seg = end < pe ? end : pe;
                    idx = seg + 1;
                }
                u64 k = idx - (pl_idx + 1);
                u64 last_valid = idx - 1;
                if (k == n0) {                                             // Entries == [] :1288
                    CR_INC(m, CR_AER_RX_EMPTY);                            // :1290
                    u64 local_last = m.last_idx;
                    bool validated;
                    if (n0 == 0 && local_last > pl_idx) {                  // :1294-1303
                        if (pl_idx < m.applied) { set_fatal(m, RA_FATAL_ASSERT); return RA_FOLLOWER; }
                        if (!log_set_last_index(m, pl_idx)) { set_fatal(m, RA_FATAL_SET_LAST_INDEX_NOT_FOUND); return RA_FOLLOWER; }
                        note(m, RA_NOTE_TRUNCATE, 0, m.last_idx, m.last_term, 0);
                        validated = true;
                    } else validated = local_last <= last_valid;
                    if (validated) {                                       // :1313-1326
                        m.commit = leader_commit;
                        evaluate_commit_index_follower(m);
                        emit_msg<MM>(m, leader, aer_reply(m, term, true));
                    } else {                                               // :1327-1346
                        u64 lvi = m.applied > last_valid ? m.applied : last_valid;
                        emit_msg<MM>(m, leader, mk_rec(0, RA_EV_AER_REPLY, 0, 0, 0, 0, 0, cur, lvi + 1, lvi,
                                                   srv_fetch_term(m, (i64)lvi), 1, 0));
                    }
                    return RA_FOLLOWER;
                }
                // [{FstIdx,_,_}|_] :1348-1371
                u64 fst = pl_idx + 1 + k;
                if (fst < m.applied) { set_fatal(m, RA_FATAL_ASSERT); return RA_FOLLOWER; }
                if (!(fst <= m.last_idx + 1) || (!log_nonempty(m) && fst != m.last_idx + 1)) {
                    set_fatal(m, RA_FATAL_WRITE_INTEGRITY); return RA_FOLLOWER;
                }
                m.commit = leader_commit;
                if (fst <= m.last_idx) {
                    u64 pt = log_fetch_term(m, (i64)fst - 1);
                    log_truncate(m, fst - 1, pt != RA_UNDEF ? pt : snap_term(m));
                }
                // remaining entries fst..stop: at most two term pieces
                u64 split = (n1 != 0) ? pl_idx + n1 : stop;       // last index of the first piece
                if (n1 != 0 && fst <= split) {
                    u64 c1 = split - fst + 1;
                    log_append(m, c1, R_d(e));
                    note(m, RA_NOTE_WAL_APPEND, 0, fst, split, R_d(e));
                    if (stop > split) {
                        if (R_e(e) == R_d(e)) { log_append(m, stop - split, R_e(e)); note(m, RA_NOTE_WAL_APPEND, 0, split + 1, stop, R_e(e)); }
                        else { log_append(m, stop - split, R_e(e)); note(m, RA_NOTE_WAL_APPEND, 0, split + 1, stop, R_e(e)); }
                    }
                } else {
                    u64 t = (n1 == 0) ? R_d(e) : R_e(e);
                    log_append(m, stop - fst + 1, t);
                    note(m, RA_NOTE_WAL_APPEND, 0, fst, stop, t);
                }
                evaluate_commit_index_follower(m);
                return RA_FOLLOWER;
            }
            if (r == 1) {                                                  // missing :1373-1387
                Rec rp = aer_reply(m, term, false);
                remember_cond_reply(m, 1, rp);
                emit_msg<MM>(m, leader, rp);
                return RA_AWAIT_CONDITION;
            }
            // term_mismatch :1388-1413 -> mismatch_append_entries_reply/3 :3587-3595
            u64 la = m.applied, lat = srv_fetch_term(m, (i64)la);
            if (lat == RA_UNDEF) { set_fatal(m, RA_FATAL_ASSERT); return RA_FOLLOWER; }
            Rec rp = mk_rec(0, RA_EV_AER_REPLY, 0, 0, 0, 0, 0, term, la + 1, la, lat, 0, 0);
            remember_cond_reply(m, 2, rp);
            emit_msg<MM>(m, leader, rp);
            return RA_AWAIT_CONDITION;
        }
        emit_msg<MM>(m, leader, aer_reply(m, cur, false));                     // :1415-1424
        return RA_FOLLOWER;
    }
    if (type == RA_EV_WRITTEN) {                                           // :1441-1458
        u64 a = m.lw_idx, b = m.lw_term;
        log_handle_written(m, R_term(e), R_a(e), R_b(e));
        u32 leader = MT_LEADER(m.meta);
        if ((a != m.lw_idx || b != m.lw_term) && leader != SLOT_NONE)
            emit_msg<MM>(m, leader, aer_reply(m, m.term, true));
        return RA_FOLLOWER;
    }
    if (type == RA_EV_PRE_VOTE) {                                          // :1459-1466
        if (MT_MEMBERSHIP(m.meta) != RA_VOTER) return RA_FOLLOWER;
        return process_pre_vote<MM>(m, RA_FOLLOWER, e);
    }
    if (type == RA_EV_REQUEST_VOTE) {                                      // :1467-1513
        if (MT_MEMBERSHIP(m.meta) != RA_VOTER) return RA_FOLLOWER;
        u64 term = R_term(e), cur = m.term;
        u32 cand = R_from(e), voted = MT_VOTED(m.meta);
        if (term == cur && voted != SLOT_NONE && voted != (cand & 15u)) {
            reply_vote<MM>(m, cand, RA_EV_REQUEST_VOTE_RES, term, 0, false);
        } else if (term >= cur) {
            update_term(m, term);
            if (log_up_to_date(R_a(e), R_b(e), m.last_idx, m.last_term)) {
                reply_vote<MM>(m, cand, RA_EV_REQUEST_VOTE_RES, term, 0, true);
                update_term_and_voted_for(m, term, cand & 15u);
            } else reply_vote<MM>(m, cand, RA_EV_REQUEST_VOTE_RES, term, 0, false);
        } else reply_vote<MM>(m, cand, RA_EV_REQUEST_VOTE_RES, cur, 0, false);
        return RA_FOLLOWER;
    }
    if (type == RA_EV_AER_REPLY) {                                         // :1514-1517
        update_term(m, R_term(e) > m.term ? R_term(e) : m.term);
        return RA_FOLLOWER;
    }
    if (type == RA_EV_ELECTION_TIMEOUT) {                                  // :1603-1610
        if (MT_MEMBERSHIP(m.meta) != RA_VOTER) return RA_FOLLOWER;
        return call_for_election<MM>(m, RA_PRE_VOTE, nq);
    }
    if (type == RA_EV_COMMAND) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, R_n(e), l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_CONSISTENT_QUERY) {                                  // only a leader answers consistent queries
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, 0, l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_HEARTBEAT_RPC) {
        if (R_term(e) >= m.term) {                                         // :1425-1434
            update_term(m, R_term(e));
            MT_SET(m.meta, 3, 4, R_from(e));
            send_heartbeat_reply<MM>(m, R_from(e), R_term(e), R_a(e));
        } else send_heartbeat_reply<MM>(m, R_from(e), m.term, R_a(e));     // :1435-1440
        return RA_FOLLOWER;
    }
    if (type == RA_EV_HEARTBEAT_REPLY) {                                   // :1518-1521
        update_term(m, R_term(e) > m.term ? R_term(e) : m.term);
        return RA_FOLLOWER;
    }
    return RA_FOLLOWER;
}

// ---- handle_leader/2 :520-1023 --------------------------------------------------------------
__device__ __forceinline__ Rec pipeline_event(const Member& m)
{
    return mk_rec(m.row, RA_EV_PIPELINE_RPCS, RA_NO_SLOT, RA_EVF_INFO, 0, 0, 0, 0, 0, 0, 0, 0, 0);
}
template <int MM>
__device__ __forceinline__ u32 step_down(Member& m, u64 term)
{
    MT_SET(m.meta, 3, 4, SLOT_NONE);
    update_term(m, term);
    return RA_FOLLOWER;
}

template <int MM>
__device__ __forceinline__ u32 handle_leader(Member& m, const Rec& e, NextQ& nq)
{
    const Cols& C = *m.C;
    const u32 type = R_type(e);
    if (type == RA_EV_AER_REPLY) {
        u64 term = R_term(e);
        u32 from = R_from(e);
        bool success = R_d(e) != 0;
        bool known = from < NMEM(C);
        if (success && term == m.term) {                                   // :522-561
            CR_INC(m, CR_REPLY_OK);                                        // :528
            if (!known) return RA_LEADER;
            ixpair nm = peer_nm<MM>(m, from);
            u64 nn = R_a(e) > nm.x ? R_a(e) : nm.x;
            u64 mm = R_b(e) > nm.y ? R_b(e) : nm.y;
            peer_nm_set<MM>(m, from, nn, mm);
            evaluate_quorum<MM>(m);
            nq_push(nq, NX_PIPELINE);
            return RA_LEADER;
        }
        if (term > m.term) {                                               // :562-576
            if (!known) return RA_LEADER;
            return step_down<MM>(m, term);
        }
        if (!success) {                                                    // :577-643
            if (!known) return RA_LEADER;
            CR_INC(m, CR_REPLY_FAIL);                                      // :590
            ixpair nm = peer_nm<MM>(m, from);
            u64 pnext = R_a(e), plast = R_b(e), plast_term = R_c(e);
            u64 t = log_fetch_term(m, (i64)plast);
            u64 nn = nm.x, mm = nm.y;
            if (t == RA_UNDEF) nn = pnext;
            else if (t == plast_term && plast >= nm.y) { mm = plast; nn = pnext; }
            else if (plast < nm.y) { mm = plast; nn = plast + 1; }
            else {
                i64 a = (i64)nm.x - 1, b = (i64)pnext;
                i64 x = a < b ? a : b;
                nn = x > (i64)nm.y ? (u64)x : nm.y;
            }
            peer_nm_set<MM>(m, from, nn, mm);
            m.pipe_clean = 0;                       // next_index may have moved back
            (void)make_pipelined_rpcs<MM>(m, false);
        }
        return RA_LEADER;
    }
    if (type == RA_EV_COMMAND) {                                           // :644-729
        u64 n = R_n(e);
        if (n == 0) return RA_LEADER;
        u64 from = m.last_idx + 1;
        log_append(m, n, m.term);                                          // append_log_leader/3
        note(m, RA_NOTE_WAL_APPEND, 0, from, from + n - 1, m.term);
        (void)make_pipelined_rpcs<MM>(m, (R_flags(e) & RA_EVF_NOOP) != 0);
        return RA_LEADER;
    }
    if (type == RA_EV_WRITTEN) {                                           // :730-735
        log_handle_written(m, R_term(e), R_a(e), R_b(e));
        evaluate_quorum<MM>(m);
        nq_push(nq, NX_PIPELINE);
        return RA_LEADER;
    }
    if (type == RA_EV_PIPELINE_RPCS) {                                     // :784-792
        if (make_pipelined_rpcs<MM>(m, false)) nq_push(nq, NX_PIPELINE);
        return RA_LEADER;
    }
    if (type == RA_EV_AER) {
        if (R_term(e) > m.term) { u32 r = step_down<MM>(m, R_term(e)); nq_push(nq, NX_REDISPATCH); return r; }   // :826-835
        if (R_term(e) == m.term) { set_fatal(m, RA_FATAL_LEADER_SAW_AER_SAME_TERM); return RA_LEADER; } // :836-840
        emit_msg<MM>(m, R_from(e), aer_reply(m, m.term, false));               // :841-845
        return RA_LEADER;
    }
    if (type == RA_EV_REQUEST_VOTE) {
        if (R_term(e) > m.term) {                                          // :919-933
            if (R_from(e) >= NMEM(C)) return RA_LEADER;
            u32 r = step_down<MM>(m, R_term(e)); nq_push(nq, NX_REDISPATCH); return r;
        }
        reply_vote<MM>(m, R_from(e), RA_EV_REQUEST_VOTE_RES, m.term, 0, false);     // :934-936
        return RA_LEADER;
    }
    if (type == RA_EV_PRE_VOTE) {
        if (R_term(e) > m.term) {                                          // :937-951
            if (R_from(e) >= NMEM(C)) return RA_LEADER;
            u32 r = step_down<MM>(m, R_term(e)); nq_push(nq, NX_REDISPATCH); return r;
        }
        make_rpcs<MM>(m, true);                                                // :952-957
        return RA_LEADER;
    }
    if (type == RA_EV_CONSISTENT_QUERY) {                  // :846-851 + make_heartbeat_rpc_effects/2 :3722-3739
        if (NMEM(C) <= 1) { note(m, RA_NOTE_QUERY_APPLY, 0, m.commit, 0, 0); return RA_LEADER; }   // no peers
        const u64 qi = ++q_index(m);
        heartbeat_rpc_effects<MM>(m, qi);
        note(m, RA_NOTE_QUERY_INDEX, 0, qi, m.commit, 0);
        return RA_LEADER;
    }
    if (type == RA_EV_HEARTBEAT_RPC) {
        if (R_term(e) > m.term) { u32 r = step_down<MM>(m, R_term(e)); nq_push(nq, NX_REDISPATCH); return r; }   // :871-880
        if (R_term(e) < m.term) { send_heartbeat_reply<MM>(m, R_from(e), m.term, R_a(e)); return RA_LEADER; }    // :881-888
        set_fatal(m, RA_FATAL_LEADER_SAW_HEARTBEAT_SAME_TERM);                                                    // :889-894
        return RA_LEADER;
    }
    if (type == RA_EV_HEARTBEAT_REPLY) {                                   // :895-918
        if (R_term(e) == m.term) {                                         // heartbeat_rpc_quorum/3 :3773-3795
            const u32 from = R_from(e);
            if (from < NMEM(C) && R_a(e) > q_peer(m, from)) { *m.C->q_used = 1u; q_peer(m, from) = R_a(e); }   // update_peer_query_index/3
            query_agreed(m, query_quorum<MM>(m));
            return RA_LEADER;
        }
        if (R_term(e) > m.term) return step_down<MM>(m, R_term(e));
        return RA_LEADER;                                                  // lower term: ignored
    }
    if (type == RA_EV_TICK) make_rpcs<MM>(m, false);                           // ra_server_proc.erl:610-613
    return RA_LEADER;
}

// ---- handle_candidate/2 :1026-1171 ----------------------------------------------------------
template <int MM>
__device__ __forceinline__ u32 handle_candidate(Member& m, const Rec& e, NextQ& nq)
{
    const u32 type = R_type(e);
    if (type == RA_EV_REQUEST_VOTE_RES) {
        if (R_d(e) && R_term(e) == m.term) {                               // :1028-1044
            u32 nv = MT_VOTES(m.meta) + 1;
            if (nv == required_quorum<MM>(m)) {
                MT_SET(m.meta, 3, 4, m.slot);
                initialise_peers<MM>(m);
                MT_SET(m.meta, 15, 4, 0);
                nq_push(nq, NX_NOOP);
                m.c_pack += 1u << 16;
                return RA_LEADER;
            }
            MT_SET(m.meta, 15, 4, nv);
            return RA_CANDIDATE;
        }
        if (R_term(e) > m.term) { update_term_and_voted_for(m, R_term(e), SLOT_NONE); return RA_FOLLOWER; }  // :1045-1052
        return RA_CANDIDATE;
    }
    if (type == RA_EV_AER) {
        if (R_term(e) >= m.term) {                                         // :1055-1058
            update_term_and_voted_for(m, R_term(e), SLOT_NONE);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        emit_msg<MM>(m, R_from(e), aer_reply(m, m.term, false));               // :1059-1063
        return RA_CANDIDATE;
    }
    if (type == RA_EV_AER_REPLY) {
        if (R_term(e) > m.term) { update_term_and_voted_for(m, R_term(e), SLOT_NONE); return RA_FOLLOWER; }  // :1082-1090
        return RA_CANDIDATE;
    }
    if (type == RA_EV_REQUEST_VOTE) {
        if (R_term(e) > m.term) {                                          // :1091-1098
            update_term_and_voted_for(m, R_term(e), SLOT_NONE);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        reply_vote<MM>(m, R_from(e), RA_EV_REQUEST_VOTE_RES, m.term, 0, false);     // :1107-1109
        return RA_CANDIDATE;
    }
    if (type == RA_EV_PRE_VOTE) {
        if (R_term(e) > m.term) {                                          // :1099-1106
            update_term_and_voted_for(m, R_term(e), SLOT_NONE);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        return process_pre_vote<MM>(m, RA_CANDIDATE, e);                       // :1110-1114
    }
    if (type == RA_EV_WRITTEN) { log_handle_written(m, R_term(e), R_a(e), R_b(e)); return RA_CANDIDATE; }
    if (type == RA_EV_ELECTION_TIMEOUT) return call_for_election<MM>(m, RA_CANDIDATE, nq);
    if (type == RA_EV_COMMAND) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, R_n(e), l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_CONSISTENT_QUERY) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, 0, l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_HEARTBEAT_RPC) {
        if (R_term(e) >= m.term) {                                         // :1064-1067
            update_term_and_voted_for(m, R_term(e), SLOT_NONE);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        send_heartbeat_reply<MM>(m, R_from(e), m.term, R_a(e));            // :1068-1073
        return RA_CANDIDATE;
    }
    if (type == RA_EV_HEARTBEAT_REPLY && R_term(e) > m.term) {             // :1074-1081
        update_term_and_voted_for(m, R_term(e), SLOT_NONE);
        return RA_FOLLOWER;
    }
    return RA_CANDIDATE;
}

// ---- handle_pre_vote/2 :1173-1261 -----------------------------------------------------------
template <int MM>
__device__ __forceinline__ u32 handle_pre_vote(Member& m, const Rec& e, NextQ& nq)
{
    const u32 type = R_type(e);
    if (type == RA_EV_AER) {
        if (R_term(e) >= m.term) {                                         // :1175-1180
            update_term(m, R_term(e));
            MT_SET(m.meta, 15, 4, 0);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        return RA_PRE_VOTE;
    }
    if (type == RA_EV_REQUEST_VOTE) {
        if (R_term(e) > m.term) {                                          // :1196-1201
            update_term(m, R_term(e));
            MT_SET(m.meta, 15, 4, 0);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        return RA_PRE_VOTE;
    }
    if (type == RA_EV_PRE_VOTE_RES) {
        if (R_term(e) > m.term) {                                          // :1202-1207
            update_term(m, R_term(e));
            MT_SET(m.meta, 15, 4, 0);
            return RA_FOLLOWER;
        }
        if (R_d(e) && R_term(e) == m.term && R_c(e) == tok(m) && MT_MEMBERSHIP(m.meta) == RA_VOTER) {  // :1212-1229
            u32 nv = MT_VOTES(m.meta) + 1;
            if (nv == required_quorum<MM>(m)) return call_for_election<MM>(m, RA_CANDIDATE, nq);
            MT_SET(m.meta, 15, 4, nv);
        }
        return RA_PRE_VOTE;
    }
    if (type == RA_EV_PRE_VOTE) return process_pre_vote<MM>(m, RA_PRE_VOTE, e);
    if (type == RA_EV_ELECTION_TIMEOUT) return call_for_election<MM>(m, RA_PRE_VOTE, nq);
    if (type == RA_EV_WRITTEN) { log_handle_written(m, R_term(e), R_a(e), R_b(e)); return RA_PRE_VOTE; }
    if (type == RA_EV_COMMAND) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, R_n(e), l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_CONSISTENT_QUERY) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, 0, l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    if (type == RA_EV_HEARTBEAT_RPC) {
        if (R_term(e) >= m.term) {                                         // :1181-1186
            update_term(m, R_term(e));
            MT_SET(m.meta, 15, 4, 0);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        send_heartbeat_reply<MM>(m, R_from(e), m.term, R_a(e));            // :1187-1191
        return RA_PRE_VOTE;
    }
    if (type == RA_EV_HEARTBEAT_REPLY && R_term(e) > m.term) {             // :1192-1195
        MT_SET(m.meta, 15, 4, 0);
        update_term(m, R_term(e));
        return RA_FOLLOWER;
    }
    return RA_PRE_VOTE;
}

// ---- handle_await_condition/2 :1900-1941 ------------------------------------------------------
template <int MM>
__device__ __forceinline__ u32 handle_await_condition(Member& m, const Rec& e, NextQ& nq)
{
    const Cols& C = *m.C;
    const u32 type = R_type(e);
    if (type == RA_EV_REQUEST_VOTE) { nq_push(nq, NX_REDISPATCH); return RA_FOLLOWER; }           // :1902-1903
    if (type == RA_EV_PRE_VOTE) return process_pre_vote<MM>(m, RA_AWAIT_CONDITION, e);    // :1904-1905
    if (type == RA_EV_ELECTION_TIMEOUT) {                                             // :1906-1913
        if (MT_MEMBERSHIP(m.meta) != RA_VOTER) return RA_AWAIT_CONDITION;
        return call_for_election<MM>(m, RA_PRE_VOTE, nq);
    }
    if (type == RA_EV_AWAIT_COND_TIMEOUT) {                                           // :1914-1927
        u32 leader = MT_LEADER(m.meta);
        if (MT_COND_VALID(m.meta) && leader != SLOT_NONE) {
            ulonglong2 c0 = C.cd[m.row], c1 = C.cd[(size_t)C.rows + m.row];
            emit_msg<MM>(m, leader, mk_rec(0, RA_EV_AER_REPLY, 0, 0, 0, 0, 0, c0.x, c0.y, c1.x, c1.y, 0, 0));
            m.status |= RA_ST_LEADER_MSG;
        }
        MT_SET(m.meta, 13, 2, 0); MT_SET(m.meta, 25, 1, 0);
        return RA_FOLLOWER;
    }
    if (type == RA_EV_WRITTEN) { log_handle_written(m, R_term(e), R_a(e), R_b(e)); return RA_AWAIT_CONDITION; }
    if (type == RA_EV_AER) {                                                          // :1932-1941
        bool ok = false;
        if (R_term(e) >= m.term) {                                                    // :2184-2202
            u32 r = has_entry(m, R_a(e), R_b(e));
            ok = (r == 0) || (r == 2 && MT_COND(m.meta) == 1);
        }
        if (ok) {
            MT_SET(m.meta, 13, 2, 0); MT_SET(m.meta, 25, 1, 0);
            nq_push(nq, NX_REDISPATCH);
            return RA_FOLLOWER;
        }
        return RA_AWAIT_CONDITION;
    }
    if (type == RA_EV_COMMAND) m.status |= RA_ST_CMD_POSTPONED;
    if (type == RA_EV_CONSISTENT_QUERY) {
        u32 l = MT_LEADER(m.meta);
        note(m, RA_NOTE_NOT_LEADER, 0, 0, l == SLOT_NONE ? RA_NO_SLOT : l, 0);
    }
    return RA_AWAIT_CONDITION;                 // heartbeat rpcs and replies are dropped here (:1938-1940)
}

// ---- the ra_server_proc shim ------------------------------------------------------------------
__device__ __forceinline__ Rec synth_event(const Member& m, u32 code, const Rec& in)
{
    switch (code) {
    case NX_PIPELINE:      return mk_rec(m.row, RA_EV_PIPELINE_RPCS, RA_NO_SLOT, RA_EVF_INFO, 0, 0, 0, 0, 0, 0, 0, 0, 0);
    case NX_SELF_PRE_VOTE: return mk_rec(m.row, RA_EV_PRE_VOTE_RES, m.slot, 0, 0, 0, 0, m.term, 0, 0, tok(m), 1, 0);
    case NX_SELF_VOTE:     return mk_rec(m.row, RA_EV_REQUEST_VOTE_RES, m.slot, 0, 0, 0, 0, m.term, 0, 0, 0, 1, 0);
    case NX_NOOP:          return mk_rec(m.row, RA_EV_COMMAND, RA_NO_SLOT, RA_EVF_NOOP, 1, 0, 0, 0, 0, 0, 0, 0, 0);
    case NX_TICK:          return mk_rec(m.row, RA_EV_TICK, RA_NO_SLOT, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0);
    default:               return in;
    }
}

template <int MM>
__device__ __forceinline__ void process_event(Member& m, const Rec& in)
{
    const Cols& C = *m.C;
    peers_ensure<MM>(m);                       // general path: any clause may touch the peer columns
    m.cold &= ~8u;                             // ... or an input of evaluate_quorum
    u32 pend = NX_REDISPATCH, np = 1;          // queue of codes, front = low nibble
    bool chased = false;
    m.c_pack += 1u;
    while (np > 0) {
        if (MT_FATAL(m.meta)) return;
        const u32 code = pend & 15u;
        pend >>= 4; np--;
        if (code == NX_PIPELINE ||
            (code == NX_REDISPATCH && R_type(in) == RA_EV_PIPELINE_RPCS && (R_flags(in) & RA_EVF_INFO))) {
            // contract: one chased pipeline pass per input event; the rest runs next step
            if (chased) { MT_SET(m.meta, 24, 1, 1); m.status |= RA_ST_PIPELINE_PENDING; continue; }
            chased = true;
        }
        const Rec e = synth_event(m, code, in);
        NextQ nq; nq.codes = 0; nq.n = 0;
        const u32 old = m_role(m);
        u32 nr;
        switch (old) {
        case RA_LEADER:          nr = handle_leader<MM>(m, e, nq); break;
        case RA_FOLLOWER:        nr = handle_follower<MM>(m, e, nq); break;
        case RA_CANDIDATE:       nr = handle_candidate<MM>(m, e, nq); break;
        case RA_PRE_VOTE:        nr = handle_pre_vote<MM>(m, e, nq); break;
        case RA_AWAIT_CONDITION: nr = handle_await_condition<MM>(m, e, nq); break;
        default:                 nr = old; break;
        }
        if (MT_FATAL(m.meta)) return;
        if (nr != old) {
            MT_SET(m.meta, 0, 3, nr);
            m.status |= RA_ST_ROLE_CHANGED;
            if (!C.pure && nr == RA_FOLLOWER)                      // become/3 :2166-2175
                m.meta &= ~(0xFFFFFFull << 32);
            if (nr == RA_LEADER) m.status |= RA_ST_BECAME_LEADER;
        }
        if (C.pure) {
            for (u32 i = 0; i < nq.n; i++) {
                Rec r = synth_event(m, (nq.codes >> (4 * i)) & 15u, e);
                R_or_flags(r, RA_EVF_NEXT_EVENT);
                emit_msg<MM>(m, m.slot, r);
            }
            continue;
        }
        // candidate -> leader: tick_timeout goes ahead of the effects' next events
        // (ra_server_proc.erl:728-730)
        u32 front = nq.codes, nf = nq.n;
        if (nr == RA_LEADER && old == RA_CANDIDATE) { front = (front << 4) | NX_TICK; nf++; }
        if (nf) {
            if (np + nf > 8) { set_fatal(m, RA_FATAL_ASSERT); return; }   // (cannot happen: <= 3 next events per clause)
            pend = (pend << (4 * nf)) | (front & ((nf >= 8) ? 0xFFFFFFFFu : ((1u << (4 * nf)) - 1u)));
            np += nf;
        }
    }
}

#endif  // !RA_NARROW_PASS

// ---- steady-state fast paths ---------------------------------------------------------------
// The flood is dominated by a handful of event shapes.  Each fast path is the general clause
// specialised under an explicit guard (every condition the general path would test on the
// way); anything else -- term changes, log mismatch, candidates, multi-run batches ... --
// takes process_event() in raft_general_kernel.  Both routes are diffed against the oracle by
// the parity tests.  Shared tails (apply, reply, quorum, rpc pass) have ONE call site each: the
// hot kernel has to stay small enough for the instruction cache.
template <int MM>
__device__ __forceinline__ bool fast_event(Member& m, const Rec& e)
{
    const u32 type = R_type(e);
    u32 role = m_role(m);
    const bool nonempty = m_nruns(m) != 0;
#ifdef RA_LEAN_FAST
    // only the five steady-state shapes stay in the hot kernel (instruction-cache footprint): elections,
    // votes and enforce-leadership go to the general kernel
    if (!(type == RA_EV_AER || type == RA_EV_WRITTEN || type == RA_EV_AER_REPLY || type == RA_EV_COMMAND)) return false;
    if (role != RA_FOLLOWER && role != RA_LEADER) return false;
#endif
#ifndef RA_LEAN_FAST
    if (role == RA_PRE_VOTE && type == RA_EV_AER && R_term(e) >= m.term && !m.C->pure) {
        // handle_pre_vote(#append_entries_rpc{}) :1175-1180: back to follower, the rpc is
        // re-queued ({next_event, Msg}) and handled as a follower right away
        update_term(m, R_term(e));
        MT_SET(m.meta, 15, 4, 0);
        MT_SET(m.meta, 0, 3, RA_FOLLOWER);
        m.status |= RA_ST_ROLE_CHANGED;
        m.meta &= ~(0xFFFFFFull << 32);                            // become/3 :2166-2175
        role = RA_FOLLOWER;
    }
#endif
    if (role == RA_FOLLOWER) {
        bool apply = false, reply = false;
        ix_t reply_term = 0;
        u32 leader = MT_LEADER(m.meta);
        if (type == RA_EV_AER) {
            // handle_follower(#append_entries_rpc{}) :1266-1371, prev entry = our last entry
            if (R_term(e) != m.term || R_n1(e) != 0 || !nonempty || R_a(e) != m.last_idx || R_b(e) != m.last_term) return false;
            const u32 n = R_n(e);
            if (n != 0 && (R_d(e) != m.last_term || m.last_idx + 1 < m.applied)) return false;
            m.c_pack += 1u;
            m.c_ref += (1ull << CR_AER_RX) + (n == 0 ? 1ull << CR_AER_RX_EMPTY : 0ull);   // :1278, :1290
            leader = R_from(e);
            m.status |= RA_ST_LEADER_MSG;
            MT_SET(m.meta, 3, 4, leader);
            m.commit = R_c(e);                                         // :1314-1315 / :1349
            if (n == 0) {                                              // validated empty AER :1313-1326
                reply = true; reply_term = R_term(e);
            } else {
                const ix_t fst = m.last_idx + 1;
                m.last_idx += n;                                       // same term: the last run grows
                note(m, RA_NOTE_WAL_APPEND, 0, fst, m.last_idx, m.last_term);
            }
            apply = true;
        } else if (type == RA_EV_WRITTEN) {
            // handle_follower({ra_log_event,{written,..}}) :1441-1458, range ends inside the last run
            // (every index of the last run has term last_term: ra_log:fetch_term(To) == Term)
            if (nonempty && !m.lrs_ok) { m.lrs = run_get(m, m_nruns(m) - 1).x; m.lrs_ok = 1; }
            if (!nonempty || !m.lrs_ok || R_term(e) != m.last_term || R_b(e) > m.last_idx || R_b(e) < m.lrs) return false;
            m.c_pack += 1u;
            reply = (m.lw_idx != R_b(e) || m.lw_term != m.last_term) && leader != SLOT_NONE;
            reply_term = m.term;
            m.lw_idx = R_b(e); m.lw_term = m.last_term;
#ifndef RA_LEAN_FAST
        } else if (type == RA_EV_PRE_VOTE) {                           // :1459-1466
            m.c_pack += 1u;
            if (MT_MEMBERSHIP(m.meta) == RA_VOTER) (void)process_pre_vote<MM>(m, RA_FOLLOWER, e);
        } else if (type == RA_EV_PRE_VOTE_RES || type == RA_EV_REQUEST_VOTE_RES) {   // :1593-1598: ignored
            m.c_pack += 1u;
        } else if (type == RA_EV_ELECTION_TIMEOUT) {
            // :1603-1610 -> call_for_election(pre_vote) :2873-2897, then the queued vote for self
            // (handle_pre_vote :1212-1229): one vote, which is not yet a quorum
            if (MT_MEMBERSHIP(m.meta) != RA_VOTER || required_quorum<MM>(m) == 1 || m.C->pure) return false;
#if RA_NARROW_PASS
            // the pre_vote record carries version | machine_version << 32 and a fresh token: both have to fit
            if ((macver(m) & 0xffffffffull) != 0 || m.C->tk[m.row].y >= RA_NARROW_LIMIT) return false;
#endif
            m.c_pack += 1u;
            NextQ nq; nq.codes = 0; nq.n = 0;
            (void)call_for_election<MM>(m, RA_PRE_VOTE, nq);
            MT_SET(m.meta, 0, 3, RA_PRE_VOTE);
            m.status |= RA_ST_ROLE_CHANGED;
            MT_SET(m.meta, 15, 4, 1);
#endif
        } else return false;
        if (apply) evaluate_commit_index_follower(m);
        if (reply) emit_msg<MM>(m, leader, aer_reply(m, reply_term, true));
        return true;
    }
    if (role == RA_LEADER) {
        if (type == RA_EV_PRE_VOTE_RES || type == RA_EV_REQUEST_VOTE_RES) {   // :958-963: ignored
            m.c_pack += 1u;
            return true;
        }
        peers_ensure<MM>(m);              // the ONE place the hot kernel stages the peer columns
        bool quorum = false, chase = false, force = false;
        u32 mode = RP_PIPELINE;
#ifndef RA_LEAN_FAST
        if (type == RA_EV_PRE_VOTE) {                                  // :952-957 enforce leadership
            // (with a consistent query in flight make_all_rpcs also re-sends heartbeats: general path)
            if (R_term(e) > m.term || ((m.meta >> 32) & 0xFFFFFFull) != 0 || q_index(m) != 0) return false;
            m.c_pack += 1u;
            mode = RP_ALL;
        } else
#endif
        if (type == RA_EV_COMMAND) {                            // :644-729
            const ix_t n = R_n(e);
            if (n == 0 || !nonempty) return false;
            m.c_pack += 1u;
            const ix_t from = m.last_idx + 1;
            log_append(m, n, m.term);
            note(m, RA_NOTE_WAL_APPEND, 0, from, from + n - 1, m.term);
            force = (R_flags(e) & RA_EVF_NOOP) != 0;
        } else if (type == RA_EV_WRITTEN) {                            // :730-735
            if (nonempty && !m.lrs_ok) { m.lrs = run_get(m, m_nruns(m) - 1).x; m.lrs_ok = 1; }
            if (!nonempty || !m.lrs_ok || R_term(e) != m.last_term || R_b(e) > m.last_idx || R_b(e) < m.lrs) return false;
            m.c_pack += 1u;
            m.lw_idx = R_b(e); m.lw_term = m.last_term;
            m.cold &= ~8u;
            quorum = chase = true;
        } else if (type == RA_EV_AER_REPLY) {                          // :522-561
            const u32 from = R_from(e);
            if (!(R_d(e) != 0 && R_term(e) == m.term && from < NMEM(*m.C))) return false;
            m.c_pack += 1u;
            CR_INC(m, CR_REPLY_OK);                                    // :528
            ixpair nm = peer_nm<MM>(m, from);
            if (R_b(e) > nm.y) m.cold &= ~8u;                          // a match index moves
            peer_nm_set<MM>(m, from, R_a(e) > nm.x ? R_a(e) : nm.x, R_b(e) > nm.y ? R_b(e) : nm.y);
            quorum = chase = true;
        } else return false;
        // exact shortcut: nothing evaluate_quorum reads has moved since it last ran in this step
        if (quorum && !(m.cold & 8u)) evaluate_quorum<MM>(m);
        // a chased {next_event, info, pipeline_rpcs}: one pass, the rest is deferred (contract 4)
#ifdef RA_LEAN_FAST
        if (rpc_pass<MM>(m, RP_PIPELINE, force, false) && chase)
#else
        if (rpc_pass<MM>(m, mode, force, false) && chase)
#endif
        { MT_SET(m.meta, 24, 1, 1); m.status |= RA_ST_PIPELINE_PENDING; }
        return true;
    }
    return false;
}
