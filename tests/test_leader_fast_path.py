"""The leader's fast path in the hot kernel (raft_logic.cuh `fast_event`: success replies, the quorum shortcut and
the pipeline pass `rpc_pass`) at the edges of its guards: the in-flight limit reached in the middle of a pass, peers
that are not `normal`, next indexes ahead of the replies, replies that do or do not move a match index in every order,
a commit index that advances more than once in a step, a fatal error raised inside the pass, 3 / 5 / 7 members, and
rows that cross 2^30 while the flood runs.

Every case is compared with the oracle (tests/oracle_lib.py) bit for bit: rows, RPC records, notes and counters.  CPU
tier: the device logic compiled for the host (tests/emu).  GPU tier: the kernels, through the C ABI.
"""
import ctypes as C
import itertools

import pytest

from emu_lib import Emu
from oracle_lib import Oracle
from ra_b200 import abi

LIM = 1 << 30


@pytest.fixture(autouse=True)
def _auto_mode(monkeypatch):
    monkeypatch.delenv("RA_STEP_WIDE", raising=False)


def _engine(*a, **kw):
    from ra_b200.engine import Engine
    return Engine(*a, **kw)


def _rows_bytes(b):
    arr = (abi.RaRowState * b.n_rows)()
    for i in range(b.n_rows):
        arr[i].row = i
    b._check(b._fn("read_rows")(b._h, arr, b.n_rows), "read_rows")
    return bytes(arr)


def _keys(out):
    msgs, notes = out
    return sorted(m.key() for m in msgs), [n.key() for n in notes]


# ---- floods: the in-flight limit and the batch size cut passes short -----------------------------------------
LIMITS = [dict(max_pipeline_count=1, max_aer_batch=1), dict(max_pipeline_count=2, max_aer_batch=1),
          dict(max_pipeline_count=2, max_aer_batch=3), dict(max_pipeline_count=1)]


def _flood(make, g, m, kw, steps, cmds, permille, base=None, term=1):
    o, e = Oracle(g, m, route_on_device=True, **kw), make(g, m, route_on_device=True, **kw)
    for b in (o, e):
        if base is None:
            b.reset_empty()
        else:
            rows = []
            for r in range(b.n_rows):
                s = abi.empty_row(r, b.n_groups, b.n_members)
                abi.set_log(s, [], last_written=(base, term), snapshot=(base, term))
                s.current_term = term
                s.commit_index = s.last_applied = base
                for p in range(b.n_members):
                    s.peers[p].next_index = base + 1
                rows.append(s)
            b.load_rows(rows)
        b.step([abi.ev_simple(b.row_of(i, 0), abi.EV_ELECTION_TIMEOUT) for i in range(g)])
    for part in (steps // 2, steps - steps // 2):
        o.flood(part, cmds, permille, seed=11, threads=1)
        e.flood(part, cmds, permille, seed=11)
    assert e.counters() == o.counters()
    assert o.counters()["commits"] > 0
    assert _rows_bytes(e) == _rows_bytes(o)
    return o.read_rows(range(o.n_rows))


@pytest.mark.parametrize("members", [3, 5, 7])
@pytest.mark.parametrize("kw", LIMITS)
@pytest.mark.parametrize("cmds", [1, 5])
def test_pipeline_limits_flood_emu(members, kw, cmds):
    _flood(Emu, 40, members, kw, 50, cmds, 30)


@pytest.mark.parametrize("members", [3, 5, 7])
def test_flood_crossing_the_narrow_limit_with_small_pipelines_emu(members):
    rows = _flood(Emu, 30, members, dict(max_pipeline_count=2, max_aer_batch=1), 90, 1, 20, base=LIM - 40, term=5)
    assert max(r.last_index for r in rows) >= LIM


# ---- closed-loop traces: loss (next_index ahead of the replies), duplicates, lagging fsync, elections ------------
TRACES = [
    # members, seed, pipeline limits, knobs
    (3, 3, dict(max_pipeline_count=1, max_aer_batch=1), dict(p_drop=0.08, p_cmd=0.9, max_cmd=4)),
    (5, 5, dict(max_pipeline_count=2, max_aer_batch=1), dict(p_drop=0.08, p_dup=0.05, p_cmd=0.9, max_cmd=6)),
    (5, 7, dict(max_pipeline_count=1), dict(p_withhold_written=0.3, p_delay=0.3, p_cmd=0.9, max_cmd=3)),
    (7, 9, dict(max_pipeline_count=2, max_aer_batch=2), dict(p_drop=0.05, p_timeout=0.03, p_adversarial=0.03, p_cmd=0.9)),
]


@pytest.mark.parametrize("m,seed,kw,knobs", TRACES)
def test_trace_with_small_pipelines_emu(m, seed, kw, knobs):
    import trace_gen
    batches = trace_gen.generate(lambda gg, mm: Oracle(gg, mm, **kw), 6, m, 180, seed, **knobs)
    assert trace_gen.replay(Emu(6, m, **kw), batches) == trace_gen.replay(Oracle(6, m, **kw), batches)


# ---- scripted leader steps --------------------------------------------------------------------------------------
T = 3          # leader's term
LAST = 20      # leader's last index; every entry has term T


def _leader_rows(b, peers, commit=10, written=LAST, first=1, snapshot=None):
    """Slot 0 of every group leads in term T with log first..LAST; peers = [(next, match, commit_sent, status), ...]
    for slots 1..; the followers hold the same log."""
    rows = []
    for r in range(b.n_rows):
        s = abi.empty_row(r, b.n_groups, b.n_members)
        abi.set_log(s, [(i, T) for i in range(first, LAST + 1)], last_written=(written, T), snapshot=snapshot)
        s.current_term = T
        s.voted_for = 0
        s.leader_slot = 0
        s.commit_index = s.last_applied = commit
        if s.self_slot == 0:
            s.role = abi.LEADER
            for p, (nx, mt, cs, st) in enumerate(peers, start=1):
                s.peers[p].next_index, s.peers[p].match_index = nx, mt
                s.peers[p].commit_index_sent, s.peers[p].status = cs, st
        rows.append(s)
    b.load_rows(rows)


def _script(b, peers, steps, **kw):
    _leader_rows(b, peers, **kw)
    out = [_keys(b.step([ev for g in range(b.n_groups) for ev in step(b, g)])) for step in steps]
    return out, _rows_bytes(b), b.counters()


def _both(make, m, peers, steps, **kw):
    o, e = Oracle(8, m), make(8, m)
    want, got = _script(o, peers, steps, **kw), _script(e, peers, steps, **kw)
    assert got[0] == want[0]
    assert got[1] == want[1]
    assert got[2] == want[2]
    return want


N = abi.PEER_NORMAL


def _replies(order, moves):
    """one success reply per peer slot in `order`; moves[slot]: the reply moves that peer's match index"""
    def step(b, g):
        return [abi.ev_aer_reply(b.row_of(g, 0), s, T, True, LAST + 1, LAST if moves[s] else 15, T) for s in order]
    return step


def _reply_steps(order, moves):
    """the replies of `order`, the first three followed by the leader's own written event in one step, the rest in the
    next step (a row takes at most RA_LOCAL_CAP = 4 host events a step)"""
    k = min(3, len(order))
    steps = [lambda b, g, o=order[:k]: _replies(o, moves)(b, g) + [abi.ev_written(b.row_of(g, 0), T, 16, LAST)]]
    if order[k:]:
        steps.append(_replies(order[k:], moves))
    return steps


@pytest.mark.parametrize("m", [3, 5, 7])
def test_replies_in_every_order_emu(m):
    """Replies that move a match index and replies that do not, in every order, followed by the leader's own written
    event in the same step (a row takes at most RA_LOCAL_CAP = 4 host events a step: the replies of peers beyond the
    third come in the next step): the commit index advances once the quorum has moved, then the pass sends it."""
    peers = [(LAST + 1, 15, 10, N)] * (m - 1)
    slots = list(range(1, m))
    orders = list(itertools.permutations(slots)) if m <= 5 else [tuple(slots), tuple(reversed(slots)), (2, 4, 1, 3, 6, 5)]
    for order in orders:
        for moves_mask in range(1 << (m - 1)):
            moves = {s: (moves_mask >> (s - 1)) & 1 for s in slots}
            _both(Emu, m, peers, _reply_steps(order, moves), written=15)


def test_commit_advances_twice_in_one_step_emu():
    """The commit index advances more than once in a step: 10 -> 12 (the first reply completes a quorum at the peers'
    old match index), -> 15, -> 20; each move re-opens the pass for the commit-only record."""
    peers = [(16, 12, 10, N)] * 4

    def step(b, g):
        r = b.row_of(g, 0)
        return [abi.ev_aer_reply(r, 1, T, True, 16, 15, T), abi.ev_aer_reply(r, 2, T, True, 16, 15, T),
                abi.ev_aer_reply(r, 1, T, True, LAST + 1, LAST, T), abi.ev_aer_reply(r, 3, T, True, LAST + 1, LAST, T)]
    out = _both(Emu, 5, peers, [step])
    commits = [n for n in out[0][0][1] if n[1] == abi.NOTE_COMMIT]
    assert len(commits) == 3 * 8                                # three COMMIT notes per group


@pytest.mark.parametrize("status", [abi.PEER_SENDING_SNAPSHOT, abi.PEER_SNAPSHOT_BACKOFF, abi.PEER_SUSPENDED,
                                    abi.PEER_DISCONNECTED])
def test_peer_not_normal_is_skipped_emu(status):
    peers = [(LAST + 1, LAST, 10, N), (15, 12, 10, status), (16, 15, 10, N), (LAST + 1, LAST, 10, N)]
    _both(Emu, 5, peers, [lambda b, g: [abi.ev_command(b.row_of(g, 0), 3)],
                          lambda b, g: [abi.ev_aer_reply(b.row_of(g, 0), 3, T, True, LAST + 4, LAST + 3, T)]])


def test_next_index_ahead_of_the_replies_emu():
    """next_index ran ahead (records in flight): in_flight = next - match - 1 reaches the limit for some peers and not
    for others within one pass."""
    peers = [(LAST + 1, 10, 10, N), (LAST + 1, 19, 10, N), (12, 11, 10, N), (LAST + 1, LAST, 10, N)]
    for kw in (dict(max_pipeline_count=1), dict(max_pipeline_count=2, max_aer_batch=1), dict(max_pipeline_count=9)):
        o, e = Oracle(8, 5, **kw), Emu(8, 5, **kw)
        steps = [lambda b, g: [abi.ev_command(b.row_of(g, 0), 2)],
                 lambda b, g: [abi.ev_aer_reply(b.row_of(g, 0), 1, T, True, 12, 11, T), abi.ev_command(b.row_of(g, 0), 1)]]
        assert _script(e, peers, steps) == _script(o, peers, steps)


def test_fatal_inside_the_pass_emu():
    """A peer whose next index is below the log with no snapshot to send: make_rpc_effect raises a fatal error in the
    middle of the pass; the peers after it in slot order get nothing."""
    peers = [(LAST + 1, LAST, 10, N), (3, 2, 10, N), (16, 15, 10, N), (16, 15, 10, N)]
    out = _both(Emu, 5, peers, [lambda b, g: [abi.ev_command(b.row_of(g, 0), 1)]], first=8, commit=10)
    assert out[2]["fatal_rows"] > 0


# ---- the kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("members", [3, 5, 7])
@pytest.mark.parametrize("kw", LIMITS)
def test_pipeline_limits_flood_gpu(members, kw):
    _flood(_engine, 3000, members, kw, 50, 3, 30)


@pytest.mark.gpu
@pytest.mark.parametrize("members", [3, 5, 7])
def test_flood_crossing_the_narrow_limit_with_small_pipelines_gpu(members):
    rows = _flood(_engine, 2000, members, dict(max_pipeline_count=2, max_aer_batch=1), 90, 1, 20, base=LIM - 40, term=5)
    assert max(r.last_index for r in rows) >= LIM


@pytest.mark.gpu
@pytest.mark.parametrize("m,seed,kw,knobs", TRACES)
def test_trace_with_small_pipelines_gpu(m, seed, kw, knobs):
    import trace_gen
    batches = trace_gen.generate(lambda gg, mm: Oracle(gg, mm, **kw), 6, m, 180, seed, **knobs)
    assert trace_gen.replay(_engine(6, m, **kw), batches) == trace_gen.replay(Oracle(6, m, **kw), batches)


def _scripted_leader_steps(make):
    for m in (3, 5, 7):
        peers = [(LAST + 1, 15, 10, N)] * (m - 1)
        slots = list(range(1, m))
        for order in (tuple(slots), tuple(reversed(slots))):
            for moves_mask in (0, 1, (1 << (m - 1)) - 1, 0b0101 & ((1 << (m - 1)) - 1)):
                moves = {s: (moves_mask >> (s - 1)) & 1 for s in slots}
                _both(make, m, peers, _reply_steps(order, moves), written=15)
    peers = [(LAST + 1, LAST, 10, N), (15, 12, 10, abi.PEER_SENDING_SNAPSHOT), (16, 15, 10, N), (LAST + 1, LAST, 10, N)]
    _both(make, 5, peers, [lambda b, g: [abi.ev_command(b.row_of(g, 0), 3)]])
    peers = [(LAST + 1, LAST, 10, N), (3, 2, 10, N), (16, 15, 10, N), (16, 15, 10, N)]
    out = _both(make, 5, peers, [lambda b, g: [abi.ev_command(b.row_of(g, 0), 1)]], first=8, commit=10)
    assert out[2]["fatal_rows"] > 0


def test_scripted_leader_steps_emu():
    """the scripts of the GPU case below, through the emulation"""
    _scripted_leader_steps(Emu)


@pytest.mark.gpu
def test_scripted_leader_steps_gpu():
    _scripted_leader_steps(_engine)
