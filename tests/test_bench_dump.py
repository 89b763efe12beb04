"""bench.py --dump-outputs: the arrays it writes hold exactly what the engine's caller reads back, stay under the
size ceiling, and are the same from run to run with the same arguments."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle_lib import Oracle
from ra_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _flooded_oracle(g=40, m=5, steps=30):
    o = Oracle(g, m, route_on_device=True)
    o.reset_empty()
    o.step([abi.ev_simple(o.row_of(i, 0), abi.EV_ELECTION_TIMEOUT) for i in range(g)])
    o.flood(steps, 1, 50, seed=7)
    return o


def _load(d):
    out = {os.path.basename(p)[:-4]: np.load(p) for p in glob.glob(os.path.join(d, "*.npy"))}
    assert out and all(a.dtype == np.float64 for a in out.values())
    return out


def _key(a, i, m):
    """RaRowState.key() rebuilt from the dumped arrays of row i"""
    nr, flags, nm = int(a["n_runs"][i]), int(a["flags"][i]), int(a["n_members"][i])
    sc = ("row", "role", "self_slot", "n_members", "leader_slot", "voted_for", "membership", "condition",
          "has_snapshot", "votes", "n_runs", "flags", "current_term", "commit_index", "last_applied", "pre_vote_token",
          "token_counter", "first_index", "last_index", "last_term", "last_written_index", "last_written_term",
          "snapshot_index", "snapshot_term")
    cond = ("cond_reply_term", "cond_reply_next_index", "cond_reply_last_index", "cond_reply_last_term")
    peers = ("next_index", "match_index", "commit_index_sent", "status", "voter")
    return (tuple(int(a[f][i]) for f in sc)
            + (tuple(int(x) for x in a["run_start"][i, :nr]), tuple(int(x) for x in a["run_term"][i, :nr]),
               tuple(int(a[f][i]) for f in cond) if flags & 2 else None,
               tuple(tuple(int(a["peer_" + f][i, p]) for f in peers) for p in range(nm))))


def test_dump_holds_every_row_exactly(tmp_path):
    o = _flooded_oracle()
    info = bench.dump_outputs(str(tmp_path), o)
    a = _load(tmp_path)
    assert info["rows"] == info["of_rows"] == o.n_rows and info["sample_seed"] is None
    assert a["row"].tolist() == list(range(o.n_rows))
    assert a["counters"].tolist() == list(o.counters().values())
    want = [r.key() for r in o.read_rows(range(o.n_rows))]
    assert [_key(a, i, o.n_members) for i in range(o.n_rows)] == want
    assert a["peer_next_index"].shape == (o.n_rows, o.n_members) and a["run_start"].shape == (o.n_rows, abi.RA_MAX_RUNS)
    # what key() does not compare is zero
    for i in range(o.n_rows):
        assert not a["run_start"][i, int(a["n_runs"][i]):].any()
    assert info["bytes"] == sum(os.path.getsize(p) for p in glob.glob(os.path.join(tmp_path, "*.npy")))


def test_dump_samples_rows_under_the_ceiling(tmp_path, monkeypatch):
    o = _flooded_oracle(g=200)
    monkeypatch.setattr(bench, "DUMP_BYTES", 2**20 + 50 * 8 * 300)    # room for about 300 rows
    info = [bench.dump_outputs(str(tmp_path / d), o) for d in ("a", "b")]
    assert info[0] == dict(info[1], dir=info[0]["dir"])
    assert 0 < info[0]["rows"] < o.n_rows and info[0]["sample_seed"] == bench.DUMP_SEED
    assert info[0]["bytes"] <= bench.DUMP_BYTES
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    ids = a["row"].astype(np.int64)
    assert len(ids) == info[0]["rows"] and (np.diff(ids) > 0).all() and ids[-1] < o.n_rows
    want = [r.key() for r in o.read_rows(ids.tolist())]
    assert [_key(a, i, o.n_members) for i in range(len(ids))] == want


@pytest.mark.gpu
def test_bench_dump_is_reproducible_and_counts_the_timed_steps(tmp_path):
    settle, warmup, steps = 20, 5, 7
    dumps = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--groups", "3000",
                            "--settle", str(settle), "--warmup", str(warmup), "--steps", str(steps),
                            "--no-e2e", "--no-cpu", "--no-extra-configs", "--no-latency", "--no-parity",
                            "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["dump"]["rows"] == 3000 * 5
        assert line["dump"]["bytes"] <= 64 * 10**6
        dumps.append(_load(tmp_path / d))
    a, b = dumps
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    names = [f for f, _ in abi.RaCounters._fields_]
    # the bootstrap step, then the untimed and the timed flood steps
    assert a["counters"][names.index("steps")] == 1 + settle + warmup + steps
    assert a["counters"][names.index("commits")] > 0
