"""Per-warp timeline of the hot kernel, without Nsight: where a flood step's time goes.

Builds the measurement variant of the engine (`-DRA_WARP_TIMELINE`, next to the default build, as
tools/build_variant.sh does), runs the bench-shaped flood (100k groups x 5, 1 % election timeouts per step, after
settling) and reads back one record per warp of each timed hot-kernel launch: tile, SM, %globaltimer at entry,
after the per-row inputs landed, after the event loop and at exit, whether all 32 rows are leaders, planes consumed.

    python tools/warp_timeline.py [--so LIB] [--extra -DFOO ...] [--steps 5] [--out summary.txt]

Prints, per timed step and as the median over steps: the kernel span (first warp entry .. last warp exit), leader-warp
lifetime p50 / p99, when the last leader warp starts and ends, when the follower phase starts and ends, and how many
leader warps started only after the first leader warp had retired (a second round on the SMs).  The probes add a
few instructions per warp, so absolute times are those of the measurement build, not of the default one.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REC = np.dtype([("t_entry", "<u8"), ("t_inputs", "<u8"), ("t_loop", "<u8"), ("t_exit", "<u8"),
                ("tile", "<u4"), ("info", "<u4"), ("pad", "<u4", 2)])
assert REC.itemsize == 48


def build(name: str, extra) -> str:
    subprocess.check_call(["bash", os.path.join(ROOT, "tools", "build_variant.sh"), name, "-DRA_WARP_TIMELINE"] + list(extra))
    return os.path.join(ROOT, "ra_b200", "csrc", "libra_engine_%s.so" % name)


def pct(a, q):
    return float(np.percentile(a, q)) if len(a) else float("nan")


def summarize(r) -> dict:
    r = r[r["t_exit"] != 0]
    t0 = int(r["t_entry"].min())
    ent = (r["t_entry"] - t0) / 1e3                       # us from the first warp's entry
    ext = (r["t_exit"] - t0) / 1e3
    inp = (r["t_inputs"] - r["t_entry"]) / 1e3
    loop = (r["t_loop"] - r["t_inputs"]) / 1e3
    life = ext - ent
    lead = ((r["info"] >> 16) & 1) == 1
    planes = r["info"] >> 24
    smid = r["info"] & 0xffff
    span = float(ext.max())
    L, F = lead, ~lead
    first_leader_exit = float(ext[L].min()) if L.any() else float("nan")
    return {
        "warps": int(len(r)), "leader_warps": int(L.sum()), "sms": int(len(np.unique(smid))),
        "span_us": span,
        "leader_life_p50_us": pct(life[L], 50), "leader_life_p99_us": pct(life[L], 99),
        "leader_inputs_p50_us": pct(inp[L], 50), "leader_loop_p50_us": pct(loop[L], 50),
        "leader_planes_p50": pct(planes[L], 50),
        "last_leader_start_us": float(ent[L].max()) if L.any() else float("nan"),
        "last_leader_end_us": float(ext[L].max()) if L.any() else float("nan"),
        "first_leader_end_us": first_leader_exit,
        "leader_second_round": int((ent[L] >= first_leader_exit).sum()),
        "follower_life_p50_us": pct(life[F], 50), "follower_planes_p50": pct(planes[F], 50),
        "follower_start_us": float(ent[F].min()) if F.any() else float("nan"),
        "follower_start_p50_us": pct(ent[F], 50),
        "follower_end_us": float(ext[F].max()) if F.any() else float("nan"),
    }


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--so", help="a library built with -DRA_WARP_TIMELINE (default: build one)")
    ap.add_argument("--name", default="timeline", help="variant name of the library this builds")
    ap.add_argument("--extra", nargs="*", default=[], help="further -D switches for the build")
    ap.add_argument("--groups", type=int, default=100_000)
    ap.add_argument("--members", type=int, default=5)
    ap.add_argument("--permille", type=int, default=10)
    ap.add_argument("--settle", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=5, help="timed steps, one hot-kernel launch each")
    ap.add_argument("--seed", type=int, default=0xA00)
    ap.add_argument("--out", help="also write the summary here")
    ap.add_argument("--raw", help="write the records of the last timed step here (.npy)")
    a = ap.parse_args()

    so = a.so or build(a.name, a.extra)
    os.environ["RA_ENGINE_SO"] = os.path.abspath(so)
    sys.path.insert(0, ROOT)
    from ra_b200 import abi
    from ra_b200.engine import Engine, lib

    L = lib()
    try:
        f = L.ra_debug_warp_timeline
    except AttributeError:
        sys.exit("%s was not built with -DRA_WARP_TIMELINE" % so)
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_int]

    e = Engine(a.groups, a.members, route_on_device=True)
    e.reset_empty()
    e.step([abi.ev_simple(e.row_of(g, 0), abi.EV_ELECTION_TIMEOUT) for g in range(a.groups)])
    e.flood(a.settle, 1, a.permille, seed=a.seed)
    e.flood(a.warmup, 1, a.permille, seed=a.seed)
    n = C.c_size_t(0)
    e._check(f(e._h, None, 0, C.byref(n), 1), "warp_timeline")
    cap = (a.groups * a.members + 31) // 32
    buf = np.zeros(cap, dtype=REC)
    rows = []
    for _ in range(a.steps):
        e.flood(1, 1, a.permille, seed=a.seed)
        e._check(f(e._h, buf.ctypes.data, cap, C.byref(n), 1), "warp_timeline")
        rec = buf[: n.value].copy()
        rows.append(summarize(rec))
    if a.raw:
        np.save(a.raw, rec)
    lines = ["# warp timeline: %d groups x %d, %d permille election timeouts, %s" % (a.groups, a.members, a.permille, os.path.basename(so))]
    keys = list(rows[0].keys())
    for i, s in enumerate(rows):
        lines.append("step %d: " % i + " ".join("%s=%.2f" % (k, v) if isinstance(v, float) else "%s=%d" % (k, v) for k, v in s.items()))
    med = {k: float(np.median([s[k] for s in rows])) for k in keys}
    lines.append("median: " + json.dumps({k: round(v, 2) for k, v in med.items()}))
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
