#!/usr/bin/env python3
"""bench.py -- candidate 3-LUT tuples/s of the `--lut` search path (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--gates n]
                  [--dump-outputs DIR]

A STEP is one pass of the hot path -- search_5lut followed by search_7lut (lut.c:553,593) -- over a
batch of synthetic search states shaped like the ones `sboxgates --lut -o 0 rijndael.txt` presents
(BASELINE.json configs[1]): target = output bit 0 of the Rijndael S-box, n gates = 8 input bits +
random 3-LUTs of earlier gates (a real seeded run of that command ends with 31 LUTs, i.e. 39 gates,
profiles/r01_dropin_runs.md, hence the default n = 40), masks as mux recursion of depth 0..3 leaves
them (sboxgates.c:478,483), the selector bits excluded (lut.c:177-185).  No state has a 5-LUT
match, and at most a late 7-LUT one, so every step is a full sweep.

Units (SURVEY.md section 8d): T-unit = one gate combination through inbits-reject + feasibility;
C-unit = one candidate decomposition decided, counted as the reference enumerates them (2,560 per
feasible 5-tuple, 70 x 65,536 per listed 7-tuple) even though the kernels decide many at once from
a per-tuple summary.  value = (T + C) / s; both are also reported separately.

N > 1 (torchrun, one rank per GPU): the search states of a step are independent (in the program
they are the 16 mux branches of create_circuit, the 8 output bits of -o -1 and the -i iterations),
so every rank takes `--batch` states of a step of N x `--batch` -- its own sbg_search_batch call --
and the ranks exchange only the result keys (one all-gather, inside the timed region): weak scaling.
The same line carries a `sharded` record: ONE search of a large state (n = 96, 128) sharded over the
ranks' GPUs across the tuple space (work items dealt round-robin; the 7-LUT hit lists all-gathered
and merged on the devices, one all-reduce(MIN) per search phase), with the one-GPU time of the same
search beside it and the results compared in the run -- strong scaling of north_star's partition.
Further records on one GPU: `replay` (recorded real calls of seeded reference runs through the C
ABI, results asserted), `graph` (wall-clock to graph: the drop-in CLI on BASELINE.json configs[1]).

--dump-outputs DIR writes the result structs the last timed step returned (sbg_search_batch, one row
per search state) as float64 arrays: DIR/r5.npy and DIR/r7.npy (search_5lut / search_7lut, columns
RESULT_COLUMNS) and DIR/node.npy (NODE_COLUMNS); 64-bit keys are split into two exact 32-bit halves.
The states of a step depend only on --gates, --batch and the step's number (seed 1000 + s, warm-up
steps counted), so
the same arguments give the same inputs in every run and two builds can be compared file by file.
With N > 1 every rank writes its own states' results, with the suffix _rank<r>.

--impl reference times the reference's own object code (oracle/_ref/libsbgref.so, built from the
unmodified sources; the oracle port if that is absent) on the host cores, one process per core, each
on a bounded sample of the same workload: the same states restricted to their first n' gates.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "candidate 3-LUT tuples/sec on rijndael.txt --lut (T-units + C-units per second)"
UNIT = "tuples/s"
C_PER_5 = 10 * 256
C_PER_7 = 70 * 65536
BYTES_T5, BYTES_T7, BYTES_C = 160, 224, 160   # SURVEY.md section 8d: algorithmic bytes per unit


# ------------------------------------------------------------------------------------------------
# workload (self-contained: the product side must not import tests/ or oracle/)

def _input_table(bit):
    w = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        if (p >> bit) & 1:
            w[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return w


def _lut(func, a, b, c):
    full = np.uint64(0xFFFFFFFFFFFFFFFF)
    out = np.zeros(4, dtype=np.uint64)
    for m in range(8):
        if (func >> m) & 1:
            out |= (a if m & 4 else a ^ full) & (b if m & 2 else b ^ full) & (c if m & 1 else c ^ full)
    return out


def _rijndael_bit(bit):
    def mul(a, b):
        r = 0
        while b:
            if b & 1:
                r ^= a
            a <<= 1
            if a & 0x100:
                a ^= 0x11B
            b >>= 1
        return r
    inv = [0] * 256
    for a in range(1, 256):
        for b in range(1, 256):
            if mul(a, b) == 1:
                inv[a] = b
                break
    w = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        x = inv[p]
        y = x
        for s in (1, 2, 3, 4):
            y ^= ((x << s) | (x >> (8 - s))) & 0xFF
        if ((y ^ 0x63) >> bit) & 1:
            w[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return w


def _mux_mask(fixed):
    w = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        if all(((p >> b) & 1) == v for b, v in fixed):
            w[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return w


def _state(n, seed):
    rs = np.random.RandomState(seed)
    tabs = [_input_table(i) for i in range(8)]
    while len(tabs) < n:
        i, j, k = rs.choice(len(tabs), 3, replace=False)
        tabs.append(_lut(int(rs.randint(1, 255)), tabs[i], tabs[j], tabs[k]))
    return np.stack(tabs[:n]).astype(np.uint64)


def _orders(rs):
    return bytes(rs.permutation(256).astype(np.uint8)), bytes(rs.permutation(256).astype(np.uint8)), \
        bytes(rs.permutation(256).astype(np.uint8))


def build_batch(n, batch, step_seed):
    """`batch` search states; masks cycle through mux depth 0..3 (popcount 256, 128, 64, 32)."""
    target = _rijndael_bit(0)
    rs = np.random.RandomState(step_seed)
    out = []
    for i in range(batch):
        depth = i % 4
        bits = rs.choice(8, depth, replace=False)
        fixed = [(int(b), int(rs.randint(0, 2))) for b in bits]
        o5, oo, om = _orders(rs)
        out.append(dict(tables=_state(n, int(rs.randint(1 << 30))), target=target,
                        mask=_mux_mask(fixed), inbits=[b for b, _ in fixed], order5=o5, outer=oo,
                        middle=om))
    return out


RESULT_COLUMNS = ("found", "ordering", "pos_outer", "pos_middle", "func_outer", "func_middle",
                  "func_inner", "inner_seen", "gate0", "gate1", "gate2", "gate3", "gate4", "gate5",
                  "gate6", "stale_outer", "index", "key_hi", "key_lo", "tuples_feasible",
                  "tuples_swept")
NODE_COLUMNS = ("found_stage", "gate0", "gate1", "gate2", "func3", "seen3", "key3_hi", "key3_lo")


def _result_row(r):
    return [r.found, r.ordering, r.pos_outer, r.pos_middle, r.func_outer, r.func_middle,
            r.func_inner, r.inner_seen] + list(r.gates) + [
        r.stale_outer, r.index, r.key >> 32, r.key & 0xFFFFFFFF, r.tuples_feasible, r.tuples_swept]


def dump_outputs(out_dir, results, suffix=""):
    """The SbgNodeResult structs of one sbg_search_batch call as float64 arrays (every field is an
    integer below 2**53 once the keys are split, so the values are exact)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"r5": [_result_row(r.r5) for r in results], "r7": [_result_row(r.r7) for r in results],
              "node": [[r.found_stage] + list(r.gates3) + [r.func3, r.seen3, r.key3 >> 32,
                                                           r.key3 & 0xFFFFFFFF] for r in results]}
    for name, rows in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.array(rows, dtype=np.float64))


def units_of(n, r5, r7):
    """(T, C) units of one state from the two results, as the reference would have enumerated."""
    t = math.comb(n, 5) if not r5.found else int(r5.index) + 1
    c = int(r5.tuples_feasible) * C_PER_5
    if r5.found:   # candidates of the matching tuple only (earlier feasible tuples are not counted)
        c = r5.ordering * 256 + r5.pos_outer + 1
    t7 = int(r7.tuples_swept)      # this rank's share; summed over ranks by the caller
    if r7.found:
        c += int(r7.index) * C_PER_7 + r7.ordering * 65536 + r7.pos_outer * 256 + r7.pos_middle + 1
    else:
        c += int(r7.tuples_feasible) * C_PER_7
    return t, t7, c


# ------------------------------------------------------------------------------------------------
# clocks

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4)
                          if r[3 + i].lower().startswith("active")})
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own object code on the host cores

def _cpu_worker(args):
    """One host core: the reference's search_5lut + search_7lut on samples (the first n' gates of a
    workload state), one after the other until the deadline.  Returns (seconds, T-units, C-units,
    samples done); the units of a sample are counted only when it completed."""
    kind, samples, deadline_s = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _support as S
    if kind == "reference":
        S.ref_lib()
    t_units = c_units = done = 0
    elapsed = 0.0
    t_start = time.perf_counter()
    for tables, target, mask, inbits, seed in samples:
        rng = S.OrcRng.from_seed(seed)
        t0 = time.perf_counter()
        if kind == "reference":
            f5, r5, _ = S.ref_search(5, tables, target, mask, inbits, rng)
            f7, r7, _ = S.ref_search(7, tables, target, mask, inbits, rng)
        else:
            f5, r5, _ = S.oracle_search(5, tables, target, mask, inbits, rng)
            f7, r7, _ = S.oracle_search(7, tables, target, mask, inbits, rng)
        elapsed += time.perf_counter() - t0
        # Unit accounting (outside the timed region) with the oracle's counters: same semantics.
        _, _, s5 = S.oracle_search(5, tables, target, mask, inbits, S.OrcRng.from_seed(seed))
        lst, s7 = S.oracle_filter7(tables, target, mask, inbits)
        t_units += int(s5.tuples_filtered) + int(s7.tuples_filtered)
        c_units += int(s5.candidates)
        if f7:
            rng2 = S.OrcRng.from_seed(seed)
            S.oracle_search(5, tables, target, mask, inbits, rng2)
            _, _, s7b = S.oracle_search(7, tables, target, mask, inbits, rng2)
            c_units += int(s7b.candidates)
        else:
            c_units += len(lst) * C_PER_7
        done += 1
        if time.perf_counter() - t_start > deadline_s:
            break
    return elapsed, t_units, c_units, done


def _pick_sample_gates(state, budget_s):
    """Largest n' whose reference run is expected to fit the budget: about 1e7 filter tuples/s and
    0.8 s per listed 7-tuple (BASELINE.md section 2), using the oracle's fast phase-1 count."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _support as S
    best = 9
    for npr in range(9, min(30, state["tables"].shape[0]) + 1):  # C(30,7) = 2.0e6 filter tuples
        lst, _ = S.oracle_filter7(state["tables"][:npr], state["target"], state["mask"],
                                  state["inbits"])
        est = math.comb(npr, 7) / 1e7 + math.comb(npr, 5) / 5e6 + 0.8 * len(lst)
        if est > budget_s:
            break
        best = npr
    return best


def cpu_arm(n, batch, seed, budget_s=12.0, cores=None):
    """Times the reference (or the oracle port) on a bounded sample, one process per host core.
    Every process works through samples of about budget_s / 4 each until budget_s has passed and
    reports its own throughput; the arm's value is the sum over the processes (all cores busy for
    the whole budget, no process waiting for the slowest)."""
    import multiprocessing as mp
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libsbgref.so")) \
        else "port"
    cores = cores or os.cpu_count() or 1
    states = build_batch(n, max(batch, 8), seed)
    per_sample = max(budget_s / 4.0, 0.05)
    sized = []
    npr_used = []
    for st in states:
        npr = _pick_sample_gates(st, per_sample)
        npr_used.append(npr)
        sized.append((st["tables"][:npr].copy(), st["target"], st["mask"],
                      [b for b in st["inbits"] if b < npr]))
    jobs = []
    for i in range(cores):
        samples = [sized[(i + k) % len(sized)] + (77 + i * 31 + k,) for k in range(16)]
        jobs.append((kind, samples, budget_s))
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    t_rate = sum(r[1] / r[0] for r in res if r[0] > 0)
    c_rate = sum(r[2] / r[0] for r in res if r[0] > 0)
    busy = max(r[0] for r in res)
    return {"value": t_rate + c_rate, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%d processes, each the reference's search_5lut+search_7lut on the first "
                      "n'=%s gates of workload states (n=%d), one sample after the other for %.1f s; "
                      "%d samples, %.3g T-units + %.3g C-units; value = sum of the processes' own "
                      "throughputs" % (cores, sorted(set(npr_used)), n, budget_s,
                                       sum(r[3] for r in res), sum(r[1] for r in res),
                                       sum(r[2] for r in res)),
            "t_units_per_s": t_rate, "c_units_per_s": c_rate, "seconds": busy,
            "wall_seconds": wall}


# ------------------------------------------------------------------------------------------------
# recorded real calls (tests/golden/run_*.bin; layout: oracle/ref_glue.c, SBGREF_RECORDER)

def read_recorded_calls(path):
    import struct
    data = open(path, "rb").read()
    off, out = 0, []
    while off < len(data):
        magic, n = struct.unpack_from("<II", data, off)
        off += 8
        which = {0x35474253: 5, 0x37474253: 7}[magic]
        tables = np.frombuffer(data, dtype="<u8", count=4 * n, offset=off).reshape(n, 4).copy()
        off += 32 * n
        target = np.frombuffer(data, dtype="<u8", count=4, offset=off).copy()
        mask = np.frombuffer(data, dtype="<u8", count=4, offset=off + 32).copy()
        off += 64
        inbits = []
        for b in np.frombuffer(data, dtype=np.int8, count=8, offset=off):   # -1 terminated
            if b == -1:
                break
            inbits.append(int(b))
        off += 8
        rng_s = list(struct.unpack_from("<16Q", data, off))
        off += 128
        rng_p, found = struct.unpack_from("<II", data, off)
        off += 8
        ret = list(struct.unpack_from("<10H", data, off))
        off += 20
        draws, ns = struct.unpack_from("<QQ", data, off)
        off += 16
        out.append(dict(which=which, tables=tables, target=target, mask=mask, inbits=inbits,
                        rng_s=rng_s, rng_p=rng_p, found=bool(found), ret=ret, ns=ns))
    return out


def replay_record(eng, sb):
    """Recorded real calls of seeded reference runs through the C ABI: results must equal the
    recorded ones (asserted), throughput in the units the reference spent on them."""
    from sboxgates_b200.rng import Xorshift1024
    out = {}
    for name in ("run_rijndael_seed1.bin", "run_sodark_seed1.bin", "run_des_s1_seed1.bin"):
        path = os.path.join(ROOT, "tests", "golden", name)
        if not os.path.exists(path) or os.path.getsize(path) == 0:
            continue
        calls = read_recorded_calls(path)
        for c in calls[:3]:   # warm-up
            fn = sb.search_5lut if c["which"] == 5 else sb.search_7lut
            fn(eng, c["tables"], c["target"], c["mask"], c["inbits"],
               Xorshift1024.from_state(c["rng_s"], c["rng_p"]))
        t_units = c_units = 0
        t0 = time.perf_counter()
        for c in calls:
            fn = sb.search_5lut if c["which"] == 5 else sb.search_7lut
            r = fn(eng, c["tables"], c["target"], c["mask"], c["inbits"],
                   Xorshift1024.from_state(c["rng_s"], c["rng_p"]))
            if (r.found, r.ret) != (c["found"], c["ret"]):
                raise SystemExit("replay of %s: result differs from the recorded reference call" % name)
            n = c["tables"].shape[0]
            if c["which"] == 5:
                t_units += (int(r.index) + 1) if r.found else math.comb(n, 5)
                c_units += (r.ordering * 256 + r.pos_outer + 1) if r.found \
                    else int(r.tuples_feasible) * C_PER_5
            else:
                t_units += int(r.tuples_swept)
                c_units += (int(r.index) * C_PER_7 + r.ordering * 65536 + r.pos_outer * 256
                            + r.pos_middle + 1) if r.found else int(r.tuples_feasible) * C_PER_7
        secs = time.perf_counter() - t0
        ref_secs = sum(c["ns"] for c in calls) * 1e-9
        out[name] = {"calls": len(calls), "seconds": secs, "us_per_call": 1e6 * secs / len(calls),
                     "units_per_s": (t_units + c_units) / secs, "t_units": t_units,
                     "c_units": c_units, "reference_seconds_when_recorded": ref_secs,
                     "parity": True}
    if out:
        out["note"] = ("through the Python mirror of the two-function interface (lut.py): each call "
                       "includes 256 / 512 draws of the Python xorshift1024 and the ctypes marshalling "
                       "of the state, which dominate the time per call; the `graph` record times the "
                       "same path from C")
    return out


# ------------------------------------------------------------------------------------------------
# wall-clock to graph: the drop-in CLI on BASELINE.json configs[1]

def graph_record():
    """`sboxgates_gpu -l -o 0 rijndael.txt` (the reference's own host code + our shim and library)
    under the two committed seeds: wall seconds, what the shim reports about itself, the file
    written, and an independent functional check of that file (sboxgates_b200/graph.py)."""
    import glob
    import re
    import tempfile
    from sboxgates_b200 import graph as G
    exe = os.path.join(ROOT, "oracle", "_ref", "sboxgates_gpu")
    sbox_path = os.path.join(ROOT, "oracle", "_ref", "sboxes", "rijndael.txt")
    if not (os.path.exists(exe) and os.path.exists(sbox_path)):
        return {"unavailable": "oracle/_ref/sboxgates_gpu not built (needs /root/reference at build time)"}
    sbox, _ = G.load_sbox(sbox_path)
    runs = []
    for seed in ("seed1", "seed2"):
        with tempfile.TemporaryDirectory() as tmp:
            env = dict(os.environ, SBG_SEEDFILE=os.path.join(ROOT, "tests", "golden", seed + ".bin"),
                       SBG_SHIM_STATS="1")
            t0 = time.perf_counter()
            res = subprocess.run([exe, "-l", "-o", "0", sbox_path], cwd=tmp, env=env,
                                 capture_output=True, text=True, timeout=600)
            wall = time.perf_counter() - t0
            files = sorted(os.path.basename(p) for p in glob.glob(os.path.join(tmp, "*.xml")))
            run = {"seed": seed, "wall_s": wall, "rc": res.returncode, "xml": files[-1] if files else None}
            if files:
                g = G.load_graph(os.path.join(tmp, files[-1]))
                run["verified_output_bits"] = G.verify_graph(g, sbox, require_bits=[0])
                run["luts"] = g.num_luts
        m = re.search(r"start-up \(sbg_create\) ([0-9.]+) s", res.stderr)
        if m:
            run["startup_s"] = float(m.group(1))
        m = re.search(r"lut_search: (\d+) calls ([0-9.]+) s \(ended at: 3-LUT (\d+), 5-LUT (\d+), "
                      r"7-LUT (\d+), nothing (\d+)\)", res.stderr)
        if m:
            calls, secs = int(m.group(1)), float(m.group(2))
            run.update({"lut_search_calls": calls, "lut_search_s": secs,
                        "us_per_call_without_startup": 1e6 * (secs - run.get("startup_s", 0.0))
                        / max(calls, 1),
                        "ended_at": {"lut3": int(m.group(3)), "lut5": int(m.group(4)),
                                     "lut7": int(m.group(5)), "nothing": int(m.group(6))}})
        m = re.search(r"(\d+) kernel launches", res.stderr)
        if m:
            run["kernel_launches"] = int(m.group(1))
        runs.append(run)
    return {"command": "sboxgates_gpu -l -o 0 rijndael.txt (reference host objects + node shim + "
                       "libsboxgates_b200.so)", "runs": runs,
            "note": "the reference itself does not finish this configuration in an hour "
                    "(BASELINE.md section 2)"}


# ------------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--gates", type=int, default=40)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="only the headline measurement (no sharded / graph / replay records)")
    ap.add_argument("--sharded-gates", default="64h,96,128",
                    help="state sizes of the tuple-space sharding record; suffix h = one mux level "
                         "deep (128 masked positions) instead of the full mask")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_states = args.batch * world
    config = {"workload": "rijndael.txt --lut -o 0 shaped: %d states/step, n=%d gates, target = "
                          "S-box bit 0, mux masks of depth 0-3, full no-match sweeps of "
                          "search_5lut+search_7lut" % (n_states, args.gates),
              "gates": args.gates, "states_per_step": n_states, "states_per_gpu": args.batch,
              "parallelism": "1 GPU" if world == 1 else (
                  "%d ranks x %d independent search states per step; result keys exchanged with one "
                  "all-gather inside the timed region" % (world, args.batch)),
              "l2": "a 256 MiB buffer is overwritten between steps (L2 flush); every step uses new states"}

    if args.impl == "reference":
        if rank != 0:
            return
        t0 = time.perf_counter()
        vals = []
        for s in range(max(1, min(args.steps, 2))):
            vals.append(cpu_arm(args.gates, args.batch, 1000 + s, budget_s=10.0))
        best = max(vals, key=lambda v: v["value"])
        line = {"impl": "reference", "metric": METRIC, "value": best["value"], "unit": UNIT,
                "n_gpus": args.gpus, "steps": len(vals), "warmup": 0,
                "ms_per_step": 1e3 * best["seconds"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u32 bitwise", "data": "synthetic", "config": config,
                "cpu_baseline": best,
                "e2e": {"value": best["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "seconds_total": time.perf_counter() - t0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import sboxgates_b200 as sb
    from sboxgates_b200.distributed import DistributedLutSearch

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = sb.LutEngine(local_rank)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    n, B = args.gates, args.batch
    total_steps = args.warmup + args.steps
    # this rank's states of every step: rank r takes states r*B .. r*B+B-1 of the step's n_states
    batches = [build_batch(n, n_states, 1000 + s)[rank * B:(rank + 1) * B] for s in range(total_steps)]

    def jobs_of(states):
        return [dict(slot=i, order5=st["order5"], outer=st["outer"], middle=st["middle"])
                for i, st in enumerate(states)]

    def stage(states):
        for i, st in enumerate(states):
            eng.stage(i, st["tables"], st["target"], st["mask"], st["inbits"])

    # The timed loops go through the same two C calls (sbg_stage_problem, sbg_search_batch) with the
    # Python-side marshalling -- numpy arrays to pointers, job structs -- done once, up front, and
    # the unit accounting done after the loop: neither is part of the path.
    prep_states = [[eng.prepare_state(st["tables"], st["target"], st["mask"], st["inbits"])
                    for st in states] for states in batches]
    prep_jobs = [eng.prepare_jobs(jobs_of(states)) for states in batches]

    def stage_step(s):
        for i, p in enumerate(prep_states[s]):
            eng.stage_prepared(i, p)

    step_keys = []

    def exchange_keys():
        """Every rank ends up knowing every state's result, as the host program would: ONE
        all-gather of the result keys of all the steps run since the last exchange (the states are
        independent, nothing needs a result before the end)."""
        if world > 1 and step_keys:
            flat = [k for ks in step_keys for k in ks]
            mine = torch.tensor(flat, dtype=torch.int64).cuda()
            allk = torch.empty(world * len(flat), dtype=torch.int64, device="cuda")
            dist.all_gather_into_tensor(allk, mine)
            torch.cuda.synchronize()
        step_keys.clear()

    def account(res, acc):
        """Result structs of one step -> keys for the exchange, units for the metric.  (One step =
        every state's search_5lut followed by search_7lut (lut.c:553,593) through ONE
        sbg_search_batch call: the states' chains overlap on the device.)"""
        keys = []
        for r in res:
            keys += [int(r.r5.key) & 0x7FFFFFFFFFFFFFFF, int(r.r7.key) & 0x7FFFFFFFFFFFFFFF]
            if acc is not None:
                t5, t7, c = units_of(n, r.r5, r.r7)
                acc["T5"] += t5
                acc["T7"] += t7
                acc["C"] += c
        step_keys.append(keys)

    def timed(resident):
        acc = {"T5": 0, "T7": 0, "C": 0}
        sampler = ClockSampler(local_rank)   # samples every 20 ms from the warm-up on
        sampler.start()
        for s in range(args.warmup):
            stage_step(s)
            account(eng.search_batch_prepared(prep_jobs[s]), None)
        exchange_keys()
        launches0 = eng.launches
        tr0 = eng.transfer_stats()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(args.steps)]
        barrier()
        t_wall = 0.0
        results = []
        for s in range(args.steps):
            k = args.warmup + s
            if resident:   # inputs resident in HBM before the timed region of this step starts
                stage_step(k)
            flush.fill_(s & 0xFF)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev[s][0].record(stream)
            if not resident:   # host tables -> device inside the timed region
                stage_step(k)
            results.append(eng.search_batch_prepared(prep_jobs[k]))   # returns with the results read
            ev[s][1].record(stream)
            torch.cuda.synchronize()
            t_wall += time.perf_counter() - t0
        for res in results:
            account(res, acc)
        t_gather0 = time.perf_counter()
        exchange_keys()
        gather_ms = 1e3 * (time.perf_counter() - t_gather0)
        clocks = sampler.stop()
        barrier()
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        # results are read from mapped memory while the stream is still draining, so the host's
        # clock and the stream's events bracket slightly different things: report the larger
        compute_ms = max(dev_ms, 1e3 * t_wall)
        own_ms = compute_ms + gather_ms
        ranks_ms, ranks_compute = [own_ms], [compute_ms]
        if world > 1:
            t = torch.tensor([own_ms, compute_ms], dtype=torch.float64, device="cuda")
            allt = torch.empty(2 * world, dtype=torch.float64, device="cuda")
            dist.all_gather_into_tensor(allt, t)
            ranks_ms, ranks_compute = allt.tolist()[0::2], allt.tolist()[1::2]
            u = torch.tensor([acc["T5"], acc["T7"], acc["C"]], dtype=torch.int64, device="cuda")
            dist.all_reduce(u, op=dist.ReduceOp.SUM)
            acc["T5"], acc["T7"], acc["C"] = (int(x) for x in u.tolist())
        acc["launches"] = eng.launches - launches0
        tr1 = eng.transfer_stats()
        acc["h2d"], acc["d2h"] = tr1[0] - tr0[0], tr1[1] - tr0[1]
        acc["gather_ms"] = gather_ms
        acc["ranks_compute"] = ranks_compute
        return max(ranks_ms), ranks_ms, acc, clocks, results[-1]

    ms_res, ranks_res, acc_res, clocks, last_results = timed(resident=True)
    ms_e2e, ranks_e2e, acc_e2e, _, _ = timed(resident=False)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_results, "_rank%d" % rank if world > 1 else "")

    # kernel families in isolation (one state at a time, CUDA events between the kernels): the
    # dominant kernel's launch durations for the roofline; not part of `value`
    eng.set_timing(True)
    fam = {"ms5": 0.0, "ms_filter": 0.0, "ms_order": 0.0, "ms_decomp": 0.0}
    by_depth = {k: [0.0] * 4 for k in ("ms5", "ms_filter", "ms_decomp")}   # mux depth 0..3 of the state
    t7_iso = 0
    for s in range(args.steps):
        states = batches[args.warmup + s]
        stage(states)
        flush.fill_(s & 0xFF)
        torch.cuda.synchronize()
        for i, j in enumerate(jobs_of(states)):
            r = eng.search_batch([j])[0]
            t7_iso += int(r.r7.tuples_swept)
            for k, w in (("ms5", 0), ("ms_filter", 1), ("ms_order", 2), ("ms_decomp", 3)):
                fam[k] += eng.kernel_ms(w)
                if k in by_depth:
                    by_depth[k][i % 4] += eng.kernel_ms(w)
    eng.set_timing(False)
    alu_peak = eng.alu_peak()
    props = torch.cuda.get_device_properties(local_rank)

    extras = {}
    if not args.no_extras:
        extras["sharded"] = sharded_record(eng, sb, DistributedLutSearch, args, rank, world)
    if rank == 0:
        units = acc_res["T5"] + acc_res["T7"] + acc_res["C"]
        value = units / (ms_res * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        filt_s = fam["ms_filter"] * 1e-3
        hbm_equiv = t7_iso * BYTES_T7 / max(filt_s, 1e-12) / 1e9
        # warp instructions of the dominant kernel: counted by ncu on these very states
        # (scripts/ncu_inst_counts.sh writes the table; see profiles/README.md)
        inst = alu_inst = None
        inst_src = os.path.join(ROOT, "profiles", "r02_filter_inst_counts.json")
        try:
            tab = json.load(open(inst_src))
            if tab.get("gates") == n and tab.get("batch") == B:
                seeds = [str(1000 + args.warmup + s) for s in range(args.steps)]
                if all(k in tab["per_step_seed"] for k in seeds):
                    inst = float(sum(sum(tab["per_step_seed"][k]) for k in seeds))
                    alu_inst = float(sum(sum(tab["alu_pipe_inst"][k]) for k in seeds))
        except (OSError, ValueError, KeyError):
            pass
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))[
                "filter7_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        launches_filter = args.steps * B
        issue_peak = 4.0 * props.multi_processor_count * 1e6 * (clocks["sm_mhz"] if clocks else 1965.0)
        roofline = {
            "bound": "alu", "kernel": "k_filter7_pm<NW,W,P,FS,SH> (search_7lut phase 1)",
            "unit": "warp-instr/s", "peak": alu_peak,
            "peak_source": "integer-ALU pipe: LOP3 issue rate measured in this run (sbg_alu_peak: 8 "
                           "independent dependent chains per thread, 8 CTAs per SM)",
            # warp instructions the kernel sent down the ALU pipe (LOP3, shifts, integer adds) per
            # second of its own CUDA-event time, against what that pipe can take
            "achieved": (alu_inst / filt_s) if alu_inst else None,
            "frac": (alu_inst / filt_s / alu_peak) if alu_inst and alu_peak > 0 else None,
            "alu_warp_instructions": alu_inst, "all_warp_instructions": inst,
            "issue_slot_frac": (inst / filt_s / issue_peak) if inst else None,
            "launches": launches_filter,
            "avg_launch_ms": fam["ms_filter"] / max(launches_filter, 1),
            "instruction_count_source": "profiles/r02_filter_inst_counts.json (ncu "
                                        "smsp__inst_executed[_pipe_alu].sum on the same states, "
                                        "scripts/ncu_inst_counts.sh)" if inst else
                                        "missing: run scripts/ncu_inst_counts.sh",
            "traffic": traffic,
            "note": "no contraction in this path and 16.5 KB of operands per search served from "
                    "shared memory: the binding resource is integer-ALU issue, not HBM or tensor "
                    "cores (SURVEY.md 8d); launch durations are CUDA-event times of the kernel "
                    "running alone; issue_slot_frac = all warp instructions against one per clock "
                    "per scheduler",
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 bitwise (LOP3)",
            "data": "synthetic", "config": config,
            "t_units_per_s": (acc_res["T5"] + acc_res["T7"]) / (ms_res * 1e-3),
            "c_units_per_s": acc_res["C"] / (ms_res * 1e-3),
            "units_per_step": {"T": (acc_res["T5"] + acc_res["T7"]) // args.steps,
                               "C": acc_res["C"] // args.steps},
            # each rank's own searches (before the exchange: ranks hold different states, so their
            # work differs) and the one key exchange that ends the timed region (NCCL all-gather
            # plus waiting for the slowest rank)
            "per_rank_ms_per_step": {"min": min(acc_res["ranks_compute"]) / args.steps,
                                     "mean": sum(acc_res["ranks_compute"]) / len(ranks_res) / args.steps,
                                     "max": max(acc_res["ranks_compute"]) / args.steps,
                                     "with_exchange_max": max(ranks_res) / args.steps,
                                     "exchange_ms_total_rank0": acc_res["gather_ms"]},
            "kernel_ms_per_step_isolated": {k: v / args.steps for k, v in fam.items()},
            # the same, split by the states' mux depth 0..3 (256, 128, 64, 32 masked positions)
            "kernel_ms_per_step_by_mask_depth": {k: [x / args.steps for x in v]
                                                 for k, v in by_depth.items()},
            "kernel_to_step_ratio": sum(fam.values()) / ms_res if world == 1 else None,
            "e2e": {"value": (acc_e2e["T5"] + acc_e2e["T7"] + acc_e2e["C"]) / (ms_e2e * 1e-3),
                    "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    # counted by the library: gate tables, targets and masks shipped (kernel
                    # arguments or copies) / result blocks read from mapped memory
                    "h2d_bytes_per_step": acc_e2e["h2d"] // args.steps,
                    "d2h_bytes_per_step": acc_e2e["d2h"] // args.steps,
                    "note": "host tables -> sbg_stage_problem -> sbg_search_batch -> result structs"},
            "gpu_launches": acc_res["launches"],
            "roofline": roofline,
            "roofline_hbm_equiv": {
                "bound": "hbm", "achieved": hbm_equiv, "peak": peak_gbs, "unit": "GB/s",
                "frac": hbm_equiv / peak_gbs,
                "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                "note": "SURVEY.md 8d unit conversion: 224 algorithmic bytes per 7-combination / "
                        "kernel time; operands never leave shared memory, so this is not a memory "
                        "utilisation and exceeds 1"},
            "clocks": clocks,
        }
        line.update(extras)
        if not args.no_extras and world == 1:
            line["replay"] = replay_record(eng, sb)
        eng.close()
        if not args.no_extras and world == 1:
            line["graph"] = graph_record()
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_arm(n, B, 2000, budget_s=12.0)
            except Exception as exc:  # keep the GPU line even if the CPU leg cannot run
                line["cpu_baseline"] = {"error": repr(exc)}
        print(json.dumps(line))
    else:
        eng.close()
    if world > 1:
        dist.destroy_process_group()


def sharded_record(eng, sb, DistributedLutSearch, args, rank, world):
    """north_star's partition: ONE search sharded over the ranks' GPUs -- work items dealt
    round-robin, the 7-LUT hit lists all-gathered and merged on the devices, one all-reduce(MIN) of
    the key per phase (replacing lut.c:137-149, 329-360, 665-740).  Large states, full-mask
    no-match sweeps.  Parity is asserted in the run: the sharded result and list must equal the
    unsharded ones computed on rank 0's GPU alone."""
    import hashlib
    import torch
    import torch.distributed as dist
    rec = {}
    target = _rijndael_bit(0)
    for spec in [x for x in args.sharded_gates.split(",") if x]:
        n, half = int(spec.rstrip("h")), spec.endswith("h")
        tabs = _state(n, 4242 + n)
        rs = np.random.RandomState(n)
        o5, oo, om = _orders(rs)
        # "h": one mux level deep (128 masked positions, the selector bit excluded): the hit list is
        # not empty, so the list all-gather / merge and the sharded phase 2 carry real data;
        # otherwise the full mask, the pure sweep
        fixed = [(7, 1)] if half else []
        mask, inb = _mux_mask(fixed), [b for b, _ in fixed]
        eng.load(tabs, target, mask, inb)

        def sync():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()

        # unsharded, one GPU (every rank does it: the ranks stay in step); once untimed first --
        # buffers for a search of this size are allocated on first use
        eng.search5(o5)
        eng.search7(oo, om)
        sync()
        t0 = time.perf_counter()
        r5 = eng.search5(o5)
        r7 = eng.search7(oo, om)
        torch.cuda.synchronize()
        ms_one = 1e3 * (time.perf_counter() - t0)
        one = (int(r5.key), int(r7.key), int(r7.tuples_feasible))
        lst = eng.filter7_part(0, 1)
        list_hash = hashlib.sha1(lst.tobytes()).hexdigest()
        entry = {"gates": n, "masked_positions": 128 if fixed else 256,
                 "t_units": math.comb(n, 5) + int(r7.tuples_swept),
                 "ms_one_gpu": ms_one, "list_len": len(lst)}
        if world > 1:
            drv = DistributedLutSearch(eng, shard_min_tuples5=0, shard_min_tuples7=0, shard_min_list=0)
            eng.load(tabs, target, mask, inb)
            drv.search5_sharded(o5)
            drv.search7_sharded(oo, om)
            drv.collective_ms = 0.0
            sync()
            c0 = drv.collectives
            t0 = time.perf_counter()
            s5 = drv.search5_sharded(o5)
            s7 = drv.search7_sharded(oo, om)
            torch.cuda.synchronize()
            own = 1e3 * (time.perf_counter() - t0)
            t = torch.tensor([own], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            got = (int(s5.key), int(s7.key), int(s7.tuples_feasible))
            # the merged list every rank ended up with
            ptr, cnt = eng.list7_device()
            merged = torch.as_tensor(sb.distributed._DeviceArray(ptr, cnt), device="cuda").cpu().numpy() \
                if cnt else np.zeros(0, dtype=np.int64)
            merged_hash = hashlib.sha1(merged.view(np.uint64).tobytes()).hexdigest()
            ok = got == one and merged_hash == list_hash
            flag = torch.tensor([1 if ok else 0], dtype=torch.int64, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) != 1:
                raise SystemExit("sharded search differs from the unsharded one: n=%d rank=%d %r vs %r"
                                 % (n, rank, got, one))
            entry.update({"ms": ms, "collectives": drv.collectives - c0,
                          "collective_ms": drv.collective_ms, "parity": True,
                          "strong_scaling_vs_one_gpu": ms_one / ms})
        else:
            entry.update({"ms": ms_one, "collectives": 0, "collective_ms": 0.0, "parity": True})
        entry["t_units_per_s"] = entry["t_units"] / (entry["ms"] * 1e-3)
        rec["n" + spec] = entry
    rec["what"] = ("one state per size, search_5lut + search_7lut of that state sharded over "
                   "the tuple space across all ranks (ms = max over ranks); ms_one_gpu = the same "
                   "search on one GPU in the same run; parity = keys and merged hit list identical")
    return rec


if __name__ == "__main__":
    main()
