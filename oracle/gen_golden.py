#!/usr/bin/env python3
"""oracle/gen_golden.py -- TEST INFRASTRUCTURE.

Regenerates tests/golden/ from the REFERENCE ITSELF (the binaries oracle/Makefile builds from the
unmodified sources under /root/reference).  Run it in the build container, where the reference is
mounted; the fixtures travel to the GPU box, the reference does not.

  python oracle/gen_golden.py [--skip-runs]

Produces
  tests/golden/seed{1,2}.bin              128-byte RNG seeds (what /dev/urandom supplied)
  tests/golden/run_<sbox>_<seed>.bin      every search_5lut/search_7lut call of a seeded reference
                                          run, recorded by oracle/_ref/sboxgates_rec: inputs, RNG
                                          state before, found/ret[10], number of RNG draws, time
  tests/golden/ref_cases.bin              the same record format for synthetic cases pushed through
                                          the reference's functions via oracle/_ref/libsbgref.so
                                          (edge cases: inbits, sparse masks, no match, stale-cache)
  tests/golden/primitives.json            check_n_lut_possible / get_lut_function /
                                          generate_lut_ttable vectors from the reference
  tests/golden/order_tables.json          the literal 70-row table of lut.c:396-415
  tests/golden/xml_names.json             output file names (gate count + Speck fingerprint,
                                          state.c:123-125) of seeded end-to-end reference runs
  tests/golden/ref_checks.json            the reference's struct layout, its answers to the seeded
                                          random searches of _support.random_ref_cases, and the
                                          graphs (XML as written, DOT from its -d converter) of
                                          seeded CLI runs
  tests/golden/sboxes/*.txt               the reference's S-box tables (data inputs of its CLI)
"""
import argparse
import glob
import json
import os
import re
import shutil
import struct
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _support as S  # noqa: E402

REF = os.environ.get("SBG_REFERENCE", "/root/reference")
REFDIR = os.path.join(ROOT, "oracle", "_ref")
GOLD = os.path.join(ROOT, "tests", "golden")


def seed_bytes(i):
    rs = np.random.RandomState(1000 + i)
    return rs.bytes(128)


def write_record(fp, which, tables, target, mask, inbits, rng_words, rng_p, found, ret, draws, ns):
    n = tables.shape[0]
    fp.write(struct.pack("<II", 0x35474253 if which == 5 else 0x37474253, n))
    fp.write(np.ascontiguousarray(tables, dtype="<u8").tobytes())
    fp.write(np.ascontiguousarray(target, dtype="<u8").tobytes())
    fp.write(np.ascontiguousarray(mask, dtype="<u8").tobytes())
    fp.write(S.inbits_array(inbits).tobytes())
    fp.write(struct.pack("<16Q", *rng_words))
    fp.write(struct.pack("<I", rng_p))
    fp.write(struct.pack("<I", 1 if found else 0))
    fp.write(struct.pack("<10H", *ret))
    fp.write(struct.pack("<Q", draws))
    fp.write(struct.pack("<Q", ns))


def run_recorder(sbox, seedfile, args, limit, out):
    env = dict(os.environ, SBG_SEEDFILE=seedfile, SBG_RECORD=out)
    if limit:
        env["SBG_RECORD_LIMIT"] = str(limit)
        env["SBG_RECORD_EXIT"] = "1"
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [os.path.join(REFDIR, "sboxgates_rec")] + args + [os.path.join(REFDIR, "sboxes", sbox)]
        subprocess.run(cmd, cwd=tmp, env=env, check=True, stdout=subprocess.DEVNULL)
        return sorted(os.path.basename(p) for p in glob.glob(os.path.join(tmp, "*.xml")))


def make_target_from_gates(tables, gate_ids, rs):
    """A random Boolean function of the given gates, as a 256-bit table (so a LUT circuit over
    those gates exists)."""
    k = len(gate_ids)
    func = rs.randint(0, 2, size=1 << k)
    out = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        idx = 0
        for g in gate_ids:
            idx = (idx << 1) | int((int(tables[g][p >> 6]) >> (p & 63)) & 1)
        if func[idx]:
            out[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return out


def random_mask(rs, popcount):
    pos = rs.choice(256, popcount, replace=False)
    out = np.zeros(4, dtype=np.uint64)
    for p in pos:
        out[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return out


def lut5_target(tables, gates, fo, fi):
    t_outer = S.lut_table(fo, tables[gates[0]], tables[gates[1]], tables[gates[2]])
    return S.lut_table(fi, t_outer, tables[gates[3]], tables[gates[4]])


def lut7_target(tables, gates, fo, fm, fi):
    t_outer = S.lut_table(fo, tables[gates[0]], tables[gates[1]], tables[gates[2]])
    t_mid = S.lut_table(fm, tables[gates[3]], tables[gates[4]], tables[gates[5]])
    return S.lut_table(fi, t_outer, t_mid, tables[gates[6]])


def synthetic_cases():
    """(which, tables, target, mask, inbits) tuples; sized so the reference answers each in at most
    a few seconds."""
    full = np.full(4, np.uint64(0xFFFFFFFFFFFFFFFF), dtype=np.uint64)
    sbox = S.rijndael_sbox()
    cases = []
    rs = np.random.RandomState(7)
    # 5-LUT: planted solutions, various n / masks / inbits.
    for i in range(24):
        n = int(rs.choice([5, 6, 8, 9, 12, 16, 24, 40]))
        tabs = S.synthetic_state(n, seed=100 + i, num_inputs=min(8, n))
        gates = sorted(rs.choice(n, 5, replace=False))
        rs.shuffle(gates)
        tgt = lut5_target(tabs, gates, int(rs.randint(1, 255)), int(rs.randint(1, 255)))
        mask = full if i % 3 == 0 else S.mux_mask([(int(rs.randint(0, 8)), int(rs.randint(0, 2)))
                                                   for _ in range(i % 3)])
        inb = [] if i % 4 else [int(rs.randint(0, min(8, n)))]
        cases.append((5, tabs, tgt, mask, inb))
    # 5-LUT: no solution (S-box bit under full mask), small n so the sweep is complete.
    for i, n in enumerate([8, 10, 14, 20]):
        tabs = S.synthetic_state(n, seed=200 + i)
        cases.append((5, tabs, S.sbox_target(sbox, i), full, []))
    # 5-LUT: sparse random masks (NW = 1, 2, 4 paths) with and without solutions.
    for i, pc in enumerate([3, 9, 17, 31, 32, 33, 64, 65, 127, 128, 129, 200]):
        n = 10 + (i % 5)
        tabs = S.synthetic_state(n, seed=300 + i)
        cases.append((5, tabs, S.sbox_target(sbox, i % 8), random_mask(rs, pc), [i % 8] if i % 2 else []))
    # 7-LUT: planted solutions.
    for i in range(12):
        n = int(rs.choice([7, 8, 9, 10, 11, 12]))
        tabs = S.synthetic_state(n, seed=400 + i, num_inputs=min(8, n))
        gates = list(rs.choice(n, 7, replace=False))
        tgt = lut7_target(tabs, gates, int(rs.randint(1, 255)), int(rs.randint(1, 255)),
                          int(rs.randint(1, 255)))
        mask = full if i % 2 == 0 else S.mux_mask([(int(rs.randint(0, 8)), int(rs.randint(0, 2)))])
        inb = [] if i % 3 else [int(rs.randint(0, min(8, n)))]
        cases.append((7, tabs, tgt, mask, inb))
    # 7-LUT: S-box bits, full and mux masks: mostly empty hit lists, some with a few feasible
    # tuples and no decomposition (full 70 x 65536 sweep each).
    for i, (n, fixed) in enumerate([(9, []), (10, [(0, 1)]), (11, [(1, 0), (5, 1)]),
                                    (12, [(2, 1), (3, 0), (7, 1)]), (13, [(0, 0), (4, 1)]),
                                    (12, [(6, 1)])]):
        tabs = S.synthetic_state(n, seed=500 + i)
        inb = [b for b, _ in fixed]
        cases.append((7, tabs, S.sbox_target(sbox, (3 * i) % 8), S.mux_mask(fixed), inb))
    # 7-LUT: sparse random masks -> many feasible tuples, match found early.
    for i, pc in enumerate([8, 12, 20, 33, 48, 70]):
        n = 9 + (i % 4)
        tabs = S.synthetic_state(n, seed=600 + i)
        cases.append((7, tabs, S.sbox_target(sbox, i % 8), random_mask(rs, pc), []))
    return cases


def _lut_bit(func, a, b, c):
    return (func >> (a << 2 | b << 1 | c)) & 1


def build_stale_cache_case(rs, outer_first_gate, extras=28):
    """An 11-gate instance whose 7-LUT hit list is exactly prev=(0,1,2,3,4,5,6), cur=(0,5,6,7,8,9,10).
    That makes the reference evaluate rows 0-3 of `cur` with the outer tables it cached for
    (1,5,6) -- its cache key drops the first gate (lut.c:379,432-435) and prev's last row left
    (1,5,6) behind -- instead of (0,5,6).

    Construction: masked positions are 11-bit gate-value vectors.  A position u = 0 with target 1
    against positions with target 0 whose supports are {0,1},{0,7},{5},{6} and {a,b} for a in 1..4,
    b in 7..10 forces every feasible 7-set to contain 5,6, all of 1..4 or all of 7..10, and 0 unless
    it holds both 1 and 7 -- so the list starts prev, cur (the other feasible sets start with 1).  The target
    is a 7-LUT over (outer_first_gate,5,6 | 7,8,9 | 10): with outer_first_gate = 0 the only true
    decomposition sits in the rows the reference evaluates with stale tables; with 1 the stale rows
    "find" a circuit that is wrong for the gates they report.  Further random positions are added
    while prev and cur stay feasible, to make prev non-decomposable."""
    skeleton = [0, (1 << 0) | (1 << 1), (1 << 0) | (1 << 7), 1 << 5, 1 << 6] \
        + [(1 << a) | (1 << b) for a in (1, 2, 3, 4) for b in (7, 8, 9, 10)]
    og = outer_first_gate

    def bit(w, g):
        return (w >> g) & 1

    for _attempt in range(200000):
        fo, fm, fi = (int(x) for x in rs.randint(1, 255, size=3))

        def F(w):
            x = _lut_bit(fo, bit(w, og), bit(w, 5), bit(w, 6))
            y = _lut_bit(fm, bit(w, 7), bit(w, 8), bit(w, 9))
            return _lut_bit(fi, x, y, bit(w, 10))
        if F(0) == 1 and all(F(v) == 0 for v in skeleton[1:]):
            break
    else:
        return None
    prev_g, cur_g = (0, 1, 2, 3, 4, 5, 6), (0, 5, 6, 7, 8, 9, 10)

    def proj(w, gates):
        return tuple(bit(w, g) for g in gates)
    vecs = list(skeleton)
    seen_prev = {proj(w, prev_g): F(w) for w in vecs}
    seen_cur = {proj(w, cur_g): F(w) for w in vecs}
    tries = 0
    while len(vecs) < len(skeleton) + extras and tries < 20000:
        tries += 1
        w = int(rs.randint(0, 1 << 11))
        t = F(w)
        if w in vecs or seen_prev.get(proj(w, prev_g), t) != t or seen_cur.get(proj(w, cur_g), t) != t:
            continue
        vecs.append(w)
        seen_prev[proj(w, prev_g)] = t
        seen_cur[proj(w, cur_g)] = t
    positions = rs.choice(256, len(vecs), replace=False)
    tabs = np.zeros((11, 4), dtype=np.uint64)
    noise = rs.randint(0, 2, size=(11, 256))
    where = {int(p): w for p, w in zip(positions, vecs)}
    tgt = np.zeros(4, dtype=np.uint64)
    mask = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        one = np.uint64(1) << np.uint64(p & 63)
        for g in range(11):
            v = bit(where[p], g) if p in where else int(noise[g][p])
            if v:
                tabs[g][p >> 6] |= one
        if p in where:
            mask[p >> 6] |= one
            if F(where[p]):
                tgt[p >> 6] |= one
        elif rs.randint(0, 2):
            tgt[p >> 6] |= one
    return tabs, tgt, mask


def find_stale_cache_cases():
    out = []
    rs = np.random.RandomState(11)
    want = {"stale_miss": 3, "stale_hit": 3}   # reference passes over / matches inside stale rows
    tries = 0
    while any(v > 0 for v in want.values()) and tries < 60:
        tries += 1
        kind = "stale_miss" if tries % 2 else "stale_hit"
        if want[kind] == 0:
            continue
        case = build_stale_cache_case(rs, 0 if kind == "stale_miss" else 1)
        if case is None:
            continue
        tabs, tgt, mask = case
        lst, _ = S.oracle_filter7(tabs, tgt, mask, [])
        if lst.tolist()[:2] != [[0, 1, 2, 3, 4, 5, 6], [0, 5, 6, 7, 8, 9, 10]]:
            continue
        rng = S.OrcRng.from_seed(tries)
        found, ret, st = S.oracle_search(7, tabs, tgt, mask, [], rng)
        if st.stale_cache_rows == 0:
            continue   # prev already matched
        if kind == "stale_hit" and not (found and st.stale_hit):
            continue
        if kind == "stale_miss" and st.stale_hit:
            continue
        want[kind] -= 1
        print("stale-cache case (%s): found=%d ret=%s" % (kind, found, ret))
        out.append((7, tabs, tgt, mask, []))
    return out


def primitives(rs):
    lib = S.ref_lib()
    vec = {"lut_ttable": [], "get_lut_function": [], "check_n_lut_possible": []}
    import ctypes as C
    for i in range(40):
        tabs = S.synthetic_state(12, seed=700 + i)
        a, b, c = (tabs[j] for j in rs.choice(12, 3, replace=False))
        func = int(rs.randint(0, 256))
        out = np.zeros(4, dtype=np.uint64)
        lib.sbgref_generate_lut_ttable(func, S._u64(a)[1], S._u64(b)[1], S._u64(c)[1],
                                       out.ctypes.data_as(S.u64p))
        vec["lut_ttable"].append({"func": func, "in": [x.tolist() for x in (a, b, c)],
                                  "out": out.tolist()})
        mask = random_mask(rs, int(rs.choice([4, 8, 16, 64, 256])))
        tgt = S.lut_table(int(rs.randint(0, 256)), a, b, c) if i % 2 else random_mask(rs, 128)
        f = C.c_uint8()
        ok = lib.sbgref_get_lut_function(S._u64(a)[1], S._u64(b)[1], S._u64(c)[1], S._u64(tgt)[1],
                                         S._u64(mask)[1], 0, C.byref(f))
        vec["get_lut_function"].append({"in": [x.tolist() for x in (a, b, c)],
                                        "target": tgt.tolist(), "mask": mask.tolist(),
                                        "ok": int(ok), "func": int(f.value)})
        for num in (3, 5, 7):
            ids = rs.choice(12, num, replace=False)
            sub = np.ascontiguousarray(tabs[ids])
            t2 = make_target_from_gates(tabs, list(ids[:num - (i % 2)]) + ([int(rs.randint(0, 12))]
                                        if i % 2 else []), rs) if i % 3 else random_mask(rs, 128)
            m2 = random_mask(rs, int(rs.choice([6, 12, 24, 64, 256])))
            okc = lib.sbgref_check_n_lut_possible(num, S._u64(t2)[1], S._u64(m2)[1], S._u64(sub)[1])
            vec["check_n_lut_possible"].append({"num": num, "tables": sub.tolist(),
                                                "target": t2.tolist(), "mask": m2.tolist(),
                                                "ok": int(okc)})
    return vec


def literal_order_table():
    """Parses the 70 x 7 literal at lut.c:396-415 (a golden vector, not code)."""
    src = open(os.path.join(REF, "lut.c")).read()
    m = re.search(r"const int order\[70 \* 7\] = \{(.*?)\};", src, re.S)
    nums = [int(x) for x in re.findall(r"\d+", m.group(1))]
    assert len(nums) == 490
    return [nums[7 * i:7 * i + 7] for i in range(70)]


# seeded reference CLI runs whose graphs ref_checks.json stores: (S-box, options, seed, keep only
# the last file written)
CLI_GRAPHS = [("crypto1_fa.txt", ["-l"], "seed1", False), ("crypto1_fc.txt", ["-l"], "seed1", False),
              ("crypto1_fc.txt", ["-l"], "seed2", False), ("des_s1.txt", ["-o", "0"], "seed1", True)]


def ref_checks():
    """What tests/test_oracle_ref.py compares with, taken from the reference's own object code."""
    import ctypes as C
    lib = S.ref_lib()
    a, b, c, d, e = (C.c_int() for _ in range(5))
    lib.sbgref_sizes(C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    layout = {"ttable": a.value, "gate": b.value, "state": c.value, "state_gates_offset": d.value}
    lib.sbgref_options_layout(C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e))
    layout.update({"options_randomize_offset": a.value, "options_lut_graph_offset": b.value,
                   "options_verbosity_offset": c.value, "options": d.value, "boolfunc": e.value})
    searches = []
    for which, tabs, tgt, mask, inb, seed in S.random_ref_cases():
        rng = S.OrcRng.from_seed(seed)
        found, ret, draws = S.ref_search(which, tabs, tgt, mask, inb, rng)
        searches.append({"which": which, "found": int(found), "ret": ret, "draws": draws,
                         "rng_after": [str(w) for w in rng.words()], "rng_p": rng.p})
    graphs = []
    exe = os.path.join(REFDIR, "sboxgates_ref")
    for sbox, cli, seed, last_only in CLI_GRAPHS:
        with tempfile.TemporaryDirectory() as tmp:
            env = dict(os.environ, SBG_SEEDFILE=os.path.join(GOLD, seed + ".bin"))
            subprocess.run([exe] + cli + [os.path.join(REFDIR, "sboxes", sbox)], cwd=tmp, env=env,
                           check=True, stdout=subprocess.DEVNULL, timeout=300)
            names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(tmp, "*.xml")))
            files = []
            for name in names[-1:] if last_only else names:
                xml = open(os.path.join(tmp, name)).read()
                dot = subprocess.run([exe, "-d", name], cwd=tmp, env=env, check=True,
                                     capture_output=True, text=True).stdout
                files.append({"name": name, "xml": xml, "dot": dot})
        graphs.append({"key": " ".join([sbox] + cli + [seed]), "names": names, "files": files})
    json.dump({"layout": layout, "searches": searches, "graphs": graphs},
              open(os.path.join(GOLD, "ref_checks.json"), "w"), indent=1)
    os.makedirs(os.path.join(GOLD, "sboxes"), exist_ok=True)
    for path in sorted(glob.glob(os.path.join(REF, "sboxes", "*.txt"))):
        shutil.copyfile(path, os.path.join(GOLD, "sboxes", os.path.basename(path)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--skip-runs", action="store_true", help="keep existing run_*.bin files")
    ap.add_argument("--only-stale", action="store_true", help="just print the stale-cache cases")
    ap.add_argument("--only-ref-checks", action="store_true",
                    help="only tests/golden/ref_checks.json and tests/golden/sboxes/")
    args = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    if not S.ref_available():
        sys.exit("oracle/_ref is not built: run `make -C oracle` where the reference sources are")

    if args.only_stale:
        print(len(find_stale_cache_cases()))
        return
    if args.only_ref_checks:
        ref_checks()
        return
    for i in (1, 2):
        with open(os.path.join(GOLD, "seed%d.bin" % i), "wb") as fp:
            fp.write(seed_bytes(i))

    xml_names = {}
    if not args.skip_runs:
        runs = [
            ("crypto1_fa.txt", ["-l"], 0), ("crypto1_fb.txt", ["-l"], 0),
            ("crypto1_fc.txt", ["-l"], 0), ("des_s1.txt", ["-l", "-o", "0"], 0),
            ("rijndael.txt", ["-l", "-o", "0"], 150), ("sodark.txt", ["-l", "-o", "0"], 120),
        ]
        for sbox, cli, limit in runs:
            for si in (1, 2):
                if limit and si == 2:
                    continue
                name = "run_%s_seed%d.bin" % (sbox.split(".")[0], si)
                open(os.path.join(GOLD, name), "wb").close()   # runs with < 5 gates record nothing
                xmls = run_recorder(sbox, os.path.join(GOLD, "seed%d.bin" % si), cli, limit,
                                    os.path.join(GOLD, name))
                if not limit:
                    xml_names["%s %s seed%d" % (sbox, " ".join(cli), si)] = xmls
                print(name, xmls)
        json.dump(xml_names, open(os.path.join(GOLD, "xml_names.json"), "w"), indent=1,
                  sort_keys=True)

    cases = synthetic_cases()
    stale = find_stale_cache_cases()
    print("synthetic cases:", len(cases), "stale-cache cases:", len(stale))
    with open(os.path.join(GOLD, "ref_cases.bin"), "wb") as fp:
        for ci, (which, tabs, tgt, mask, inb) in enumerate(cases + stale):
            rng = S.OrcRng.from_seed(5000 + ci)
            words, p = rng.words(), rng.p
            import time
            t0 = time.time()
            found, ret, draws = S.ref_search(which, tabs, tgt, mask, inb, rng)
            ns = int((time.time() - t0) * 1e9)
            write_record(fp, which, tabs, tgt, mask, inb, words, p, found, ret, draws, ns)
            print("case %3d: %dLUT n=%2d found=%d draws=%d %.2fs" % (ci, which, tabs.shape[0], found,
                                                                    draws, ns / 1e9))

    json.dump(primitives(np.random.RandomState(3)), open(os.path.join(GOLD, "primitives.json"), "w"))
    json.dump(literal_order_table(), open(os.path.join(GOLD, "order_tables.json"), "w"))
    ref_checks()
    print("done")


if __name__ == "__main__":
    main()
