"""Test-side helpers: ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when it was
built, for the reference's own object code (oracle/_ref/libsbgref.so), plus readers for the
fixtures under tests/golden/.

TEST INFRASTRUCTURE -- nothing under sboxgates_b200/ imports this module or anything in oracle/.
"""
import ctypes as C
import os
import struct
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")

u64p = C.POINTER(C.c_uint64)
u16p = C.POINTER(C.c_uint16)
i8p = C.POINTER(C.c_int8)
u8p = C.POINTER(C.c_uint8)


class OrcRng(C.Structure):
    _fields_ = [("s", C.c_uint64 * 16), ("p", C.c_int32), ("draws", C.c_uint64)]

    @classmethod
    def from_seed(cls, seed):
        """State = 16 little-endian words of `seed` bytes (what sboxgates.c:254 reads)."""
        if isinstance(seed, int):
            rs = np.random.RandomState(seed)
            seed = rs.bytes(128)
        r = cls()
        for i, w in enumerate(struct.unpack("<16Q", seed)):
            r.s[i] = w
        r.p = 0
        r.draws = 0
        return r

    def copy(self):
        r = OrcRng()
        C.memmove(C.byref(r), C.byref(self), C.sizeof(OrcRng))
        return r

    def words(self):
        return [int(x) for x in self.s]


class OrcStats(C.Structure):
    _fields_ = [("tuples_filtered", C.c_uint64), ("tuples_feasible", C.c_uint64),
                ("candidates", C.c_uint64), ("stale_cache_rows", C.c_uint64),
                ("stale_hit", C.c_uint64)]


def _u64(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a, a.ctypes.data_as(u64p)


def inbits_array(inbits):
    arr = np.full(8, -1, dtype=np.int8)
    arr[:len(inbits)] = inbits
    return arr


_oracle = None


def oracle_lib():
    """Loads oracle/liboracle.so, building it first if the source is newer or it is missing."""
    global _oracle
    if _oracle is not None:
        return _oracle
    so = os.path.join(ORACLE_DIR, "liboracle.so")
    src = os.path.join(ORACLE_DIR, "sbg_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.run(["make", "-C", ORACLE_DIR, "oracle"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.orc_rng_next.restype = C.c_uint64
    lib.orc_rng_next.argtypes = [C.POINTER(OrcRng)]
    lib.orc_n_choose_k.restype = C.c_int64
    lib.orc_n_choose_k.argtypes = [C.c_int, C.c_int]
    lib.orc_nth_combination.argtypes = [C.c_int64, C.c_int, C.c_int, u16p]
    lib.orc_combination_rank.restype = C.c_int64
    lib.orc_combination_rank.argtypes = [C.c_int, C.c_int, u16p]
    lib.orc_lut_ttable.argtypes = [C.c_uint8, u64p, u64p, u64p, u64p]
    lib.orc_check_n_lut_possible.argtypes = [C.c_int, u64p, u64p, u64p]
    lib.orc_get_lut_function.argtypes = [u64p, u64p, u64p, u64p, u64p, C.c_int,
                                         C.POINTER(OrcRng), u8p]
    lib.orc_solve_inner.argtypes = [u64p, u64p, u64p, u64p, u64p, u8p, u8p]
    for name in ("orc_search_5lut", "orc_search_7lut"):
        getattr(lib, name).argtypes = [u64p, C.c_int, u64p, u64p, i8p, C.POINTER(OrcRng), u16p,
                                       C.POINTER(OrcStats)]
    lib.orc_filter_7lut.argtypes = [u64p, C.c_int, u64p, u64p, i8p, u16p, C.c_int,
                                    C.POINTER(OrcStats)]
    lib.orc_search5_key.restype = C.c_uint64
    lib.orc_search5_key.argtypes = [u64p, C.c_int, u64p, u64p, i8p, u8p, C.c_int, C.c_int]
    lib.orc_decomp7_key.restype = C.c_uint64
    lib.orc_decomp7_key.argtypes = [u64p, u64p, u64p, u16p, C.c_int, u8p, u8p, C.c_int, C.c_int]
    lib.orc_order7_row.argtypes = [C.c_int, C.POINTER(C.c_int)]
    lib.orc_order5_row.argtypes = [C.c_int, C.POINTER(C.c_int)]
    _oracle = lib
    return lib


def oracle_search(which, tables, target, mask, inbits, rng):
    """Runs orc_search_{5,7}lut; returns (found, ret[10] list, stats); rng is advanced in place."""
    lib = oracle_lib()
    tables, tp = _u64(tables)
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    ib = inbits_array(inbits)
    ret = (C.c_uint16 * 10)()
    stats = OrcStats()
    fn = lib.orc_search_5lut if which == 5 else lib.orc_search_7lut
    found = fn(tp, tables.shape[0], gp, mp, ib.ctypes.data_as(i8p), C.byref(rng), ret,
               C.byref(stats))
    return bool(found), [int(x) for x in ret], stats


def oracle_filter7(tables, target, mask, inbits, cap=100000):
    lib = oracle_lib()
    tables, tp = _u64(tables)
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    ib = inbits_array(inbits)
    out = np.zeros((cap, 7), dtype=np.uint16)
    stats = OrcStats()
    cnt = lib.orc_filter_7lut(tp, tables.shape[0], gp, mp, ib.ctypes.data_as(i8p),
                              out.ctypes.data_as(u16p), cap, C.byref(stats))
    return out[:cnt].copy(), stats


def _order(order):
    return (C.c_uint8 * 256).from_buffer_copy(bytes(order))


def oracle_search5_key(tables, target, mask, inbits, func_order, part=0, nparts=1):
    lib = oracle_lib()
    tables, tp = _u64(tables)
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    ib = inbits_array(inbits)
    return int(lib.orc_search5_key(tp, tables.shape[0], gp, mp, ib.ctypes.data_as(i8p),
                                   _order(func_order), part, nparts))


def oracle_decomp7_key(tables, target, mask, tuples, outer, middle, part=0, nparts=1):
    """tuples: (count, 7) uint16 array = the feasible list in lexicographic order."""
    lib = oracle_lib()
    tables, tp = _u64(tables)
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    lst = np.ascontiguousarray(tuples, dtype=np.uint16).reshape(-1, 7)
    return int(lib.orc_decomp7_key(tp, gp, mp, lst.ctypes.data_as(u16p), lst.shape[0],
                                   _order(outer), _order(middle), part, nparts))


def order7_rows():
    lib = oracle_lib()
    rows = []
    for k in range(70):
        r = (C.c_int * 7)()
        lib.orc_order7_row(k, r)
        rows.append([int(x) for x in r])
    return rows


def order5_rows():
    lib = oracle_lib()
    rows = []
    for k in range(10):
        r = (C.c_int * 5)()
        lib.orc_order5_row(k, r)
        rows.append([int(x) for x in r])
    return rows


_ref = None


def ref_available():
    return os.path.exists(os.path.join(REF_DIR, "libsbgref.so"))


def ref_lib():
    """The reference's own object code behind pointer-based wrappers (oracle/ref_glue.c)."""
    global _ref
    if _ref is not None:
        return _ref
    lib = C.CDLL(os.path.join(REF_DIR, "libsbgref.so"))
    lib.sbgref_rng_set.argtypes = [u64p, C.c_int]
    lib.sbgref_rng_get.argtypes = [u64p, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    lib.sbgref_check_n_lut_possible.argtypes = [C.c_int, u64p, u64p, u64p]
    lib.sbgref_get_lut_function.argtypes = [u64p, u64p, u64p, u64p, u64p, C.c_int, u8p]
    lib.sbgref_generate_lut_ttable.argtypes = [C.c_int, u64p, u64p, u64p, u64p]
    for name in ("sbgref_search_5lut", "sbgref_search_7lut"):
        getattr(lib, name).argtypes = [u64p, C.c_int, u64p, u64p, i8p, u16p]
    lib.sbgref_set_fake_rank.argtypes = [C.c_int, C.c_int]
    _ref = lib
    return lib


def ref_search(which, tables, target, mask, inbits, rng):
    """Runs the reference's search_{5,7}lut from RNG state `rng` (an OrcRng, advanced in place to
    the state the reference left).  Returns (found, ret[10], draws)."""
    lib = ref_lib()
    tables, tp = _u64(tables)
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    ib = inbits_array(inbits)
    s = (C.c_uint64 * 16)(*rng.words())
    lib.sbgref_rng_set(s, rng.p)
    ret = (C.c_uint16 * 10)()
    fn = lib.sbgref_search_5lut if which == 5 else lib.sbgref_search_7lut
    found = fn(tp, tables.shape[0], gp, mp, ib.ctypes.data_as(i8p), ret)
    p = C.c_int()
    draws = C.c_uint64()
    lib.sbgref_rng_get(s, C.byref(p), C.byref(draws))
    for i in range(16):
        rng.s[i] = s[i]
    rng.p = p.value
    rng.draws += draws.value
    return bool(found), [int(x) for x in ret], int(draws.value)


# ------------------------------------------------------------------------------------------------
# Recorded search calls (oracle/ref_glue.c, SBGREF_RECORDER).

class Record:
    __slots__ = ("which", "n", "tables", "target", "mask", "inbits", "rng_s", "rng_p", "found",
                 "ret", "draws", "ns")

    def rng(self):
        r = OrcRng()
        for i, w in enumerate(self.rng_s):
            r.s[i] = w
        r.p = self.rng_p
        r.draws = 0
        return r

    def inbits_list(self):
        out = []
        for b in self.inbits:
            if b == -1:
                break
            out.append(int(b))
        return out


def read_records(path):
    data = open(path, "rb").read()
    off = 0
    recs = []
    while off < len(data):
        magic, n = struct.unpack_from("<II", data, off)
        off += 8
        r = Record()
        r.which = {0x35474253: 5, 0x37474253: 7}[magic]
        r.n = n
        r.tables = np.frombuffer(data, dtype="<u8", count=4 * n, offset=off).reshape(n, 4).copy()
        off += 32 * n
        r.target = np.frombuffer(data, dtype="<u8", count=4, offset=off).copy()
        off += 32
        r.mask = np.frombuffer(data, dtype="<u8", count=4, offset=off).copy()
        off += 32
        r.inbits = np.frombuffer(data, dtype=np.int8, count=8, offset=off).copy()
        off += 8
        r.rng_s = list(struct.unpack_from("<16Q", data, off))
        off += 128
        (r.rng_p,) = struct.unpack_from("<I", data, off)
        off += 4
        (found,) = struct.unpack_from("<I", data, off)
        off += 4
        r.found = bool(found)
        r.ret = list(struct.unpack_from("<10H", data, off))
        off += 20
        (r.draws,) = struct.unpack_from("<Q", data, off)
        off += 8
        (r.ns,) = struct.unpack_from("<Q", data, off)
        off += 8
        recs.append(r)
    return recs


# ------------------------------------------------------------------------------------------------
# Synthetic states (SURVEY.md section 8d): input-bit tables followed by random 3-LUTs of earlier
# gates, which is what a graph under construction looks like.

def input_table(bit):
    """generate_target(bit, false), state.c:232-250: position p holds bit `bit` of p."""
    words = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        if (p >> bit) & 1:
            words[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return words


def sbox_target(sbox, bit):
    """generate_target(bit, true): position p holds bit `bit` of sbox[p]."""
    words = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        if (sbox[p] >> bit) & 1:
            words[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return words


def lut_table(func, a, b, c):
    out = np.zeros(4, dtype=np.uint64)
    full = np.uint64(0xFFFFFFFFFFFFFFFF)
    for m in range(8):
        if (func >> m) & 1:
            x = a if m & 4 else a ^ full
            y = b if m & 2 else b ^ full
            z = c if m & 1 else c ^ full
            out |= x & y & z
    return out


def synthetic_state(n, seed, num_inputs=8):
    rs = np.random.RandomState(seed)
    tabs = [input_table(i) for i in range(num_inputs)]
    while len(tabs) < n:
        i, j, k = rs.choice(len(tabs), 3, replace=False)
        f = int(rs.randint(1, 255))
        tabs.append(lut_table(f, tabs[i], tabs[j], tabs[k]))
    return np.stack(tabs[:n]).astype(np.uint64)


def rijndael_sbox():
    """The AES S-box from its definition (inverse in GF(2^8) mod x^8+x^4+x^3+x+1, then the affine
    map); equals sboxes/rijndael.txt (tests/golden/sboxes/), which tests/test_oracle_ref.py checks."""
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
    out = []
    for a in range(256):
        x = inv[a]
        y = x
        for s in (1, 2, 3, 4):
            y ^= ((x << s) | (x >> (8 - s))) & 0xFF
        out.append(y ^ 0x63)
    return out


def mux_mask(fixed):
    """Mask left after mux recursion fixed input bit b to value v for each (b, v) in `fixed`
    (create_circuit, sboxgates.c:478,483: mask & ~fsel / mask & fsel)."""
    words = np.zeros(4, dtype=np.uint64)
    for p in range(256):
        if all(((p >> b) & 1) == v for b, v in fixed):
            words[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
    return words


def oracle_check(num, target, mask, tables):
    """check_n_lut_possible (lut.c:34-66) of the CPU oracle; tables: list of `num` 4-word arrays."""
    lib = oracle_lib()
    target, gp = _u64(target)
    mask, mp = _u64(mask)
    tabs, tp = _u64(np.stack(tables))
    return bool(lib.orc_check_n_lut_possible(num, gp, mp, tp))


def random_ref_cases():
    """The 30 x 2 seeded random searches tests/golden/ref_checks.json holds the reference's answers
    to: yields (which, tables, target, mask, inbits, seed bytes) in the order they were recorded."""
    sbox = rijndael_sbox()
    rs = np.random.RandomState(123)
    for i in range(30):
        n = int(rs.choice([7, 8, 9, 10, 11]))
        tabs = synthetic_state(n, seed=3000 + i, num_inputs=min(8, n))
        pos = rs.choice(256, int(rs.choice([6, 10, 16, 24, 40])), replace=False)
        mask = np.zeros(4, dtype=np.uint64)
        for p in pos:
            mask[p >> 6] |= np.uint64(1) << np.uint64(p & 63)
        tgt = sbox_target(sbox, int(rs.randint(0, 8)))
        inb = [int(rs.randint(0, min(8, n)))] if i % 3 == 0 else []
        for which in (5, 7):
            yield which, tabs, tgt, mask, inb, rs.bytes(128)


def oracle_get_lut_function(in1, in2, in3, target, mask, rng, randomize=True):
    """get_lut_function (lut.c:79-109) of the CPU oracle: (ok, func); rng advanced as the reference
    would (one draw iff the solved function has unconstrained bits)."""
    lib = oracle_lib()
    arrs = [_u64(x) for x in (in1, in2, in3, target, mask)]
    func = C.c_uint8()
    ok = lib.orc_get_lut_function(*[a[1] for a in arrs], 1 if randomize else 0, C.byref(rng),
                                  C.byref(func))
    return bool(ok), int(func.value)
