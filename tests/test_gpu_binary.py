"""Every scan-kernel instantiation of test_scan_variants.VARIANTS against the oracle on BINARY input: uniform bytes, ASCII
text salted with bytes >= 0x80, NUL and 0x80 filler.  Matches are planted on the 1 KiB borders of each unit -- which are
also 16-byte lane, 512-byte row, 2 KiB RUN block and 4 KiB slice borders, and at 64 KiB tile borders -- and at the unit end,
each next to near misses that differ in one byte by exactly what a SWAR filter is blind to (bit 7, bit 5, 0x00, 0xff).  Class runs get ASCII slices with a single high byte at the
slice's first or last byte, only in its 16-byte look-ahead, or just before it, and runs of run_min - 1 / run_min /
run_min + 1 across slice and tile borders.  Each row runs on a fresh context and again after a scan of 0xff / 0x80 data,
from host units and from device units packed at 16-byte strides, in ALL, FIRST and LINE mode.

The generators are shared with test_oracle_vs_ref.py, which pins the oracle itself to the reference on such inputs."""
import random
import time

import numpy as np
import pytest

import grab_b200 as G
import oracle_py as O
from test_scan_variants import VARIANTS, family

MODES = (G.MODE_ALL, G.MODE_FIRST, G.MODE_LINE)
SLICE = 4096
EDGE_LENS = (2047, 2048, 2049, 4095, 4096, 4097, 65535, 65536, 65537)
BIG_LEN = 200 * 1024 + 37  # several 64 KiB tiles


# ---- a sample match of a pattern ------------------------------------------------------------------------------------
def _byte_class(pat, i):
    """[...] at pat[i] -> (set of bytes, index behind it)"""
    i += 1
    neg = pat[i] == "^"
    if neg:
        i += 1
    out, first = set(), True
    while pat[i] != "]" or first:
        first = False
        lo, i = _one_byte(pat, i)
        if pat[i] == "-" and pat[i + 1] != "]":
            hi, i = _one_byte(pat, i + 1)
            out.update(range(lo, hi + 1))
        else:
            out.add(lo)
    return (set(range(256)) - out if neg else out), i + 1


_ESC = {"n": 10, "t": 9, "r": 13, "f": 12}


def _one_byte(pat, i):
    if pat[i] != "\\":
        return ord(pat[i]), i + 1
    if pat[i + 1] == "x":
        return int(pat[i + 2:i + 4], 16), i + 4
    c = pat[i + 1]
    return _ESC.get(c, ord(c)), i + 2


_CLASS_ESC = {"w": set(b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789_"), "d": set(b"0123456789")}


def _atoms(alt, icase):
    """one alternative -> [(bytes it may hold, min, max)]; None if outside the subset this generator reads"""
    atoms, i = [], 0
    while i < len(alt):
        c = alt[i]
        if c == "[":
            s, i = _byte_class(alt, i)
        elif c == ".":
            s, i = set(range(256)) - {10}, i + 1
        elif c == "\\" and alt[i + 1] in _CLASS_ESC:
            s, i = set(_CLASS_ESC[alt[i + 1]]), i + 2
        elif c in "()|*?^$":
            return None
        else:
            b, i = _one_byte(alt, i)
            s = {b}
        if icase:
            s |= {x ^ 0x20 for x in s if 0x41 <= (x & 0xdf) <= 0x5a}
        lo = hi = 1
        if i < len(alt) and alt[i] == "+":
            lo, hi, i = 1, None, i + 1
        elif i < len(alt) and alt[i] == "{":
            j = alt.index("}", i)
            a, _, b = alt[i + 1:j].partition(",")
            lo = int(a)
            hi = lo if not _ else (int(b) if b else None)
            i = j + 1
        atoms.append((sorted(s), lo, hi))
    return atoms


def sample_match(pat, rnd):
    """bytes one alternative of `pat` matches (a random one), or None for patterns outside the generator's subset:
    (?i), top-level |, literals, \\xHH, ., [...], \\w, \\d, +, {n}, {n,}, {n,m}"""
    icase = pat.startswith("(?i)")
    body = pat[4:] if icase else pat
    alts = body.split("|")
    atoms = _atoms(rnd.choice(alts), icase)
    if atoms is None:
        return None
    out = bytearray()
    for s, lo, hi in atoms:
        n = lo + rnd.randint(0, 2 if hi is None else hi - lo)
        out += bytes(rnd.choice(s) for _ in range(n))
    return bytes(out)


# ---- backgrounds and plants ------------------------------------------------------------------------------------------
def background(rnd, n, kind):
    """kind 0: uniform 0..255; 1: ASCII text (letters, digits, space, newline) with about one byte in 16 >= 0x80"""
    g = np.random.default_rng(rnd.getrandbits(32))
    if kind == 0:
        return g.integers(0, 256, n, dtype=np.uint8)
    txt = np.frombuffer(b"etaoinshrdlucmfwypvbgkqjxz ETAOIN0123456789_  \n", dtype=np.uint8)
    a = txt[g.integers(0, txt.size, n)]
    hi = g.random(n) < 1 / 16
    a[hi] = g.integers(0x80, 256, int(hi.sum()), dtype=np.uint8)
    return a


def near_misses(m, rnd):
    """copies of m with one byte changed by bit 7, by bit 5, to 0x00 and to 0xff"""
    out = []
    for f in (lambda b: b ^ 0x80, lambda b: b ^ 0x20, lambda b: 0, lambda b: 0xff):
        c = bytearray(m)
        k = rnd.randrange(len(c))
        c[k] = f(c[k])
        out.append(bytes(c))
    return out


def plant(a, pos, m):
    if 0 <= pos and pos + len(m) <= a.size:
        a[pos:pos + len(m)] = np.frombuffer(m, dtype=np.uint8)


def small_units(pat, rnd, max_len=4096):
    """seeded binary inputs of at most max_len bytes for one pattern (also what test_oracle_vs_ref feeds the reference)"""
    units = []
    for n in list(range(1, 65)) + [200, 511, 512, 513, 2047, 2049, 4095, 4096]:
        if n > max_len:
            continue
        a = background(rnd, n, n % 2)
        m = sample_match(pat, rnd)
        if m and len(m) <= n and rnd.random() < 0.7:
            pos = rnd.choice([0, n - len(m), rnd.randrange(n - len(m) + 1)])
            plant(a, pos, m)
            for k, x in enumerate(near_misses(m, rnd)):
                plant(a, pos + len(m) + 1 + k * (len(m) + 1), x)
        units.append(a)
    return units


def edge_units(pat, rnd):
    """units of EDGE_LENS and BIG_LEN bytes: a match planted around the unit's 1 KiB borders (every one for matches up to
    240 bytes, every k-th for longer ones) and at the unit end.  The offset against the border (-len-1 .. +1: the match
    straddles it, starts on it, ends on it, ...) cycles across the 1 KiB borders, and separately across the 4 KiB slice
    borders among them, so slices see every offset too.  Each match is followed by its near misses; NUL and 0x80 filler
    in the big unit"""
    units = []
    for n in EDGE_LENS + (BIG_LEN,):
        a = background(rnd, n, n % 2)
        m0 = sample_match(pat, rnd)
        if m0:
            L = len(m0)
            step = 1024 * -(-(4 * L + 64) // 1024)  # room for the match and its near misses
            for edge in range(step, n, step):
                m = sample_match(pat, rnd)
                k = edge // SLICE if edge % SLICE == 0 else edge // 1024
                d = -L - 1 + (k % (L + 3))  # -L-1 .. +1 against the border
                plant(a, edge + d, m)
                for j, x in enumerate(near_misses(m, rnd)):
                    plant(a, edge + d + len(m) + 17 + j * (len(m) + 3), x)
            for d in (1, 0):  # ending on the unit's last byte and one before it
                m = sample_match(pat, rnd)
                plant(a, n - len(m) - d, m)
        if n == BIG_LEN:
            a[40000:48192] = 0x00
            a[90000:98192] = 0x80
        units.append(a)
    return units


def run_units(pat, run_min, rnd, n_slices=6):
    """class runs: ASCII slices with one high byte each, at the slice's first byte, its last byte, only in the look-ahead
    of the slice before, or before it; runs of run_min - 1 / run_min / run_min + 1 ending on and crossing the borders"""
    atoms = _atoms(pat, False)
    if not atoms or len(atoms) != 1:
        return []
    cls = set(atoms[0][0])  # the run's byte class
    ascii_cls = sorted(b for b in cls if b < 0x80) or sorted(cls)
    # background: bytes outside the class (printable ASCII and newline where the class leaves any), so a planted run has
    # exactly its planted length
    out_cls = ([b for b in list(range(0x20, 0x7f)) + [10] if b not in cls] or [b for b in range(0x80) if b not in cls]
               or [b for b in range(256) if b not in cls])
    units = []
    for where in ("first", "last", "lookahead", "before", "none"):
        n = n_slices * SLICE + 777
        g = np.random.default_rng(rnd.getrandbits(32))
        a = np.array(out_cls, dtype=np.uint8)[g.integers(0, len(out_cls), n)]
        for s in range(1, n_slices + 1):
            border = s * SLICE
            L = max(1, run_min + (s % 3) - 1)  # run_min - 1, run_min, run_min + 1
            start = border - L + (s % 2) * min(L // 2, 8)  # ends on the border or crosses it
            run = bytes(rnd.choice(ascii_cls) for _ in range(L))
            plant(a, start, run)
            hb = ((rnd.choice(ascii_cls) | 0x80) if s % 2 else rnd.choice([0x80, 0xc1, 0xe1, 0xff]))
            pos = {"first": border, "last": border - 1, "lookahead": border + rnd.randrange(16), "before": border - 2,
                   "none": None}[where]
            if pos is not None and pos < n:
                a[pos] = hb
        units.append(a)
    # a run across a 64 KiB tile border
    n = 2 * 65536 + 99
    a = np.array(out_cls, dtype=np.uint8)[np.random.default_rng(rnd.getrandbits(32)).integers(0, len(out_cls), n)]
    run = bytes(rnd.choice(ascii_cls) for _ in range(run_min + 1))
    plant(a, 65536 - len(run) // 2, run)
    units.append(a)
    return units


def pattern_units(pat, rnd, info):
    units = small_units(pat, rnd) + edge_units(pat, rnd)
    if info["scan_kernel"] == G.KERNEL_RUN and info["engine"] == G.ENGINE_RUN:
        units += run_units(pat, info["minlen"], rnd)
    return units


# ---- the differential -----------------------------------------------------------------------------------------------
def by_unit(r, n):
    got = [[] for _ in range(n)]
    for fid, s, l in zip(r["file_id"].tolist(), r["start"].tolist(), r["match_len"].tolist()):
        got[fid].append((s, l))
    return got


def check(ctx, p, units, want, what):
    for mode in MODES:
        got = by_unit(ctx.scan(p, units, mode=mode), len(units))
        for i, u in enumerate(units):
            assert got[i] == want[mode][i], (what, mode, i, len(u))


def check_device_packed(ctx, p, units, want, what):
    """the same units resident on the device, packed at 16-byte strides: the bytes behind a unit's end up to the next
    granule are 0xff / 0x80, and the next unit follows at once"""
    starts = np.zeros(len(units), dtype=np.int64)
    lens = np.array([u.size for u in units], dtype=np.int64)
    starts[1:] = np.cumsum((lens[:-1] + 15) & ~15)
    total = int(starts[-1] + ((lens[-1] + 15) & ~15)) + 16
    img = np.tile(np.array([0xff, 0x80], dtype=np.uint8), total // 2 + 1)[:total]
    for s, u in zip(starts, units):
        img[s:s + u.size] = u
    d = ctx.device_alloc(total)
    try:
        ctx.h2d(d, img)
        du = np.zeros(len(units), dtype=G.UNIT_DTYPE)
        du["ptr"] = d + starts.astype(np.uint64)
        du["len"] = lens
        du["file_id"] = np.arange(len(units), dtype=np.uint32)
        du["flags"] = G.UNIT_DEVICE
        for mode in MODES:
            got = by_unit(ctx.scan_units(p, du, mode=mode), len(units))
            for i, u in enumerate(units):
                assert got[i] == want[mode][i], (what, "device", mode, i, len(u))
    finally:
        ctx.device_free(d)


POISON = [np.full(n, b, dtype=np.uint8) for n in (4096, 70000, 33) for b in (0xff, 0x80)]


_T0 = [None]


@pytest.fixture(scope="module", autouse=True)
def _timer():
    _T0[0] = time.time()
    yield
    print("\ntest_gpu_binary: %.1f s" % (time.time() - _T0[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS), ids=str)
def test_binary_differential(variant, monkeypatch):
    monkeypatch.delenv("GSCAN_TILE_SHIFT", raising=False)
    monkeypatch.delenv("GSCAN_HASH_PRE", raising=False)
    monkeypatch.delenv("GSCAN_NO_FIXEDB", raising=False)
    fam = family(variant)
    for pat in VARIANTS[variant]:
        rnd = random.Random("%s|%s" % (variant, pat))
        p = G.Pattern(pat)
        units = pattern_units(pat, rnd, p.info)
        o = O.Regex(pat)
        want = {mode: [o.scan_window(u.tobytes(), mode=mode) for u in units] for mode in MODES}
        assert any(want[G.MODE_ALL]), (pat, "no match planted: the row tests nothing")
        ctx = G.Context(0)  # fresh: nothing left in shared memory or in the segment table by an earlier scan
        try:
            check(ctx, p, units, want, (pat, "fresh"))
            for mode in MODES:
                ctx.scan(p, POISON, mode=mode)
            check(ctx, p, units, want, (pat, "after 0xff/0x80"))
            check_device_packed(ctx, p, units, want, pat)
            if fam in ("FixedBEngine", "RunEngine"):
                for sh in ("12", "16"):
                    monkeypatch.setenv("GSCAN_TILE_SHIFT", sh)
                    check(ctx, p, units, want, (pat, "tile shift", sh))
                monkeypatch.delenv("GSCAN_TILE_SHIFT")
            if fam == "HashEngine":
                for pre in ("0", "1"):
                    monkeypatch.setenv("GSCAN_HASH_PRE", pre)
                    check(ctx, G.Pattern(pat), units, want, (pat, "GSCAN_HASH_PRE", pre))
                monkeypatch.delenv("GSCAN_HASH_PRE")
        finally:
            ctx.close()
