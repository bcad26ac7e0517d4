"""Pins the oracle port to the UNMODIFIED reference binary (grab master built against the PCRE2 shim) on seeded random
patterns x random inputs, and to GNU grep -P (same libpcre2) as an independent second opinion.  CPU only.

The reference's stdout for every (pattern, flags, input) compared here is recorded in tests/golden/ref_stdout.json.gz
(sha-256 digests, written by tests/golden/make_golden.py from a run of the reference), so the comparison needs neither
the reference's sources nor its binary."""
import functools
import gzip
import hashlib
import json
import os
import random
import shutil
import subprocess

import pytest

import oracle_py as O
from test_gpu_random_patterns import gen_pattern

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "ref_stdout.json.gz")
REF_TIMEOUT_S = 20  # a reference run longer than this was recorded as a timeout: the pattern is not compared


def digest(stdout):
    return hashlib.sha256(stdout).hexdigest()[:32]


def input_key(data):
    return hashlib.sha256(data).hexdigest()[:16]


@functools.lru_cache(maxsize=None)
def recorded():
    """(pattern, flags, input key) -> digest of the reference's stdout, or None where its run timed out."""
    with gzip.open(GOLDEN, "rt") as f:
        return {(pat, tuple(flags), key): d for pat, flags, key, d in json.load(f)}


def ref_stdout(pattern, data, flags=("-O", "-l")):
    """Digest of the reference's stdout for `grab <flags> <pattern> <file holding data>`; raises
    subprocess.TimeoutExpired where the reference's run timed out when it was recorded."""
    k = (pattern, tuple(flags), input_key(data))
    assert k in recorded(), "no recorded reference output for %r: regenerate %s" % (k, GOLDEN)
    if recorded()[k] is None:
        raise subprocess.TimeoutExpired(["grab"] + list(flags) + [pattern], REF_TIMEOUT_S)
    return recorded()[k]


def random_inputs(rnd, n):
    out = []
    for k in range(n):
        alpha = [b"abc", b"abcx \n", b"ab", b"abc abc\n\n", b"aabbcc_x1 \t\n"][k % 5]
        ln = rnd.choice([0, 1, 2, 3, 7, 16, 33, 64, 130, 300, 513])
        out.append(bytes(rnd.choice(alpha) for _ in range(ln)))
    return out


def test_random_patterns_stdout_identical():
    rnd = random.Random(20260924)
    inputs = random_inputs(rnd, 10)
    checked = 0
    for _ in range(150):
        pat = gen_pattern(rnd)
        try:
            o = O.Regex(pat)
        except O.OracleError:
            continue
        if o.nullable:  # the reference never terminates on these (Q4)
            continue
        try:
            for flags, kw in ((("-O", "-l"), dict(offsets=True, line=False)), ((), dict()), (("-s", "-O"), dict(offsets=True, single=True))):
                for data in inputs:
                    assert digest(o.grab(data, **kw)) == ref_stdout(pat, data, flags), (pat, flags, len(data))
        except (O.OracleError, subprocess.TimeoutExpired):
            continue  # pathological backtracking: either side hit its match limit / time budget
        checked += 1
    assert checked >= 60


OPTION_PATTERNS = [r"(?U)a+b", r"(?U)a+?b", r"(?U)a{2,}", r"(?U)\w+ ", r"(?U:a+)b", r"(?U)a*b", r"(?U)(?:ab)+c", r"a(?U)b+c?", r"(?U)a++b",
                   r"(?x) a b c", "(?x)a b # comment\n c", r"(?x)a\ b", r"(?x)a[ ]b", r"(?x)a +b", r"(?xi)A B", r"(?x)a b | b c", r"a(?x) b c",
                   r"(?x)a{2} b", r"(?x: a b ) c", r"(?x) [ab] {2} c", "(?x)# only a comment\nab",
                   r"a(?#hello)b", r"(?#c)a|b(?#d)c", r"a(?#x)+b"]


def test_inline_options_ungreedy_extended_comment():
    """(?U), (?x) and (?#...) as the reference's PCRE build treats them: identical stdout in all three output modes."""
    rnd = random.Random(5)
    inputs = random_inputs(rnd, 15) + [b"aaab ab\nfoo  bar # x\nabcabc aXb a\nb\n", b"a b c abc a  b\n", b"aab aaab abbc abc\n"]
    checked = 0
    for pat in OPTION_PATTERNS:
        o = O.Regex(pat)
        if o.nullable:
            continue
        for data in inputs:
            for flags, kw in ((("-O", "-l"), dict(offsets=True, line=False)), ((), dict()), (("-s", "-O"), dict(offsets=True, single=True))):
                assert digest(o.grab(data, **kw)) == ref_stdout(pat, data, flags), (pat, flags, data)
        checked += 1
    assert checked >= 20


def test_minlen_quirk_q1_against_reference():
    # the strict '<' of grab.cc:175 for every length around minlen
    for pat, unit in (("abc", b"abc"), ("[ab]{4,}", b"abab"), ("ab|abcd", b"ab")):
        o = O.Regex(pat)
        for reps in range(0, 4):
            for tail in (b"", b"x", b"\n"):
                data = unit * reps + tail
                assert digest(o.grab(data, offsets=True, line=False)) == ref_stdout(pat, data), (pat, data)


@pytest.mark.skipif(shutil.which("grep") is None, reason="no grep")
def test_second_opinion_gnu_grep_P(tmp_path):
    """grep -P -a -b -o prints every non-overlapping match start like the reference's -O -l, except for the reference's
    quirks (Q1 tail, Q2 captures) and for matches that span '\\n' -- so: inputs end in '\\n', patterns cannot match '\\n'."""
    probe = subprocess.run(["grep", "-P", "-a", "-b", "-o", "a", "/dev/null"], stderr=subprocess.PIPE)
    if probe.returncode not in (0, 1):
        pytest.skip("grep -P unavailable")
    rnd = random.Random(7)
    pats = ["foo|bar|baz|quux", "[A-Za-z0-9_]{5,}", "qz", r"\d{2}-\d{2}", "(?i)ab+c", r"a[^b\n]*b", r"\bfoo\b", "x+y+?"]
    for pat in pats:
        o = O.Regex(pat)
        for _ in range(6):
            lines = []
            for _ in range(rnd.randint(1, 40)):
                lines.append(bytes(rnd.choice(b"abcfoqzxy019-_ Bbar") for _ in range(rnd.randint(0, 60))))
            data = b"\n".join(lines) + b"\n"
            p = tmp_path / "g"
            p.write_bytes(data)
            g = subprocess.run(["grep", "-P", "-a", "-b", "-o", pat, str(p)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            assert g.returncode in (0, 1), g.stderr
            want = [int(l.split(b":", 1)[0]) for l in g.stdout.split(b"\n") if l]
            got = [s for s, _ in o.scan_window(data)]
            assert got == want, (pat, data)


def test_binary_inputs_stdout_identical():
    """Every pattern of test_scan_variants.VARIANTS (high bytes, NUL, (?i) next to bytes >= 0x80 -- which PCRE's C locale does
    not fold) on seeded binary inputs of test_gpu_binary's generators: the oracle the GPU tests trust holds on binary input."""
    import numpy as np
    from test_gpu_binary import small_units
    from test_scan_variants import VARIANTS
    checked = 0
    for key in sorted(VARIANTS, key=str):
        for pat in VARIANTS[key]:
            o = O.Regex(pat)
            units = small_units(pat, random.Random("ref|" + pat))
            for u in (units[62], units[-1]):  # 63 bytes of text salted with high bytes, 4096 uniform bytes
                data = np.asarray(u, dtype=np.uint8).tobytes()
                for flags, kw in ((("-O", "-l"), dict(offsets=True, line=False)), ((), dict()), (("-s", "-O"), dict(offsets=True, single=True))):
                    assert digest(o.grab(data, **kw)) == ref_stdout(pat, data, flags), (pat, flags, len(data))
                    checked += 1
    assert checked >= 300


def test_long_lines_line_mode_against_reference():
    """Line output on lines longer than the 511 bytes the reference prints behind a match (grab.cc:194-196): the next search
    resumes in the middle of the line -- for class runs possibly in the middle of a run, where PCRE then reports a match at
    the resume point itself.  The resolve pass's chain path for class runs (k_chain_next / k_chain_entry) is built on
    exactly this behaviour of the oracle: pinned here against the unmodified reference's stdout, line mode and -O."""
    rnd = random.Random(511)
    inputs = []
    for alpha, n, newline_every in ((b"ab", 700, 0), (b"ab", 3000, 0), (b"aab_ 1", 2500, 0), (b"abc ", 4000, 1300), (b"aab_1 \n", 3000, 0),
                                    (b"a", 1200, 0), (b"ab", 511, 0), (b"ab", 512, 0), (b"ab", 1023, 0), (b"ab", 1024, 0)):
        b = bytearray(rnd.choice(alpha) for _ in range(n))
        if newline_every:
            for i in range(newline_every, n, newline_every):
                b[i] = 10
        inputs.append(bytes(b))
    pats = ["[ab]{2,}", "[ab]{5,}", "a{3,}", "\\w{3,}", "[^b]{2,}", "[a_1]{2,}", "[ab\\n]{4,}", "ab", "aa|ab", "ab+a", "a[ab]*b", "\\w+ ", "a+"]
    checked = 0
    for pat in pats:
        o = O.Regex(pat)
        for i, data in enumerate(inputs):
            for flags, kw in (((), dict()), (("-O",), dict(offsets=True)), (("-O", "-l"), dict(offsets=True, line=False))):
                assert digest(o.grab(data, **kw)) == ref_stdout(pat, data, flags), (pat, flags, i, len(data))
                checked += 1
    assert checked == len(pats) * len(inputs) * 3
