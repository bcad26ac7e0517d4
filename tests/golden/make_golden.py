#!/usr/bin/env python
"""Regenerates tests/golden/*.json by RUNNING THE UNMODIFIED REFERENCE (oracle/_ref/grab_ref,
built by `make -C oracle ref` from /root/reference/src + oracle/shim/pcre.h -> libpcre2-8 10.42)
and, for the minimum-length figures, libpcre2-8.so.0 itself.

The reference ships no tests or golden vectors (SURVEY.md section 4), so these fixtures are the
pin for both the oracle port (oracle/grab_oracle.c) and the CUDA engine.  Run from the repo root:

    make -C oracle ref && python tests/golden/make_golden.py [--big]

--big also regenerates big.json (Appendix B.2 / B.3: 40 MiB and 256 MiB inputs; ~1 min).
ref_stdout.json.gz and host_ref.json hold the reference's output on the inputs that tests/test_oracle_vs_ref.py and
tests/test_hostcheck.py generate (seeded): those tests compare with these recordings instead of running the reference.
"""
import base64
import ctypes
import gzip
import hashlib
import json
import os
import pathlib
import random
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpus  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "grab_ref")


def run_ref(args, cwd=None):
    p = subprocess.run([REF] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=cwd, timeout=600)
    return p.returncode, p.stdout, p.stderr


def b64(b):
    return base64.b64encode(b).decode()


# --------------------------------------------------------------------------------------------
# 1. known-answer cases on tiny inputs (SURVEY.md Appendix B.1 and more edge cases)
# --------------------------------------------------------------------------------------------
T1 = b"xxfoobarxx\nbazquux foo\nnothing\nfoo"
LONGLINE = b"x" * 600 + b"NEEDLE" + b"y" * 600 + b"NEEDLE" + b"zzzzz\n"

KAT = [
    # (name, input bytes, flags, pattern)
    ("alt_all", T1, ["-O", "-l"], "foo|bar|baz|quux"),
    ("alt_lines_off", T1, ["-O"], "foo|bar|baz|quux"),
    ("alt_lines", T1, [], "foo|bar|baz|quux"),
    ("single_off", T1, ["-s", "-O", "-l"], "foo|bar"),
    ("single_line", T1, ["-s"], "foo"),
    ("l_only", T1, ["-l"], "foo"),
    ("q2_capture", T1, ["-O", "-l"], "(foo|bar|baz|quux)"),
    ("q2_noncapture", T1, ["-O", "-l"], "(?:foo|bar|baz|quux)"),
    ("skip_small", b"fo", ["-O", "-l"], "foo"),
    ("q1_exact", b"foo", ["-O", "-l"], "foo"),
    ("q1_foofoo", b"foofoo", ["-O", "-l"], "foo"),
    ("q1_foofoox", b"foofoox", ["-O", "-l"], "foo"),
    ("xfoo", b"xfoo", ["-O", "-l"], "foo"),
    ("nonoverlap", b"aaaaa\n", ["-O", "-l"], "aa"),
    ("first_alt", b"xabcx\n", ["-O"], "ab|abc"),
    ("first_alt2", b"xabcx\n", ["-O", "-l"], "abc|ab"),
    ("classrun", b"a" * 20 + b" " + b"B_9" * 11 + b" short\n", ["-O", "-l"], "[A-Za-z0-9_]{16,}"),
    ("icase", b"FoO fOo\n", ["-O", "-l"], "(?i)foo"),
    ("q1_run16", b"a" * 16, ["-O", "-l"], "[A-Za-z0-9_]{16,}"),
    ("q1_run17", b"a" * 17, ["-O", "-l"], "[A-Za-z0-9_]{16,}"),
    ("longline", LONGLINE, ["-O"], "NEEDLE"),
    ("longline_noO", LONGLINE, [], "NEEDLE"),
    ("empty_file", b"", ["-O", "-l"], "a"),
    ("one_byte", b"a", ["-O", "-l"], "a"),
    ("two_byte", b"aa", ["-O", "-l"], "a"),
    ("three_byte", b"aaa", ["-O", "-l"], "a"),
    ("dot", b"a.c abc a\nc\n", ["-O", "-l"], "a.c"),
    ("dot_nl", b"a\nc a\n\nc", ["-O", "-l"], "a..c"),
    ("esc", b"1+1=2 1.1 (x) [y] {z} a|b \\ ^ $", ["-O", "-l"], r"\+|\.|\(|\)|\[|\]|\{|\}|\||\\|\^|\$"),
    ("digits", b"tel 555-1234 or 5551234, 12-3456\n", ["-O", "-l"], r"\d\d\d-\d\d\d\d"),
    ("word", b"a_b c-d\tE9 \n", ["-O", "-l"], r"\w\w\w"),
    ("space", b"a b\tc\nd\x0be\x0cf\rg", ["-O", "-l"], r"\s"),
    ("nonspace", b"  ab  c \n", ["-O", "-l"], r"\S+"),
    ("negclass", b"abc,def;ghi\n", ["-O", "-l"], r"[^,;\n]+"),
    ("hexesc", b"a\x00b\xffc\x80\n", ["-O", "-l"], r"\x00|\xff|\x80"),
    ("highbytes", bytes(range(256)) * 2, ["-O", "-l"], r"[\x80-\xff]{8,}"),
    ("plus", b"aaa b aa\n", ["-O", "-l"], "a+"),
    ("exact_rep", b"aaaaaaa\n", ["-O", "-l"], "a{3}"),
    ("bounded_rep", b"aaaaaaaaaa b aaaa\n", ["-O", "-l"], "a{2,4}"),
    ("bounded_rep2", b"0123456789012 12 123\n", ["-O", "-l"], r"\d{3,5}"),
    ("opt", b"color colour colr\n", ["-O", "-l"], "colou?r"),
    ("star", b"ac abc abbbc\n", ["-O", "-l"], "ab*c"),
    ("lazy", b"<a><b>\n", ["-O", "-l"], "<.+?>"),
    ("greedy", b"<a><b>\n", ["-O", "-l"], "<.+>"),
    ("seq", b"foo123bar foo1bar foobar\n", ["-O", "-l"], r"foo\d+bar"),
    ("group_rep", b"abab ab ababab\n", ["-O", "-l"], "(?:ab){2,}"),
    ("icase_class", b"Hello hELLO\n", ["-O", "-l"], "(?i)h[a-z]+o"),
    ("icase_group", b"abAB aB\n", ["-O", "-l"], "(?i:a)b"),
    ("posix", b"ab12 cd\n", ["-O", "-l"], "[[:alpha:]]+[[:digit:]]+"),
    ("class_edge", b"a]b-c^d\n", ["-O", "-l"], r"[]^-]"),
    ("selfoverlap", b"abababababab\n", ["-O", "-l"], "abab"),
    ("selfoverlap2", b"aaaaaaaaaaa", ["-O", "-l"], "aaa"),
    ("prefix_alt", b"foobar foo fo\n", ["-O", "-l"], "fo|foo|foobar"),
    ("prefix_alt2", b"foobar foo fo\n", ["-O", "-l"], "foobar|foo|fo"),
    ("anchor_bol", b"foo\nfoo\n", ["-O", "-l"], "^foo"),
    ("anchor_eol", b"foo\nfoo", ["-O", "-l"], "foo$"),
    ("wordb", b"foo foobar barfoo foo\n", ["-O", "-l"], r"\bfoo\b"),
    ("quoted", b"a.b a+b axb\n", ["-O", "-l"], r"\Qa.b\E|a\+b"),
    ("nl_in_pat", b"ab\ncd\nab\ncd", ["-O", "-l"], "b\\nc"),
    ("line_two_on_line", b"foo bar foo\nfoo\n", [], "foo"),
    ("line_two_on_line_O", b"foo bar foo\nfoo\n", ["-O"], "foo"),
    ("tail_nl", b"abc\nfoo", ["-O", "-l"], "foo"),
    # Q2 in full: pcre_exec (ovecsize 3) returns 0 only for a match in which a capturing group TOOK PART -- the loop prints
    # until the first such match and leaves the window there
    ("q2_alt_mixed", b"foo bar foo\nfoo\n", ["-O", "-l"], "foo|(bar)"),
    ("q2_alt_mixed_lines", b"foo x\nfoo bar foo\nfoo\n", [], "foo|(bar)"),
    ("q2_opt_group", b"foo xfoo foo\n", ["-O", "-l"], "(x)?foo"),
    ("q2_opt_group_lines", b"foo\nzfoo\nxfoo\nfoo\n", [], "(x)?foo"),
    ("q2_group_in_rep", b"bc abc bc\n", ["-O", "-l"], "(?:(a)|b)+c"),
    ("q2_group_in_rep2", b"b ab b\n", ["-O", "-l"], "(?:(a)|b)+c"),
    ("q2_backtracked_group", b"ab ab aab ab\n", ["-O", "-l"], "(a)?ab"),
    ("q2_star_group", b"b b ab b\n", ["-O", "-l"], "(a)*b"),
    ("q2_always", b"bc abc bc\n", ["-O", "-l"], "(a|b)"),
    ("q2_nested_noncap", b"xy xzy xy\n", ["-O", "-l"], "x(?:(z)|)y"),
    ("q2_single", b"foo bar foo\n", ["-s", "-O", "-l"], "foo|(bar)"),
    ("q2_first_is_group", b"bar foo foo\n", ["-O", "-l"], "foo|(bar)"),
    # look-arounds, atomic groups, possessive quantifiers (round 2: served by the device VM)
    ("look_behind", b"foobar xbar foobar\n", ["-O", "-l"], "(?<=foo)bar"),
    ("look_ahead", b"foobar foobaz foobar\n", ["-O", "-l"], "foo(?=bar)"),
    ("look_ahead_neg", b"foobar foobaz foo\n", ["-O", "-l"], "foo(?!bar)"),
    ("look_behind_neg", b"xbar bar ybar\n", ["-O", "-l"], "(?<!x)bar"),
    ("look_behind_neg_lines", b"xbar bar\nybar\nbar\n", [], "(?<!x)bar"),
    ("atomic", b"aaab aaa ab\n", ["-O", "-l"], "(?>a+)b"),
    ("atomic_nomatch", b"aaab ab\n", ["-O", "-l"], "(?>a+)ab"),
    ("possessive_set", b"aaab ab b\n", ["-O", "-l"], "a++b"),
    ("possessive_group", b"ababc abab abc\n", ["-O", "-l"], "(?:ab)++c"),
    ("possessive_group2", b"ababab\n", ["-O", "-l"], "(?:ab)*+ab"),
    ("look_behind_alt", b"ad bcd cd xd\n", ["-O", "-l"], "(?<=a|bc)d"),
    ("look_behind_neg_alt", b"ad bcd cd xd d\n", ["-O", "-l"], "(?<!a|bc)d"),
    ("look_ahead_word", b"one three two four\n", ["-O", "-l"], r"\b(?=\w{3}\b)\w+"),
    ("look_ahead_line", b"abcz\nabc\nazz\n", ["-O", "-l"], r"(?=.*z)a\w+"),
    ("look_ahead_neg_line", b"xab y\nxab\n", ["-O", "-l"], r"x(?!.*y)\w*"),
    ("look_behind_bol", b"ab,cd,ef\ngh\n", ["-O", "-l"], r"(?<=^|,)\w+"),
    ("look_behind_icase", b"fooBAR FOObar\n", ["-O", "-l"], "(?i)(?<=FOO)bar"),
    ("look_behind_digits", b"123-456 12-34 1234-5\n", ["-O", "-l"], r"(?<=\d{3})-\d+"),
    ("q2_group_in_lookahead", b"foobar foobaz\n", ["-O", "-l"], "foo(?=(bar))"),
    ("q2_group_in_neg_lookahead", b"ab b\n", ["-O", "-l"], "(?!(a))b"),
    ("look_at_window_start", b"barfoobar\n", ["-O", "-l"], "(?<=foo)bar|bar"),
    ("bigalt", b"the quick brown fox jumps over the lazy dog\n" * 3, ["-O", "-l"],
     "fox|dog|the|quick|lazy|over|jumps|brown"),
]

MULTI = [
    # (name, [(filename, bytes)], flags, pattern, paths as given on the command line)
    ("two_paths", [("t1.txt", T1), ("t2.txt", T1)], ["-O", "-l"], "quux", ["t1.txt", "t2.txt"]),
    ("two_paths_lines", [("t1.txt", T1), ("t2.txt", b"quux\n")], [], "quux", ["t1.txt", "t2.txt"]),
    ("two_paths_l", [("t1.txt", T1), ("t2.txt", b"zzz\n")], ["-l"], "quux", ["t1.txt", "t2.txt"]),
]

RECURSIVE = [
    ("rec_off", {"d/a": T1, "d/sub/b": T1, "d/sub/c": b"nothing here\n"}, ["-r", "-O", "-l"], "quux", "d"),
    ("rec_l", {"d/a": T1, "d/sub/b": T1}, ["-r", "-l"], "quux", "d"),
    ("rec_n2", {"d/a": T1, "d/sub/b": T1, "d/x/y/z": b"qquuxquux"}, ["-n", "2", "-r", "-O", "-l"], "quux", "d"),
]

# --------------------------------------------------------------------------------------------
# 2. seeded differential cases: random inputs over small alphabets x patterns
# --------------------------------------------------------------------------------------------
DIFF_PATTERNS = [
    "ab", "aa", "aba", "abab", "a", "abc|bc|c", "ab|abc", "abc|ab", "a|b", "aab|ab|b",
    "[ab]{3,}", "[ab]{2}", "a{2,}", "b+", "[^a\\n]{2,}", "a.b", "a..", "(?i)AB", "(?:ab|ba)a",
    "a[ab]b", "ab{2}", "[a-c]{4,}", "b[^b]b", "abcabc", "cab|abc|bca",
]
ALPHABETS = [b"ab", b"abc", b"ab\n", b"abc \n"]


def diff_cases(n_per=3, seed=20260924):
    rnd = random.Random(seed)
    out = []
    for pi, pat in enumerate(DIFF_PATTERNS):
        for k in range(n_per):
            alpha = ALPHABETS[(pi + k) % len(ALPHABETS)]
            ln = rnd.choice([0, 1, 2, 3, 5, 8, 13, 31, 64, 100, 257, 600])
            data = bytes(rnd.choice(alpha) for _ in range(ln))
            out.append(("diff_%d_%d" % (pi, k), data, ["-O", "-l"], pat))
    return out


def offsets_of(stdout):
    offs = []
    for line in stdout.split(b"\n"):
        if line.startswith(b"Match at offset "):
            offs.append(int(line[len(b"Match at offset "):]))
    return offs


def gen_small():
    cases = []
    with tempfile.TemporaryDirectory() as td:
        for name, data, flags, pat in KAT + diff_cases():
            fn = os.path.join(td, "in.bin")
            with open(fn, "wb") as f:
                f.write(data)
            rc, so, se = run_ref(flags + [pat, fn])
            cases.append({"name": name, "input": b64(data), "flags": flags, "pattern": pat,
                          "rc": rc, "stdout": b64(so)})
    multi = []
    for name, files, flags, pat, paths in MULTI:
        with tempfile.TemporaryDirectory() as td:
            for fn, data in files:
                with open(os.path.join(td, fn), "wb") as f:
                    f.write(data)
            rc, so, se = run_ref(flags + [pat] + paths, cwd=td)
            multi.append({"name": name, "files": [[fn, b64(d)] for fn, d in files], "flags": flags,
                          "pattern": pat, "paths": paths, "rc": rc, "stdout": b64(so)})
    rec = []
    for name, tree, flags, pat, root in RECURSIVE:
        with tempfile.TemporaryDirectory() as td:
            for fn, data in tree.items():
                os.makedirs(os.path.dirname(os.path.join(td, fn)), exist_ok=True)
                with open(os.path.join(td, fn), "wb") as f:
                    f.write(data)
            rc, so, se = run_ref(flags + [pat, root], cwd=td)
            # cross-file order is readdir order (Q6): parity is on SORTED lines (README.md:206-215)
            rec.append({"name": name, "tree": {k: b64(v) for k, v in tree.items()}, "flags": flags,
                        "pattern": pat, "root": root, "rc": rc,
                        "sorted_lines": [b64(l) for l in sorted(so.split(b"\n")) if l]})
    # CLI error surface (SURVEY.md section 8(b), "exit codes")
    cli = []
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "dir"))
        with open(os.path.join(td, "f"), "wb") as f:
            f.write(T1)
        for name, args in [("usage", []), ("usage1", ["foo"]), ("badregex", ["(", "f"]), ("missing", ["foo", "nope"]),
                           ("n_without_r", ["-n", "2", "foo", "f"]), ("dir_no_r", ["foo", "dir"]),
                           ("badflag", ["-Z", "foo", "f"])]:
            rc, so, se = run_ref(args, cwd=td)
            cli.append({"name": name, "args": args, "rc": rc, "stdout": b64(so), "stderr": b64(se)})
    return {"cases": cases, "multi": multi, "recursive": rec, "cli": cli}


# --------------------------------------------------------------------------------------------
# 3. PCRE_INFO_MINLENGTH straight from libpcre2-8 (grab.cc:120)
# --------------------------------------------------------------------------------------------
MINLEN_PATTERNS = sorted(set([c[3] for c in KAT] + DIFF_PATTERNS + [
    "foobardoesnotexist", "[A-Za-z0-9_]{16,}", "(foo|bar|baz|quux)", "a{3,5}b", "(?:a|bc)(?:d|efg)", "x*y",
    "a?b?c", "(?i)linus", "[[:alpha:]]{2}x", "ab|", "(a)(b)?c", r"\d{3}-\d{4}", "a|b{2}|c{3}", corpus.literals100(),
]))


def gen_minlen():
    lib = ctypes.CDLL("libpcre2-8.so.0")
    lib.pcre2_compile_8.restype = ctypes.c_void_p
    lib.pcre2_compile_8.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32,
                                    ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    lib.pcre2_pattern_info_8.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]
    out = []
    for p in MINLEN_PATTERNS:
        ec, eo = ctypes.c_int(0), ctypes.c_size_t(0)
        pb = p.encode("latin-1")
        code = lib.pcre2_compile_8(pb, len(pb), 0, ctypes.byref(ec), ctypes.byref(eo), None)
        if not code:
            out.append({"pattern": p, "compiles": False})
            continue
        v = ctypes.c_uint32(0)
        lib.pcre2_pattern_info_8(code, 16, ctypes.byref(v))      # PCRE2_INFO_MINLENGTH
        ncap = ctypes.c_uint32(0)
        lib.pcre2_pattern_info_8(code, 4, ctypes.byref(ncap))    # PCRE2_INFO_CAPTURECOUNT
        out.append({"pattern": p, "compiles": True, "minlen": v.value, "captures": ncap.value})
    return out


# --------------------------------------------------------------------------------------------
# 4. big inputs (recipes in tests/corpus.py): Appendix B.2 chunk overlap, Appendix B.3 256 MiB
# --------------------------------------------------------------------------------------------
def gen_big():
    out = {"overlap": [], "b3": [], "synth": []}
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
        fn = os.path.join(td, "ov.bin")
        corpus.overlap_file().tofile(fn)
        for flags in (["-L"] * 5 + ["-O", "-l"], ["-O", "-l"]):
            rc, so, se = run_ref(flags + ["NEEDLE", fn])
            out["overlap"].append({"gen": "overlap_file", "flags": flags, "pattern": "NEEDLE", "offsets": offsets_of(so)})
        corpus.overlap_run_file().tofile(fn)
        for flags in (["-L"] * 5 + ["-O", "-l"], ["-O", "-l"]):
            rc, so, se = run_ref(flags + ["[A-Za-z0-9_]{16,}", fn])
            out["overlap"].append({"gen": "overlap_run_file", "flags": flags, "pattern": "[A-Za-z0-9_]{16,}",
                                   "offsets": offsets_of(so)})
        # B.3
        a = corpus.b3_corpus()
        out["b3_file_md5"] = hashlib.md5(a.tobytes()).hexdigest()
        fn = os.path.join(td, "f256")
        a.tofile(fn)
        for pat in ["foobardoesnotexist", "foo|bar|baz|quux", "[A-Za-z0-9_]{16,}", "qz", corpus.literals100(),
                    "(?i)linus", "e{2,}", r"\d{5}"]:
            rc, so, se = run_ref(["-O", "-l", pat, fn])
            offs = offsets_of(so)
            txt = "".join("%d\n" % o for o in offs).encode()
            out["b3"].append({"pattern": pat, "n": len(offs), "md5": hashlib.md5(txt).hexdigest(),
                              "first": offs[:3], "last": offs[-1:]})
        # a 32 MiB prefix of the same stream: small enough for the (slow) oracle port on CPU
        fn2 = os.path.join(td, "f32")
        a[:32 << 20].tofile(fn2)
        out["b3_32"] = []
        for pat in ["foobardoesnotexist", "foo|bar|baz|quux", "[A-Za-z0-9_]{16,}", "qz", corpus.literals100()]:
            rc, so, se = run_ref(["-O", "-l", pat, fn2])
            offs = offsets_of(so)
            txt = "".join("%d\n" % o for o in offs).encode()
            out["b3_32"].append({"pattern": pat, "n": len(offs), "md5": hashlib.md5(txt).hexdigest()})
        # the bench generator (device twin in grab_b200/csrc/corpus_gen.cu): 8 files x 1 MiB, seed 2
        os.makedirs(os.path.join(td, "syn"))
        needle = b"foobardoesexist"
        for fid in range(8):
            corpus.synth_file(2, fid, 1 << 20, needle, 4).tofile(os.path.join(td, "syn", "f%03d" % fid))
        for pat in ["foobardoesexist", "foo|bar|baz|quux", "[A-Za-z0-9_]{16,}", corpus.literals100()]:
            per_file = {}
            for fid in range(8):
                rc, so, se = run_ref(["-O", "-l", pat, os.path.join(td, "syn", "f%03d" % fid)])
                per_file[str(fid)] = offsets_of(so)
            out["synth"].append({"seed": 2, "file_len": 1 << 20, "needle": needle.decode(), "needle_every": 4,
                                 "pattern": pat, "offsets": per_file})
    return out


# --------------------------------------------------------------------------------------------
# 5. the reference's output on the seeded inputs of test_oracle_vs_ref.py and test_hostcheck.py
# --------------------------------------------------------------------------------------------
def gen_ref_stdout():
    """Runs each test of test_oracle_vs_ref.py once with its lookup of the recording replaced by a run of the reference,
    so the recording holds exactly the (pattern, flags, input) triples the tests ask for."""
    import test_oracle_vs_ref as T
    rows = {}

    def run(pattern, data, flags=("-O", "-l")):
        k = (pattern, tuple(flags), T.input_key(data))
        with tempfile.NamedTemporaryFile() as f:
            f.write(data)
            f.flush()
            try:
                p = subprocess.run([REF] + list(flags) + [pattern, f.name], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                                   timeout=T.REF_TIMEOUT_S)
            except subprocess.TimeoutExpired:
                rows[k] = None
                raise
        assert p.returncode == 0, p.stderr
        rows[k] = T.digest(p.stdout)
        return rows[k]

    T.ref_stdout = run
    for name in ("test_random_patterns_stdout_identical", "test_inline_options_ungreedy_extended_comment",
                 "test_minlen_quirk_q1_against_reference", "test_long_lines_line_mode_against_reference",
                 "test_binary_inputs_stdout_identical"):
        getattr(T, name)()
    return [[pat, list(flags), key, d] for (pat, flags, key), d in sorted(rows.items(), key=lambda kv: json.dumps(kv[0]))]


def gen_host_ref():
    import test_hostcheck as H
    out = {"tree": {}, "f4": {}}
    with tempfile.TemporaryDirectory() as td:
        H._tree(pathlib.Path(td))
        for flags in H.TREE_FLAGS:
            rc, so, se = run_ref(flags + ["foo|bar|baz|quux", "tree"], cwd=td)
            assert rc == 0, se
            out["tree"][" ".join(flags)] = H.sorted_lines_digest(so)
    with tempfile.TemporaryDirectory() as td:
        fn = os.path.join(td, "big.bin")
        H._f4_file(fn)
        for flags in H.F4_FLAGS:
            rc, so, se = run_ref(["-L"] * 5 + flags + ["NEEDLE", fn])
            assert rc == 0, se
            out["f4"][" ".join(flags)] = b64(so)
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "a"), "wb") as f:
            f.write(b"xx foo yy\nzz foo\n\n")
        rc, so, se = run_ref(["-O", "-l", "foo", "a", "nope"], cwd=td)
        out["good_then_missing"] = {"rc": rc, "stdout": b64(so), "stderr": b64(se)}
    return out


def main():
    if not os.path.exists(REF):
        sys.exit("build the reference first: make -C oracle ref")
    with open(os.path.join(HERE, "kat.json"), "w") as f:
        json.dump(gen_small(), f, indent=0)
    with open(os.path.join(HERE, "minlen.json"), "w") as f:
        json.dump(gen_minlen(), f, indent=0)
    rows = gen_ref_stdout()
    with open(os.path.join(HERE, "ref_stdout.json.gz"), "wb") as f:
        f.write(gzip.compress(json.dumps(rows, indent=0).encode(), 9, mtime=0))
    host = gen_host_ref()
    with open(os.path.join(HERE, "host_ref.json"), "w") as f:
        json.dump(host, f, indent=1)
    if "--big" in sys.argv:
        with open(os.path.join(HERE, "big.json"), "w") as f:
            json.dump(gen_big(), f, indent=0)


if __name__ == "__main__":
    main()
