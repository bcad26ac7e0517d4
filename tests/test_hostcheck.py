"""Host side of the product on a box WITHOUT a GPU: grab_b200/host (FileGrep mirror, batching, scan lanes, output
sequencer, command line) linked against a test double of the engine ABI (tests/hostcheck/gscan_double.c, which
answers gscan_scan_batch() with the CPU oracle).  Expected bytes are the ones recorded from the unmodified
reference binary (tests/golden/kat.json, tests/golden/host_ref.json) or produced by the oracle's FileGrep::find
restatement here.

The double is test infrastructure: grab_b200/bin/grab-b200 links libgscan.so and fails loudly without a GPU."""
import base64
import functools
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import oracle_py as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KAT = json.load(open(os.path.join(HERE, "golden", "kat.json")))
BUILD = os.path.join(HERE, "_build")
BIN = os.path.join(BUILD, "grab-hostcheck")

LANES = [dict(), dict(GRAB_B200_NDEV="2", GRAB_B200_LANES="2", GRAB_B200_BATCH_BYTES="1", GSCAN_DOUBLE_JITTER="1")]
LANE_IDS = ["1lane", "2gpu_x2lanes_jitter"]


@pytest.fixture(scope="module", autouse=True)
def hostcheck_binary():
    os.makedirs(BUILD, exist_ok=True)
    srcs = [os.path.join(ROOT, "grab_b200", "host", f) for f in ("filegrep.cc", "filegrep.h", "main.cc")]
    srcs += [os.path.join(HERE, "hostcheck", "gscan_double.c"), os.path.join(ROOT, "oracle", "grab_oracle.c"),
             os.path.join(ROOT, "include", "gscan.h")]
    if os.path.exists(BIN) and all(os.path.getmtime(BIN) >= os.path.getmtime(s) for s in srcs):
        return
    cc = ["gcc", "-O2", "-Wall", "-c"]
    subprocess.run(cc + [os.path.join(HERE, "hostcheck", "gscan_double.c"), "-o", os.path.join(BUILD, "gscan_double.o")], check=True)
    subprocess.run(cc + [os.path.join(ROOT, "oracle", "grab_oracle.c"), "-o", os.path.join(BUILD, "grab_oracle.o")], check=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", os.path.join(ROOT, "grab_b200", "host", "filegrep.cc"),
                    os.path.join(ROOT, "grab_b200", "host", "main.cc"), os.path.join(BUILD, "gscan_double.o"),
                    os.path.join(BUILD, "grab_oracle.o"), "-pthread", "-o", BIN], check=True)


@functools.lru_cache(maxsize=None)
def host_ref():
    """The reference's output on the inputs of the tests below (written by tests/golden/make_golden.py)."""
    return json.load(open(os.path.join(HERE, "golden", "host_ref.json")))


def run(args, cwd=None, env=None, binary=None):
    e = dict(os.environ)
    for k in [k for k in e if k.startswith("GRAB_B200_") or k.startswith("GSCAN_DOUBLE_")]:
        del e[k]
    if env:
        e.update(env)
    p = subprocess.run([binary or BIN] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=cwd, env=e, timeout=300)
    return p.returncode, p.stdout, p.stderr


def oracle_ok(pat):
    try:
        O.Regex(pat)
        return True
    except O.OracleError:
        return False


@pytest.mark.parametrize("lanes", LANES, ids=LANE_IDS)
@pytest.mark.parametrize("case", KAT["cases"], ids=lambda c: c["name"])
def test_host_stdout(case, lanes, tmp_path):
    if not oracle_ok(case["pattern"]):
        pytest.skip("pattern outside the oracle's subset")
    fn = tmp_path / "in.bin"
    fn.write_bytes(base64.b64decode(case["input"]))
    rc, so, se = run(case["flags"] + [case["pattern"], str(fn)], env=lanes)
    assert rc == case["rc"], se
    assert so == base64.b64decode(case["stdout"])


@pytest.mark.parametrize("lanes", LANES, ids=LANE_IDS)
@pytest.mark.parametrize("case", KAT["multi"], ids=lambda c: c["name"])
def test_host_multi_path(case, lanes, tmp_path):
    for fn, d in case["files"]:
        (tmp_path / fn).write_bytes(base64.b64decode(d))
    rc, so, se = run(case["flags"] + [case["pattern"]] + case["paths"], cwd=str(tmp_path), env=lanes)
    assert rc == case["rc"], se
    assert so == base64.b64decode(case["stdout"])


@pytest.mark.parametrize("lanes", LANES, ids=LANE_IDS)
@pytest.mark.parametrize("case", KAT["recursive"], ids=lambda c: c["name"])
def test_host_recursive_sorted(case, lanes, tmp_path):
    for fn, d in case["tree"].items():
        p = tmp_path / fn
        p.parent.mkdir(parents=True, exist_ok=True)
        p.write_bytes(base64.b64decode(d))
    rc, so, se = run(case["flags"] + [case["pattern"], case["root"]], cwd=str(tmp_path), env=lanes)
    assert rc == case["rc"], se
    assert sorted(l for l in so.split(b"\n") if l) == [base64.b64decode(l) for l in case["sorted_lines"]]


def sorted_lines_digest(stdout):
    """The reference's line order across files is readdir order (Q6): output is compared as a sorted multiset of lines."""
    return hashlib.sha256(b"\n".join(sorted(stdout.split(b"\n")))).hexdigest()


def _tree(tmp_path, n_files=300, seed=5):
    rng = np.random.default_rng(seed)
    words = [b"foo", b"bar", b"baz", b"quux", b"lorem", b"ipsum", b"dolor", b"\n", b" ", b"sit", b"\n"]
    d = tmp_path / "tree"
    for i in range(n_files):
        sub = d / ("d%d" % (i % 7))
        sub.mkdir(parents=True, exist_ok=True)
        n = int(rng.integers(0, 400))
        (sub / ("f%03d.txt" % i)).write_bytes(b"".join(words[j] for j in rng.integers(0, len(words), n)))
    return d


TREE_FLAGS = [["-r", "-O", "-l"], ["-r"], ["-r", "-O"], ["-r", "-l"], ["-r", "-s", "-O", "-l"]]


@pytest.mark.parametrize("flags", TREE_FLAGS, ids=lambda f: "".join(f))
def test_host_lanes_do_not_change_stdout(flags, tmp_path):
    """Many tiny batches finishing out of order over 6 lanes on 3 'GPUs': stdout must be byte-identical to the
    single-lane run (submission order), and as a multiset of lines identical to the reference."""
    _tree(tmp_path)
    pat = "foo|bar|baz|quux"
    rc1, one, se = run(flags + [pat, "tree"], cwd=str(tmp_path))
    assert rc1 == 0, se
    for bb in ("1", "2000", "100000"):
        rc, many, se = run(flags + [pat, "tree"], cwd=str(tmp_path),
                           env=dict(GRAB_B200_NDEV="3", GRAB_B200_LANES="2", GRAB_B200_BATCH_BYTES=bb, GSCAN_DOUBLE_JITTER="1"))
        assert rc == 0, se
        assert many == one
    assert sorted_lines_digest(one) == host_ref()["tree"][" ".join(flags)]


def test_host_threads_with_lanes(tmp_path):
    """-n 4 (one FileGrep per thread, each with its own lane) : same lines as the reference, any order (Q6)."""
    _tree(tmp_path, n_files=120, seed=9)
    pat = "foo|bar|baz|quux"
    rc1, one, se = run(["-r", "-O", "-l", pat, "tree"], cwd=str(tmp_path))
    if (os.cpu_count() or 1) < 4:
        pytest.skip("needs 4 cores for the reference's affinity rule")
    rc, so, se = run(["-r", "-n", "4", "-O", "-l", pat, "tree"], cwd=str(tmp_path), env=dict(GRAB_B200_NDEV="2", GSCAN_DOUBLE_JITTER="1"))
    assert rc == 0, se
    assert sorted(so.split(b"\n")) == sorted(one.split(b"\n"))


def _big_file(path, size, needles):
    a = np.full(size, ord("."), dtype=np.uint8)
    a[63::64] = 10
    for off in needles:
        a[off:off + 6] = np.frombuffer(b"NEEDLE", dtype=np.uint8)
    a.tofile(path)
    return a


F4_CHUNK = 1 << 25  # -L x5
F4_FLAGS = [["-O", "-l"], ["-s", "-O", "-l"], ["-s"], ["-l"], ["-O"]]


def _f4_file(path):
    """Three 32 MiB windows and a tail, needles at the window edges and inside the 4 KiB overlaps."""
    C = F4_CHUNK
    size = 3 * C + 12345
    return _big_file(path, size, [1000, C - 4096 + 100, C - 3, 2 * (C - 4096) + 77, size - 6, size - 400])


@pytest.mark.parametrize("flags", F4_FLAGS, ids=lambda f: "".join(f))
def test_host_one_file_over_several_gpus(flags, tmp_path):
    """f4: the windows of ONE file (chunk 32 MiB, 4 KiB overlap) go round 3 'GPUs' as separate batches; stdout is the
    reference's, including the Q3 duplicate in the overlap and -s stopping the FILE after the first printing window
    (grab.cc:232-233) even though later windows were scanned by other lanes."""
    C = F4_CHUNK
    fn = str(tmp_path / "big.bin")
    img = _f4_file(fn)
    L5 = ["-L"] * 5
    env = dict(GRAB_B200_NDEV="3", GRAB_B200_BATCH_BYTES="1", GSCAN_DOUBLE_JITTER="1")
    rc, so, se = run(L5 + flags + ["NEEDLE", fn], env=env)
    assert rc == 0, se
    want = O.Regex("NEEDLE").grab(img.tobytes(), offsets="-O" in flags, line="-l" not in flags, single="-s" in flags,
                                  chunk_size=C)
    assert so == want
    assert so == base64.b64decode(host_ref()["f4"][" ".join(flags)])
    rc, one, se = run(L5 + flags + ["NEEDLE", fn])
    assert rc == 0 and one == so


def test_host_lane_failure_is_loud(tmp_path):
    """A failing engine call on one GPU: the run reports it (stderr + exit code of a failing find, main.cc:252-256)
    and never prints output of later batches as if nothing happened on that lane."""
    _tree(tmp_path, n_files=40, seed=3)
    rc, so, se = run(["-r", "-O", "-l", "foo", "tree"], cwd=str(tmp_path),
                     env=dict(GRAB_B200_NDEV="2", GRAB_B200_BATCH_BYTES="1", GSCAN_DOUBLE_FAIL_DEVICE="1"))
    assert b"injected failure on device 1" in se
    rc, so, se = run(["-O", "-l", "foo", "tree/d0/f000.txt"], cwd=str(tmp_path), env=dict(GRAB_B200_DEVICE="9"))
    assert rc == 255 and b"no such device" in se and so == b""


@pytest.mark.parametrize("san", ["address,undefined", "thread"], ids=["asan_ubsan", "tsan"])
def test_host_pipeline_under_sanitizers(san, tmp_path):
    """The host side built with ASan+UBSan / TSan (engine double included): 6 lanes on 3 'GPUs', tiny batches, jitter,
    also under -n 4 -- no report, and the same stdout as the plain build."""
    tag = san.split(",")[0]
    exe = str(tmp_path / ("hc_" + tag))
    objs = []
    for src in (os.path.join(HERE, "hostcheck", "gscan_double.c"), os.path.join(ROOT, "oracle", "grab_oracle.c")):
        o = str(tmp_path / (os.path.basename(src) + ".o"))
        subprocess.run(["gcc", "-O1", "-g", "-fsanitize=" + san, "-c", src, "-o", o], check=True)
        objs.append(o)
    subprocess.run(["g++", "-O1", "-g", "-fsanitize=" + san, "-std=c++17", os.path.join(ROOT, "grab_b200", "host", "filegrep.cc"),
                    os.path.join(ROOT, "grab_b200", "host", "main.cc")] + objs + ["-pthread", "-o", exe], check=True)
    _tree(tmp_path, n_files=200, seed=11)
    env = dict(GRAB_B200_NDEV="3", GRAB_B200_LANES="2", GRAB_B200_BATCH_BYTES="2000", GSCAN_DOUBLE_JITTER="1",
               TSAN_OPTIONS="halt_on_error=1 exitcode=66", ASAN_OPTIONS="detect_leaks=0 exitcode=66", UBSAN_OPTIONS="halt_on_error=1 exitcode=66")
    variants = [["-r", "-O", "-l"], ["-r"], ["-r", "-s"]]
    if (os.cpu_count() or 1) >= 4:
        variants.append(["-r", "-n", "4", "-O", "-l"])
    for flags in variants:
        rc, so, se = run(flags + ["foo|bar|baz|quux", "tree"], cwd=str(tmp_path), env=env, binary=exe)
        assert rc == 0 and b"Sanitizer" not in se, (flags, se.decode()[-2000:])
        rc0, plain, _ = run(flags + ["foo|bar|baz|quux", "tree"], cwd=str(tmp_path))
        assert rc0 == 0
        if "-n" in flags:
            assert sorted(so.split(b"\n")) == sorted(plain.split(b"\n"))
        else:
            assert so == plain


def test_host_many_tiny_files_stay_below_the_mapping_limit(tmp_path):
    """80 000 files of 14 bytes: batches are cut by windows as well as by bytes, so the live mappings never reach
    vm.max_map_count (65530) -- every file is searched, nothing aborts (the reference maps one window at a time)."""
    n = 80000
    d = tmp_path / "tiny"
    d.mkdir()
    for k in range(0, n, 1000):
        sub = d / ("s%03d" % (k // 1000))
        sub.mkdir()
        for i in range(k, k + 1000):
            (sub / ("f%05d" % i)).write_bytes(b"xx foo %05d\n\n" % i if i % 7 == 0 else b"nothing here.\n")
    rc, so, se = run(["-r", "-O", "-l", "foo", "tiny"], cwd=str(tmp_path))
    assert rc == 0 and se == b"", se[-500:]
    lines = so.split(b"\n")
    assert len([x for x in lines if x]) == len(range(0, n, 7))
    assert all(x.endswith(b":Match at offset 3") for x in lines if x)


def test_host_good_path_then_missing_path(tmp_path):
    """`grab foo a nope`: the matches of `a` are printed before the stat error of `nope` ends the run (rc 255)."""
    (tmp_path / "a").write_bytes(b"xx foo yy\nzz foo\n\n")
    rc, so, se = run(["-O", "-l", "foo", "a", "nope"], cwd=str(tmp_path))
    assert rc == 255
    assert so == b"a:Match at offset 3\na:Match at offset 13\n"
    assert b"FileGrep::find::stat" in se
    ref = host_ref()["good_then_missing"]
    assert (ref["rc"], base64.b64decode(ref["stdout"])) == (rc, so) and base64.b64decode(ref["stderr"]) == se


@pytest.mark.parametrize("flags", [["-r", "-O", "-l"], ["-r", "-l"], ["-r", "-s", "-O", "-l"]], ids=lambda f: "".join(f))
def test_host_descriptor_feed_equals_mapped_feed(flags, tmp_path):
    """Without line output the windows travel as descriptors (GSCAN_UNIT_FD: read by the engine's staging threads, never
    mapped); GRAB_B200_FEED=mmap keeps the reference's mappings.  Same bytes on stdout either way, also with a descriptor
    limit so tight that batches are cut by descriptors (ulimit -n 400: about 90 windows per batch) and with one so tight
    that the feed falls back to mappings (ulimit -n 200)."""
    _tree(tmp_path)
    pat = "foo|bar|baz|quux"
    rc, mapped, se = run(flags + [pat, "tree"], cwd=str(tmp_path), env=dict(GRAB_B200_FEED="mmap"))
    assert rc == 0, se
    rc, by_fd, se = run(flags + [pat, "tree"], cwd=str(tmp_path), env=dict(GRAB_B200_TRACE="1"))
    assert rc == 0 and by_fd == mapped, se
    assert b"as descriptors)" in se and b"(0 as descriptors)" not in se
    assert b"(0 as descriptors)" in run(flags + [pat, "tree"], cwd=str(tmp_path), env=dict(GRAB_B200_TRACE="1", GRAB_B200_FEED="mmap"))[2]
    assert b"(0 as descriptors)" in run(["-r", "-O", pat, "tree"], cwd=str(tmp_path), env=dict(GRAB_B200_TRACE="1"))[2]  # line output: mapped
    for limit in ("400", "200"):
        sh = "ulimit -Hn %s; exec %s %s '%s' tree" % (limit, BIN, " ".join(flags), pat)
        e = {k: v for k, v in os.environ.items() if not k.startswith("GRAB_B200_")}
        p = subprocess.run(["bash", "-c", sh], stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=str(tmp_path), env=e, timeout=300)
        assert p.returncode == 0 and p.stdout == mapped, (limit, p.stderr[-500:])


def test_host_descriptor_feed_one_file_many_windows(tmp_path):
    """One file cut into windows (chunk 32 MiB): every window of a descriptor feed holds its own descriptor (dup), the
    last one the file's; stdout equals the mapped feed's and the oracle's FileGrep::find restatement (Q3 duplicates)."""
    C = 1 << 25
    size = 2 * C + 999
    fn = str(tmp_path / "big.bin")
    img = _big_file(fn, size, [1000, C - 4096 + 100, C - 3, size - 6])
    args = ["-L"] * 5 + ["-O", "-l", "NEEDLE", fn]
    rc, so, se = run(args)
    assert rc == 0, se
    assert so == O.Regex("NEEDLE").grab(img.tobytes(), offsets=True, line=False, single=False, chunk_size=C)
    rc, mapped, se = run(args, env=dict(GRAB_B200_FEED="mmap"))
    assert rc == 0 and mapped == so
