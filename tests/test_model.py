"""What the pattern compiler hands to the device, interpreted on the CPU and compared with the oracle (no GPU):
tests/model_check.cc runs the compiled Program the way the resolve kernels do -- with the device VM's own source,
extracted verbatim from grab_b200/csrc/resolve_kernels.cu and compiled for the host -- inside the reference's loop."""
import os
import subprocess

import test_gpu_random_patterns as R
import test_gpu_parity as P
from test_scan_variants import VARIANTS

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BEGIN = "// ---- device backtracking VM (general patterns) ----"
END = "// ---- 4. generic u32 block sums / exclusive scan (per-unit match counts -> output slots) ----"


def test_compiled_programs_match_the_oracle(tmp_path):
    src = open(os.path.join(ROOT, "grab_b200", "csrc", "resolve_kernels.cu")).read()
    assert BEGIN in src and END in src
    snippet = src[src.index(BEGIN):src.index(END)]
    assert "vm_exec" in snippet and "k_walk_vm" in snippet and "<<<" not in snippet
    (tmp_path / "vm_snippet.inc").write_text(snippet)
    pats = list(R.PATTERNS) + R.make_cases(400, 777) + list(P.DIFF_PATTERNS) + [
        "foo|bar|baz|quux", "[A-Za-z0-9_]{16,}", "[0-9]{2,}", "(?i)ab|ba", "a.c", "ab?c", "a{2,4}", "\\d{2}-\\d{2}", "<[a-z]+>", "qz\\w+;",
        "(?U)a+b", "(?U)a+?b", "(?U)a{2,}", "(?U)\\w+ ", "(?U:a+)b", "(?U)a*b", "(?U)(?:ab)+c", "a(?U)b+c?", "(?x) a b c", "(?x)a +b",
        "(?xi)A B", "(?x)a b | b c", "a(?x) b c", "(?x)a{2} b", "(?x) [ab] {2} c", "a(?#hello)b", "(?#c)a|b(?#d)c", "a(?#x)+b",
        "foo|(bar)", "(x)?foo", "(?:(a)|b)+c", "(a)?ab", "(a)*b", "(a|b)", "x(?:(z)|)y", "a(b)?c", "(ab|a)c|b", "(?:a(b))?c", "((a)|b)x|c", "a(?:b|(c))+",
        "(?<=a)b", "a(?=b)", "a(?!b)", "(?<!a)b", "(?>a+)b", "(?>a+)ab", "a++b", "(?:ab)++c", "(?:ab)*+ab", "(?<=a|bc)x", "(?<!a|bc)x",
        "\\b(?=\\w{3}\\b)\\w+", "(?=.*c)a\\w+", "x(?!.*b)\\w*", "(?<=^|c)[ab]+", "(?i)(?<=AB)c", "a(?=(b))", "(?!(a))b", "(?<=ab)c|c", "(?>a|ab)c",
        "[^a]{2,}", "[^b]{3,}", "\\s{2,}", "[\\n ab]{2,}", "\\W{2,}", "[ab]{2,}", "[ab]{5,}", "a{3,}", "[^\\n]{4,}", "\\w{3,}", "[a-c ]{6,}",
        "a+b+", "(?:a|b)+c", "^a.*c$", "\\bab\\b", "a.*?c", "[ab]+?c", "x*ab", "(?:ab)*c", "ab|abc|a", "a(?:b|bc)c"]
    import json
    kat = json.load(open(os.path.join(HERE, "golden", "kat.json")))
    pats += sorted({c["pattern"] for c in kat["cases"]})  # the reference's recorded cases
    pats += [p for key in sorted(VARIANTS, key=str) for p in VARIANTS[key]]  # every scan-kernel instantiation, high bytes and NUL
    (tmp_path / "patterns.txt").write_text("\n".join(p for p in pats if "\n" not in p) + "\n")
    exe = str(tmp_path / "model_check")
    subprocess.run(["gcc", "-O2", "-c", os.path.join(ROOT, "oracle", "grab_oracle.c"), "-o", str(tmp_path / "oracle.o")], check=True)
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")  # kernels.h names cudaError_t / cudaStream_t
    subprocess.run(["g++", "-O2", "-std=c++17", "-w", "-I", str(tmp_path), "-I", cuda_inc, os.path.join(HERE, "model_check.cc"),
                    os.path.join(ROOT, "grab_b200", "csrc", "pattern.cc"), str(tmp_path / "oracle.o"), "-I", os.path.join(ROOT, "include"),
                    "-o", exe], check=True)
    p = subprocess.run([exe, str(tmp_path / "patterns.txt")], stdout=subprocess.PIPE, timeout=900)
    out = p.stdout.decode()
    assert p.returncode == 0 and "model ok" in out, out[-3000:]
    # the sample must actually exercise the engines
    tail = out.strip().splitlines()[-2]
    assert int(tail.split("strict (Q2) patterns ")[1].split(";")[0]) >= 12, tail
    assert int(tail.split("flat write checks ")[1].split(";")[0]) >= 1000, tail
    assert int(tail.split("; chain checks ")[1].split(";")[0]) >= 1000, tail
    assert int(tail.split("; vm chain checks ")[1].split(";")[0]) >= 1000, tail
    assert int(tail.split("; dense vm chain checks ")[1].split(";")[0]) >= 1000, tail
    assert int(tail.split("two-unit chain checks ")[1].split(";")[0]) >= 1000, tail
    served = int(tail.split("served ")[1].split(" ")[0])
    vm = int(tail.split("served ")[1].split("(")[1].split(" ")[0])
    assert served > 300 and vm > 100, tail
