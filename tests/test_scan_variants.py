"""Which scan-kernel instantiation serves a pattern, checked on the CPU.

scan_kernels.cu dispatches every FIXED and RUN pattern to one of ~150 template instantiations (launch_scan_fixed,
launch_fixed3, launch_fixedb_k, launch_run_hf, launch_scan_hash).  VARIANTS names, per instantiation, the patterns that
reach it -- wherever the family allows, one with bytes >= 0x80 or NUL -- and is the one list of variant patterns the
binary differential (test_gpu_binary.py) and the reference pin (test_oracle_vs_ref.py) run.  A compiler change that moves
one of these patterns elsewhere fails here, instead of silently thinning what the GPU tests cover.  Every case of the
dispatch switches is either in VARIANTS or in UNREACHABLE with the reason no pattern can get there."""
import itertools
import os
import re

import pytest

import grab_b200 as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# 600 distinct three-letter lowercase keys: more than 512 table slots, so one copy of the table; one narrow byte range, so
# the sparse path is possible
HASH_WIDE = "|".join("".join(chr(0x61 + (k // 26 ** j) % 26) for j in range(3)) for k in ((i * 7919) % 26 ** 3 for i in range(600)))

# key: ("FixedEngine", D, K, EX), ("Fixed3Engine", K, EX), ("FixedBEngine", D, K, ALIGNED), ("RunEngine", NLO, NHI, NFO),
# ("HashEngine", sparse path possible, table copies) -- the template arguments, not the raw values of scan_variant
VARIANTS = {
    # ---- pair filter FixedEngine<D, K, EX>: D = filter_delta, K = tests (5 -> 6, 7 -> 8), EX = every test exact ----
    ("FixedEngine", 0, 1, False): ["\\xff", "\\x00", "a"],
    ("FixedEngine", 0, 2, False): ["\\xff|bb"],
    ("FixedEngine", 0, 3, False): ["b\\x00|a|.\\x80"],
    ("FixedEngine", 0, 4, False): ["aa|b|\\xff\\x00|\\x00."],
    ("FixedEngine", 0, 6, False): ["\\xe0|\\xe1\\xe2|\\xe3\\xe4|\\xe5\\xe6|\\xe7\\xe8", "a|bc|de|fg|hi|jk"],
    ("FixedEngine", 0, 8, False): ["a|bc|de|fg|hi|jk|lm", "\\x80|\\x81\\x82|\\x83\\x84|\\x85\\x86|\\x87\\x88|\\x89\\x8a|\\x8b\\x8c|\\x00\\x01"],
    ("FixedEngine", 1, 1, False): ["\\xf7.", "(?i)ab"],
    ("FixedEngine", 1, 1, True): ["\\xff\\xfe", "\\x00\\x01", "[a-z]{100}QZ"],
    ("FixedEngine", 1, 2, False): ["\\xff.|aa"],
    ("FixedEngine", 1, 2, True): ["aa|b\\x80b"],
    ("FixedEngine", 1, 3, False): ["ab|b.|\\x00a", "ab|ba|ca|cb|bc"],
    ("FixedEngine", 1, 3, True): ["z\\x8d|\\x87z|y\\x8c"],
    ("FixedEngine", 1, 4, False): ["b\\x80|ab|.a|aa|\\x80\\xff"],
    ("FixedEngine", 1, 4, True): ["b\\xff|\\xffba\\x80|a\\xff|\\x00a"],
    ("FixedEngine", 1, 6, False): ["[\\x00-\\xff]{3}bo|b.|ud|k.|wb|gy"],
    ("FixedEngine", 1, 6, True): ["[\\x00-\\xff]{2}ab|[\\x00-\\xff]{2}cd|[\\x00-\\xff]{2}ef|[\\x00-\\xff]{2}gh|[\\x00-\\xff]{2}ij"],
    ("FixedEngine", 1, 8, False): ["[\\x00-\\xff]{3}hs|bq|ld|xu|qgk|lx|xhrt|dr"],
    ("FixedEngine", 1, 8, True): ["[\\x00-\\xff]{3}iy|[\\x00-\\xff]{3}woc|[\\x00-\\xff]{3}nfk|[\\x00-\\xff]{3}lli|[\\x00-\\xff]{3}zwfc|"
                                  "[\\x00-\\xff]{3}qdqlo|[\\x00-\\xff]{3}jlw"],
    ("FixedEngine", 2, 1, False): ["(?i)\\x8b.x"],
    ("FixedEngine", 2, 1, True): ["(?i)\\xe9t\\xe9", "x.\\x80"],
    ("FixedEngine", 2, 2, False): ["(?i)\\x8f.x|\\x8b\\x84\\x83"],
    ("FixedEngine", 2, 3, False): ["[\\xf7\\xfb].\\xee|\\xe5\\xe0\\xed|\\xe3\\xf5\\xf2"],
    ("FixedEngine", 2, 4, False): ["\\x87\\x88\\x83.|y\\x83\\x86z|\\x8a.\\x8b\\x85|\\x82\\x87[\\x8b\\x8a]\\x87"],
    ("FixedEngine", 2, 6, False): ["\\x8d\\x84z\\x8ay\\x80|\\x81[\\x8e\\x83][\\x89\\x8c]\\x80|.[\\x8f\\x88].\\x84|x\\x80\\x89z|.\\x81\\x88\\x86"],
    ("FixedEngine", 2, 8, False): ["\\xff\\x80.\\x00|.\\xff\\xff.|\\x80b\\xffa|[\\x80\\x80].\\xffb|\\x80\\x00bb|\\x80ba\\xff|\\xff\\x80\\x00b|ba\\xffb|"
                                   "a\\x00\\x00\\xff"],
    ("FixedEngine", 2, 8, True): ["[\\x00-\\xff]{3}\\xff\\x80b|[\\x00-\\xff]{3}\\x00.\\xff\\x80a|[\\x00-\\xff]{3}\\x80\\x80\\x80|"
                                  "[\\x00-\\xff]{3}\\xff\\x00a\\x80|[\\x00-\\xff]{3}a[\\xff\\x00]b|[\\x00-\\xff]{3}[bb]\\x00\\x80|"
                                  "[\\x00-\\xff]{3}\\x00\\x00\\xff|[\\x00-\\xff]{3}b\\x80\\x00|[\\x00-\\xff]{3}\\x00\\xff\\x80.\\x00[\\x00b]"],
    ("FixedEngine", 3, 1, False): ["(?i)baa\\x80"],
    ("FixedEngine", 3, 1, True): ["ba.\\x80"],
    ("FixedEngine", 3, 2, False): ["\\x8f.\\x89\\x8a|[\\x82\\x88]\\x85.\\x81"],
    ("FixedEngine", 3, 3, False): ["\\xe0.\\xec\\xfe|\\xf9\\xea.\\xe6|\\xe8\\xe2\\xe1[\\xff\\xfd]"],
    ("FixedEngine", 3, 4, False): ["\\x07\\x0b\\x03\\x04|\\x0d.\\x04[\\x0f\\x00]|\\x0c\\x07\\x02\\x08|\\x08\\x0b.\\x0e"],
    ("FixedEngine", 3, 6, False): ["\\x8fz.\\x8b|\\x80\\x86\\x8az|\\x8e.\\x8c\\x84|\\x82\\x8dx\\x87|\\x87\\x8c\\x8c[\\x81\\x84]\\x80\\x8c"],
    ("FixedEngine", 3, 8, False): ["[\\x00-\\xff]{2}\\xff\\x80|abb\\xffb|.\\x80\\x80\\x00b|\\x80[bb][\\xffa]a[ab]|aa\\xff\\x00a|b[\\x00\\x80]\\x80b.|"
                                   "b\\x80\\x00b\\xff|\\x00\\xffaa|\\xff\\x00b\\x00b"],
    ("FixedEngine", 3, 8, True): ["\\x80a\\x80a\\xff\\x00|\\x00\\xffa\\x80\\xffa|a.ba\\x80\\x80|\\x80bb\\x00\\x00a|b\\x80[\\x00\\xff]\\xff|\\xff\\x00b\\xffa|"
                                  "\\x80[\\xffb]b\\x80\\xff\\x80|[\\x00\\x00]\\xff.aa\\x00|ba[\\x80\\xff][\\xff\\xff]\\x80a"],
    ("FixedEngine", 4, 1, False): ["(?i)\\x00bbab."],
    ("FixedEngine", 4, 1, True): ["b.ab\\x00", "foobardoesexist"],
    ("FixedEngine", 4, 2, False): ["\\x00\\x00[a\\x00][\\x80a][\\x00b]|baabb"],
    ("FixedEngine", 4, 2, True): ["\\x00ba\\xff\\xffa|a.[\\xffb].\\xff\\x00|abb\\xff\\xff"],
    ("FixedEngine", 4, 3, False): ["[\\x00-\\xff]{2}..h[nt]n|bv[tn].v|[id]wvap"],
    ("FixedEngine", 4, 3, True): ["\\x80\\xff.ab.|\\x80[\\x00\\xff]a\\xffba|\\xff\\xff.b\\xff|a[\\x80\\x80]a\\xff\\x00\\xff"],
    ("FixedEngine", 4, 4, True): ["a..\\xff\\x00|a.b.\\x80|a\\xff.bb|b\\x00\\xff\\xff\\xff|a.a\\x00\\x80|a\\x00a\\xff\\x00"],
    ("FixedEngine", 4, 4, False): ["ab\\x00[\\x00\\x00]\\x80|ba[\\x80\\xff]\\xff\\xff|...b\\x80|\\x00\\xff\\x00ab"],
    ("FixedEngine", 4, 6, True): ["[\\x00-\\xff]{3}hbbhf|[\\x00-\\xff]{3}ad..b|[\\x00-\\xff]{3}cceeb|[\\x00-\\xff]{3}ceehb|[\\x00-\\xff]{3}gaafc|[\\x00-\\xff]{3}jd.jj"],
    ("FixedEngine", 4, 6, False): ["[\\x00-\\xff]{3}[nb]w|njfdb|ovmqc|lvf.k|z.hi."],
    ("FixedEngine", 4, 8, False): ["\\x80[\\x80a]\\xffa\\xff|\\x00\\x00\\x80.\\xff|\\x00\\xff\\x00[b\\xff][\\x00b]|\\xffb.a[ba]|b\\x80b.\\x80|\\x00.\\xffaa|"
                                   "\\xffa[\\x00a]aa|\\xff\\x00\\x00\\x00\\x80"],
    # ---- triple filter Fixed3Engine<K, EX>: K = third-byte tests (5 -> 6, 7.. -> 8) ----
    ("Fixed3Engine", 1, False): ["\\xfa..", "(?i)linus", "a.b"],
    ("Fixed3Engine", 1, True): ["a\\xffa"],
    ("Fixed3Engine", 2, False): ["..b|\\xffa."],
    ("Fixed3Engine", 2, True): ["a\\x80\\xffa|.\\x80\\x00a"],
    ("Fixed3Engine", 3, False): ["abb|a.\\x80\\x00a|b.."],
    ("Fixed3Engine", 3, True): ["[bb]\\x00\\x00\\x80|a\\x00\\xff\\xff|a.\\xffa"],
    ("Fixed3Engine", 4, False): ["a.b.|ab\\x80a|\\x80b.\\x00|..\\x00b"],
    ("Fixed3Engine", 4, True): ["\\x80\\x00aa|.\\x00\\x80b\\x00|\\xffab\\xff|\\xff\\x00\\xffa"],
    ("Fixed3Engine", 6, False): ["[\\x00-\\xff]{2}j|wjt.|wxlp|btk|zvah"],
    ("Fixed3Engine", 6, True): ["\\x00\\x00\\xff|b\\x00\\x80\\xff|\\x00\\x00\\x80|\\xffb\\x00a|\\x80\\x00a\\x80"],
    ("Fixed3Engine", 8, False): ["[\\x00-\\xff]{2}.kd|.gy|xs.|tfs|[cx]wm|hk.|hp[ws]"],
    # ---- balanced pair filter FixedBEngine<D, K, AL>: D 1..4, K = tests (5 -> 6, 7 -> 8), AL = aligned stage 2 ----
    ("FixedBEngine", 1, 2, False): ["z\\x83|\\x8fz"],
    ("FixedBEngine", 1, 2, True): ["b\\xff.|\\x00ba", "\\xff\\xfe\\xfd|\\xe0\\xe1\\xe2"],
    ("FixedBEngine", 1, 3, False): ["\\x00\\x01|\\x02\\x03|\\x04\\x05", "\\x80y|\\x81\\x86|\\x83\\x80"],
    ("FixedBEngine", 1, 3, True): ["foo|bar|baz|quux", "\\x80y\\x84|\\x8a\\x87.|y\\x8bx"],
    ("FixedBEngine", 1, 4, False): ["\\xe2\\xeb|\\xfd\\xf7|\\xe7\\xe8|\\xed\\xf1"],
    ("FixedBEngine", 1, 4, True): ["aaa|b\\x80b|bba|a\\x00\\x00"],
    ("FixedBEngine", 1, 6, False): ["(?i)\\xe3\\xf9\\xfd\\xf6\\xff|\\xf0\\xf9.\\xe7\\xe6|.\\xf1\\xfd\\xf7\\xf0|\\xe1\\xef\\xf1\\xf7\\xe2|.\\xf9\\xef\\xea\\xf3"],
    ("FixedBEngine", 1, 6, True): ["\\x80\\x00\\xffbbb|b.\\x80\\x80a|.\\x80a\\x00..|a.ab\\xff.|b.\\xff\\x80ba",
                                   "[\\x00-\\xff]{2}abc|[\\x00-\\xff]{2}cde|[\\x00-\\xff]{2}efg|[\\x00-\\xff]{2}ghi|[\\x00-\\xff]{2}ijk"],
    ("FixedBEngine", 1, 8, False): ["[\\x00-\\xff]{2}\\x0c\\x0d\\x07\\x0e\\x0a|[\\x00-\\xff]{2}\\x06\\x00|[\\x00-\\xff]{2}\\x0f\\x0d|[\\x00-\\xff]{2}\\x05\\x0e|"
                                    "[\\x00-\\xff]{2}\\x08\\x03\\x06.|[\\x00-\\xff]{2}\\x02\\x0f|[\\x00-\\xff]{2}\\x00\\x06"],
    ("FixedBEngine", 1, 8, True): ["[\\x00-\\xff]{2}roowju|[\\x00-\\xff]{2}sbs[dy]|[\\x00-\\xff]{2}qxey|[\\x00-\\xff]{2}mw.|[\\x00-\\xff]{2}gpy|"
                                   "[\\x00-\\xff]{2}tag|[\\x00-\\xff]{2}dgy"],
    ("FixedBEngine", 2, 2, False): [".\\xff[\\x80\\x80]\\x00|b\\xffa\\x00|\\x80\\xffa\\xff"],
    ("FixedBEngine", 2, 2, True): ["bbb.a|a.\\x00", "foo|bar"],
    ("FixedBEngine", 2, 3, False): ["\\x0b\\x0d\\x09\\x02|\\x00\\x0d\\x08|\\x05.\\x02|\\x0b\\x0a\\x09"],
    ("FixedBEngine", 2, 3, True): ["b.\\x80|\\x80.b|\\xff.\\xff"],
    ("FixedBEngine", 2, 4, False): ["\\x82\\x87\\x86x|\\x82y\\x85\\x84z\\x85|\\x8f\\x80\\x81[x\\x85]\\x82\\x86|\\x85yz\\x80\\x8b\\x87|\\x82\\x88\\x86\\x8f\\x8e\\x87"],
    ("FixedBEngine", 2, 4, True): ["\\x80[\\x80b]b|baa|\\x00.\\xff|a\\x00\\x00"],
    ("FixedBEngine", 2, 6, False): ["[\\x00-\\xff]{3}\\xe2\\xf5\\xef\\xf8|[\\x00-\\xff]{3}\\xf7\\xe1\\xe3\\xe2|[\\x00-\\xff]{3}\\xfa.\\xe6\\xeb|"
                                    "[\\x00-\\xff]{3}\\xfb\\xe1\\xea[\\xec\\xfa]|[\\x00-\\xff]{3}\\xf7\\xf0\\xe3.|[\\x00-\\xff]{3}\\xf1.\\xfa\\xe7\\xea\\xea"],
    ("FixedBEngine", 2, 6, True): ["[\\x00-\\xff]{2}ab\\x00\\x00\\xff|.\\x00\\xffa\\x00|b\\x00a\\xff\\xff|ab\\x00a\\xff|.\\xffa.b|\\xffa\\x00aa"],
    ("FixedBEngine", 2, 8, False): ["[\\x00-\\xff]{3}\\x01.\\x0d|[\\x00-\\xff]{3}\\x0e\\x0b\\x00[\\x06\\x03]\\x02\\x05|[\\x00-\\xff]{3}\\x0e\\x00\\x00\\x08.\\x00|"
                                    "[\\x00-\\xff]{3}\\x0a\\x0d\\x01\\x02\\x08\\x05|[\\x00-\\xff]{3}\\x0e\\x00\\x01\\x0f\\x09\\x00|[\\x00-\\xff]{3}\\x06\\x07\\x06\\x02\\x07\\x0b|"
                                    "[\\x00-\\xff]{3}\\x02\\x03\\x03\\x08\\x0a\\x03|[\\x00-\\xff]{3}\\x08\\x08\\x09\\x0e\\x0c[\\x03\\x02]"],
    ("FixedBEngine", 2, 8, True): ["[\\x00-\\xff]{3}klhcwg|[\\x00-\\xff]{3}sovy|[\\x00-\\xff]{3}nyi.|[\\x00-\\xff]{3}fpuk|[\\x00-\\xff]{3}l.iw|"
                                   "[\\x00-\\xff]{3}s.b.|[\\x00-\\xff]{3}pmp[sw]|[\\x00-\\xff]{3}wnhr"],
    ("FixedBEngine", 3, 2, False): ["[\\x00-\\xff]{3}\\x0b\\x0e\\x0a\\x07\\x00\\x0f|[\\x00-\\xff]{3}\\x07\\x0e\\x02\\x09\\x00|[\\x00-\\xff]{3}\\x0a\\x05\\x08\\x06\\x0d"],
    ("FixedBEngine", 3, 2, True): ["babb|\\x80aa\\x00a"],
    ("FixedBEngine", 3, 3, False): ["\\x80\\xffb\\x00.\\xff|\\x80\\x80[\\x80a]\\x80\\x00\\xff|\\x00bb\\xff[a\\x80]a|\\x80b\\x00\\x00[\\x80a]b"],
    ("FixedBEngine", 3, 4, False): ["[\\x00-\\xff]{3}\\xff.\\xe1\\xe9\\xf0\\xfd\\xf8|[\\x00-\\xff]{3}..\\xe4\\xf2\\xf4\\xed\\xed|[\\x00-\\xff]{3}\\xe7\\xee\\xe1\\xf4\\xe7\\xeb\\xe2|"
                                    "[\\x00-\\xff]{3}\\xe9.\\xe1\\xea\\xfb\\xfd\\xed|[\\x00-\\xff]{3}\\xfe\\xe9\\xf3.\\xe3\\xed\\xe1"],
    ("FixedBEngine", 3, 3, True): ["\\x80\\xffaa|b\\x00ab|b.\\x00\\xff"],
    ("FixedBEngine", 3, 6, False): [".\\x06\\x0b\\x05\\x09\\x0b|\\x0c\\x09\\x0d\\x07.\\x06|\\x0e\\x01\\x00\\x0f\\x04\\x03|\\x06.\\x00\\x0d\\x0d\\x03|..\\x00\\x0a\\x0a\\x0f|\\x0f\\x01\\x0d\\x04\\x06\\x03"],
    ("FixedBEngine", 3, 4, True): ["\\xffba\\xffaa|a.aa|\\x80a\\x00\\xff|aa.\\x80"],
    ("FixedBEngine", 3, 6, True): ["\\x07\\x04\\x08\\x08|\\x0b\\x0f\\x04\\x09|\\x0d\\x0d\\x0a\\x03|\\x0c\\x0f\\x02\\x06\\x00\\x02|\\x0c..\\x07"],
    ("FixedBEngine", 3, 8, False): ["[\\x00-\\xff]{2}\\x80\\xc0\\xc1\\x81|[\\x00-\\xff]{2}\\x80\\xc2\\xc3\\x81|[\\x00-\\xff]{2}\\x82\\xc4\\xc5\\x83|[\\x00-\\xff]{2}\\x82\\xc6\\xc7\\x83|[\\x00-\\xff]{2}\\x84\\xc8\\xc9\\x85|[\\x00-\\xff]{2}\\x84\\xca\\xcb\\x85|[\\x00-\\xff]{2}\\x86\\xcc\\xcd\\x87|[\\x00-\\xff]{2}\\x86\\xce\\xcf\\x87|[\\x00-\\xff]{2}\\x88\\xd0\\xd1\\x89|[\\x00-\\xff]{2}\\x88\\xd2\\xd3\\x89|[\\x00-\\xff]{2}\\x8a\\xd4\\xd5\\x8b|[\\x00-\\xff]{2}\\x8a\\xd6\\xd7\\x8b|[\\x00-\\xff]{2}\\x8c\\xd8\\xd9\\x8d|[\\x00-\\xff]{2}\\x8c\\xda\\xdb\\x8d|[\\x00-\\xff]{2}\\x8e\\xdc\\xdd\\x8f|[\\x00-\\xff]{2}\\x8e\\xde\\xdf\\x8f",
                                    "[\\x00-\\xff]{2}\\x80\\xc0\\xe0\\x81|[\\x00-\\xff]{2}\\x80\\xc1\\xe1\\x81|[\\x00-\\xff]{2}\\x80\\xc2\\xe2\\x81|[\\x00-\\xff]{2}\\x82\\xc3\\xe0\\x83|[\\x00-\\xff]{2}\\x82\\xc4\\xe1\\x83|[\\x00-\\xff]{2}\\x82\\xc5\\xe2\\x83|[\\x00-\\xff]{2}\\x84\\xc6\\xe0\\x85|[\\x00-\\xff]{2}\\x84\\xc7\\xe1\\x85|[\\x00-\\xff]{2}\\x84\\xc8\\xe2\\x85|[\\x00-\\xff]{2}\\x86\\xc9\\xe0\\x87|[\\x00-\\xff]{2}\\x86\\xca\\xe1\\x87|[\\x00-\\xff]{2}\\x86\\xcb\\xe2\\x87|[\\x00-\\xff]{2}\\x88\\xcc\\xe0\\x89|[\\x00-\\xff]{2}\\x88\\xcd\\xe1\\x89|[\\x00-\\xff]{2}\\x88\\xce\\xe2\\x89|[\\x00-\\xff]{2}\\x8a\\xcf\\xe0\\x8b|[\\x00-\\xff]{2}\\x8a\\xd0\\xe1\\x8b|[\\x00-\\xff]{2}\\x8a\\xd1\\xe2\\x8b|[\\x00-\\xff]{2}\\x8c\\xd2\\xe0\\x8d|[\\x00-\\xff]{2}\\x8c\\xd3\\xe1\\x8d|[\\x00-\\xff]{2}\\x8c\\xd4\\xe2\\x8d"],
    ("FixedBEngine", 3, 8, True): ["\\x82\\x88\\x81\\x85.|\\x8a[\\x8e\\x82]\\x8c\\x84\\x80|\\x8d\\x81[\\x88\\x8b]\\x83\\x8f|\\x81\\x8d.\\x85\\x82|\\x8a.y\\x82|"
                                   "\\x82\\x83\\x87xx|y.\\x84\\x8e\\x87\\x88"],
    ("FixedBEngine", 4, 2, False): ["\\x80\\x00ab\\x00|\\x00...\\x00|\\x80.\\x80\\x00\\x00"],
    ("FixedBEngine", 4, 2, True): ["b\\x80.bbb|\\x80b.b.\\x00"],
    ("FixedBEngine", 4, 3, False): ["\\x80[b\\x80]\\x80.b|\\x80[ab]a\\x00\\x00|\\x00aa\\xff\\x80|\\x80aa[\\x00a]b"],
    ("FixedBEngine", 4, 3, True): ["b\\xffb\\x00\\x80|\\x00\\xff\\x00a\\xff|\\x80b\\x00ba"],
    ("FixedBEngine", 4, 4, False): ["[\\x00-\\xff]{2}\\xfe\\xf4\\xee.\\xfe\\xee\\xff|[\\x00-\\xff]{2}\\xe7\\xf4\\xfa\\xfa\\xff\\xf8\\xe5|[\\x00-\\xff]{2}\\xe7\\xe9\\xf0\\xe7\\xff\\xfe.|"
                                    "[\\x00-\\xff]{2}\\xf0\\xf4\\xed.\\xe6\\xec\\xf8|[\\x00-\\xff]{2}\\xe7.\\xe1\\xe5\\xf1.\\xe9"],
    ("FixedBEngine", 4, 4, True): ["\\x00aaa\\x00|ab\\x80\\x80b\\x80|b[ba]a[\\xffb]a|b\\xff.a\\x80"],
    ("FixedBEngine", 4, 6, False): ["[\\x00-\\xff]{3}\\x0b.\\x0d\\x04\\x0b\\x02|[\\x00-\\xff]{3}\\x03\\x0c\\x07\\x0f\\x06\\x00|[\\x00-\\xff]{3}\\x00\\x00\\x07\\x0b\\x07\\x0b|"
                                    "[\\x00-\\xff]{3}\\x05\\x06[\\x00\\x0e]\\x0c\\x00\\x06|[\\x00-\\xff]{3}\\x04\\x0f.\\x00\\x08\\x06|[\\x00-\\xff]{3}\\x01\\x06[\\x01\\x03]\\x0b\\x06\\x00|"
                                    "[\\x00-\\xff]{3}\\x05\\x01.\\x08\\x00\\x0d"],
    ("FixedBEngine", 4, 6, True): ["\\x00.[bb]aa\\xff|\\x00\\x80.\\x00\\x00b|\\x00\\xff\\x00\\x00b\\xff|ba[b\\xff]\\xffb.|\\x80\\x00..aa"],
    ("FixedBEngine", 4, 8, False): ["[\\x00-\\xff]{2}\\x0f\\x03\\x03\\x03\\x0c\\x03|[\\x00-\\xff]{2}\\x0a\\x0b\\x00\\x07\\x0c\\x09|[\\x00-\\xff]{2}\\x06\\x0c\\x0a..\\x03|"
                                    "[\\x00-\\xff]{2}.\\x05.\\x08\\x08\\x00|[\\x00-\\xff]{2}\\x0d\\x0b\\x07..\\x04|[\\x00-\\xff]{2}\\x0a\\x0d\\x07\\x09\\x0c\\x0c|"
                                    "[\\x00-\\xff]{2}.\\x0b\\x0d\\x03.\\x09|[\\x00-\\xff]{2}\\x09\\x0d..\\x04\\x03"],
    ("FixedBEngine", 4, 8, True): ["\\x80b[\\x00\\x80]a\\x00|\\x00ab\\x00\\xff\\xff|b\\x80a[ba]a|\\xff\\x80a[\\x80b]b\\x00|bb\\xffa\\xffb|a.a[a\\x80]\\x00\\x80|"
                                   "\\x00a.[\\xffa]\\x80\\xff"],
    # exact pair / triple filters that the balanced filter does not take: 9-16 third-byte tests (no triple stage 1, stage 2 not
    # aligned with the pair tests) and a pair prior above 0.01 / 512 (common bytes)
    ("FixedEngine", 2, 2, True): ["eaeb|ebec|eced|edee|eeef|tatb|tbtc|tctd|tdte",
                                  "e\\x80e\\xff|e\\x81e\\x80|e\\x82e\\x81|e\\x83e\\x82|e\\x84e\\x83|t\\x80t\\x84|t\\x81t\\x85|t\\x82t\\x86|t\\x83t\\x87"],
    ("FixedEngine", 2, 3, True): ["e\\x80e\\xff|e\\x81e\\x80|e\\x82e\\x81|e\\x83e\\x82|e\\x84e\\x83|t\\x80t\\x84|t\\x81t\\x85|t\\x82t\\x86|t\\x83t\\x87|aaaa|"
                                  "a\\xffa\\x00"],
    ("FixedEngine", 2, 4, True): ["eaeb|ebec|eced|edee|eeef|tatb|tbtc|tctd|tdte|aaaa|abba",
                                  "e\\x80e\\xff|e\\x81e\\x80|e\\x82e\\x81|e\\x83e\\x82|e\\x84e\\x83|t\\x80t\\x84|t\\x81t\\x85|t\\x82t\\x86|t\\x83t\\x87|aaaa|"
                                  "a\\xffa\\x00|h\\x00h\\x01"],
    ("FixedEngine", 3, 2, True): ["eaaeb|ebbec|ecced|eddee|eeeef|taatb|tbbtc|tcctd|tddte"],
    ("FixedEngine", 3, 3, True): ["eaaeb|ebbec|ecced|eddee|eeeef|taatb|tbbtc|tcctd|tddte|aeeaa|affab"],
    ("FixedEngine", 3, 4, True): ["eaaeb|ebbec|ecced|eddee|eeeef|taatb|tbbtc|tcctd|tddte|aeeaa|affab|hiihh|hjjhk",
                                  "e\\x80\\x80e\\xff|e\\x81\\x81e\\x80|e\\x82\\x82e\\x81|e\\x83\\x83e\\x82|e\\x84\\x84e\\x83|t\\x80\\x80t\\x84|t\\x81\\x81t\\x85|"
                                  "t\\x82\\x82t\\x86|t\\x83\\x83t\\x87|a\\xee\\xeea\\x00|a\\xef\\xefa\\xff|h\\x00\\x00h\\x01|h\\x02\\x02h\\x03"],
    ('FixedEngine', 2, 6, True): ["t..i.n|h.hi.n|n..ien|h.at.n|hhneah|hheshh|heesai|hhosah|hhesah|hasinn|ha.nno"],
    ('FixedEngine', 3, 6, True): ["e\\x00. |e..\\x00|e.\\x80\\xff|e .\\xff|\\xff e\\x00|  . |\\xff .\\x00| \\xff\\x80 |e\\xff\\x80\\x80|et\\x80 "],
    ('FixedEngine', 4, 8, True): ["t\\xff te|tt ee|\\x80\\x80.\\xff\\xff|\\x80\\x80.\\x80 | .. \\x00| ... | .e. |e.e.\\x00|e\\x80\\x80 t"],
    ('Fixed3Engine', 8, True): ["tt\\x80e|\\x00t\\x80\\x00|tte |\\x00t\\x80 |\\x00te\\xff|\\x00t t|\\x80\\x80 \\xff|\\x00t \\x00|\\x00e \\xff"],
    # ---- class runs RunEngine<NLO, NHI, NFO>: NLO = ranges below 0x80 (0 -> 1, 5 -> 6, 7 -> 8), NHI = high ranges, NFO = fold ----
    ("RunEngine", 1, 0, False): ["[a-z]{2,}", "[a-z]{16,}", "[a-z]{17,}", "[a-z]{18,}", "[a-z]{1024,}", "[\\x00-\\x08]{2,}"],
    ("RunEngine", 1, 0, True): ["[a-zA-Z]{8,}"],
    ("RunEngine", 1, 1, False): ["[\\x80-\\xff]{8,}", "[a-c\\xe0-\\xef]{3,}", "[\\x80-\\x9f]{2,}"],
    ("RunEngine", 1, 1, True): ["[A-Za-z\\xf8-\\xff]{8,}", "[A-Za-z\\x80-\\xff]{2,}"],
    ("RunEngine", 1, 2, False): ["[\\xf8-\\xff\\x80-\\x9f]{3,}"],
    ("RunEngine", 1, 2, True): ["[a-zA-Z\\xf8-\\xff\\x80-\\x9f]{8,}"],
    ("RunEngine", 2, 0, False): ["[ \\x00-\\x08]{2,}"],
    ("RunEngine", 2, 0, True): ["[A-Za-z0-9_]{16,}", "[A-Z0-9\\x00-\\x08a-z]{17,}"],
    ("RunEngine", 2, 1, False): ["[ _\\xf8-\\xff]{3,}", "[^\\n]{5,}"],
    ("RunEngine", 2, 1, True): ["[A-Z 0-9a-z\\xe0-\\xef]{18,}"],
    ("RunEngine", 2, 2, False): ["[ _\\xc0-\\xdf\\x80-\\x9f]{2,}"],
    ("RunEngine", 2, 2, True): ["[_a-zA-Z \\xe0-\\xef\\xf8-\\xff]{8,}"],
    ("RunEngine", 3, 0, False): ["[\\x00-\\x080-9 ]{3,}"],
    ("RunEngine", 3, 0, True): ["[\\x00-\\x08a-z 0-9A-Z]{18,}"],
    ("RunEngine", 3, 1, False): ["[ 0-9_\\x80-\\x9f]{2,}"],
    ("RunEngine", 3, 1, True): ["[A-Z a-z0-9_\\xe0-\\xef]{18,}"],
    ("RunEngine", 3, 2, False): ["[ 0-9_\\xe0-\\xef\\x80-\\x9f]{2,}"],
    ("RunEngine", 3, 2, True): ["[\\x0e-\\x1f 0-9A-Z_a-z\\x80-\\x9f\\xf8-\\xff]{3,}"],
    ("RunEngine", 4, 0, False): ["[_A-Z \\x00-\\x08]{2,}"],
    ("RunEngine", 4, 0, True): ["[ a-z0-9A-Z_\\x00-\\x08]{16,}"],
    ("RunEngine", 4, 1, False): ["[_A-Z0-9 \\x80-\\x9f]{2,}"],
    ("RunEngine", 4, 1, True): ["[A-Z\\x00-\\x08a-z_0-9\\x0e-\\x1f\\xf8-\\xff]{3,}"],
    ("RunEngine", 4, 2, False): ["[ _0-9a-z\\xc0-\\xdf\\xf8-\\xff]{3,}"],
    ("RunEngine", 4, 2, True): ["[\\x21-\\x2f_\\x00-\\x08A-Z\\x0e-\\x1fa-z\\xe0-\\xef\\x80-\\x9f]{8,}"],
    ("RunEngine", 6, 0, False): ["[ \\x7b-\\x7eA-Z\\x00-\\x08_]{3,}"],
    ("RunEngine", 6, 0, True): ["[\\x00\\x2cBVdjv]{3,}"],
    ("RunEngine", 6, 1, False): ["[a-z\\x00-\\x08 \\x3a-\\x40_\\xc0-\\xdf]{3,}"],
    ("RunEngine", 6, 1, True): ["[\\x12\\x32VZlvz\\xc0-\\xdf]{18,}"],
    ("RunEngine", 6, 2, False): ["[\\x7b-\\x7e _0-9A-Z\\xe0-\\xef\\x80-\\x9f]{17,}"],
    ("RunEngine", 6, 2, True): ["[\\x14\\x30\\x36JVdfj\\xc0-\\xdf\\x80-\\x9f]{2,}"],
    ("RunEngine", 8, 0, False): ["[\\x00\\x0a0Xhnt]{18,}"],
    ("RunEngine", 8, 1, False): ["[6BFPVdx\\xf8-\\xff]{2,}"],
    ("RunEngine", 8, 2, False): ["[\\x08 BVXhz\\xf8-\\xff\\xc0-\\xdf]{2,}"],
    # ---- hashed engine: (sparse path possible, table copies) ----
    ("HashEngine", False, 1): ["(?i)\\x80\\x00a|ba\\x80|\\x00b\\x80|a\\xffa|.a\\x00"],
    ("HashEngine", False, 32): ["\\x00\\x01|\\x02\\x03|\\x04\\x05|\\x06\\x07|\\x08\\x09", "\\xe0\\xe1|\\xe2\\xe3|\\xe4\\xe5|\\xe6\\xe7|\\xe8\\xe9",
                                "\\x89\\x86|x\\x8c|\\x83x|.\\x8f|\\x8dy"],
    ("HashEngine", True, 1): [HASH_WIDE],
    ("HashEngine", True, 32): ["\\x0f\\x01|\\x02\\x0d\\x00|\\x0c\\x0f|\\x08\\x0c|\\x05\\x0f|\\x03\\x06"],
}

_NO_EXACT_D0 = "a single-byte filter (delta 0) is never exact: gscan_compile clears `exact` so its zero-mask second term vanishes"
UNREACHABLE = {
    **{("FixedEngine", 0, k, True): _NO_EXACT_D0 for k in (1, 2, 3, 4, 6, 8)},
    ("HashEngine", False, 16): "hash_table_copies() (device_types.h) gives 32 or 1 copies; 16 only in a -DGS_HASH_COPIES=16 build",
    ("HashEngine", True, 16): "hash_table_copies() (device_types.h) gives 32 or 1 copies; 16 only in a -DGS_HASH_COPIES=16 build",
    **{("RunEngine", 8, h, True): "the fold removes two of at most kMaxRunRangesLow = 8 low ranges (pattern.h), leaving at most 6"
       for h in (0, 1, 2)},
}


def family(key):
    return key[0]


def kmap(n):
    """raw test count -> the K the launchers instantiate (5 -> 6, 7 -> 8; scan_kernels.cu launch_fixed_de and friends)"""
    return n if n <= 4 else (6 if n <= 6 else 8)


def instantiation(info):
    """gscan_pattern_info -> VARIANTS key of the kernel that scans for the pattern (None: no scan kernel)"""
    v, k = info["scan_variant"], info["scan_kernel"]
    if k == G.KERNEL_RUN:
        nlo, nhi = v & 15, (v >> 4) & 3
        return ("RunEngine", 1 if nlo == 0 else kmap(nlo), min(nhi, 2), bool(v & 0x40))
    if k == G.KERNEL_HASH:
        return ("HashEngine", bool(v & 4), (v >> 3) & 63)
    if k == G.KERNEL_BALANCED:
        d = (v >> 4) & 7  # launch_scan_fixed: delta 1..3 -> D = delta, anything else -> 4
        return ("FixedBEngine", d if 1 <= d <= 3 else 4, kmap(v & 15), bool(v & 0x200))
    if k == G.KERNEL_TRIPLE:
        return ("Fixed3Engine", kmap((v >> 11) & 31), bool(v & 0x10000))
    if k == G.KERNEL_PAIR:
        return ("FixedEngine", min((v >> 4) & 7, 4), kmap(v & 15), bool(v & 0x80))
    return None


def dispatch_cases():
    """every instantiation the launchers of scan_kernels.cu can reach, read from their switch statements"""
    src = open(os.path.join(ROOT, "grab_b200", "csrc", "scan_kernels.cu")).read()
    ks = lambda eng, rest: sorted({int(x) for x in re.findall(r"launch(?:_g)?<%s<(?:D, )?(\d+), %s>" % (eng, rest), src)})
    ds_fixed = sorted({int(x) for x in re.findall(r"launch_fixed_de<(\d), (?:true|false)>", src)})
    ds_bal = sorted({int(x) for x in re.findall(r"launch_fixedb<(\d)>", src)})
    nlo = sorted({int(x) for x in re.findall(r"launch<RunEngine<(\d), NHI, NFO>", src)})
    hf = sorted({(int(a), int(b)) for a, b in re.findall(r"launch_run_hf<(\d), (\d)>", src)})
    cases = set()
    cases |= {("FixedEngine", d, k, ex) for d, k, ex in itertools.product(ds_fixed, ks("FixedEngine", "EX"), (False, True))}
    cases |= {("Fixed3Engine", k, ex) for k, ex in itertools.product(ks("Fixed3Engine", "EX"), (False, True))}
    cases |= {("FixedBEngine", d, k, al) for d, k, al in itertools.product(ds_bal, ks("FixedBEngine", "AL"), (False, True))}
    cases |= {("RunEngine", n, h, bool(f)) for n, (h, f) in itertools.product(nlo, hf)}
    cases |= {("HashEngine", sp, c) for sp, c in itertools.product((False, True), (1, 16, 32))}
    return cases


def test_dispatch_cases_parsed():
    c = dispatch_cases()
    # 5 distances x 6 test counts x 2, 6 x 2, 4 x 5 x 2, 6 x 3 x 2, 2 x 3
    assert len(c) == 60 + 12 + 40 + 36 + 6, len(c)


def test_every_dispatch_case_is_covered_or_unreachable():
    cases = dispatch_cases()
    assert not set(VARIANTS) & set(UNREACHABLE)
    assert set(VARIANTS) | set(UNREACHABLE) == cases, (sorted(cases - set(VARIANTS) - set(UNREACHABLE)),
                                                       sorted((set(VARIANTS) | set(UNREACHABLE)) - cases))
    assert all(UNREACHABLE.values())
    assert all(VARIANTS.values())


def test_high_bytes_in_every_family():
    hb = re.compile(r"\\x(?:00|[89a-f][0-9a-f])")
    for fam in ("FixedEngine", "Fixed3Engine", "FixedBEngine", "RunEngine", "HashEngine"):
        rows = [k for k in VARIANTS if k[0] == fam]
        assert sum(any(hb.search(p) for p in VARIANTS[k]) for k in rows) >= len(rows) * 3 // 4, fam


@pytest.mark.parametrize("key", sorted(VARIANTS, key=str), ids=str)
def test_pattern_routes_to_its_instantiation(key, monkeypatch):
    for env in ("GSCAN_HASH_PRE", "GSCAN_NO_FIXEDB"):  # compile-time switches of the routing
        monkeypatch.delenv(env, raising=False)
    for pat in VARIANTS[key]:
        assert instantiation(G.Pattern(pat).info) == key, pat
