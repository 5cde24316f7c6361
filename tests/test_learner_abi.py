"""CPU check of the learner's C-ABI structs (gm_opt_entry, gm_opt_pair, gm_opt_hparams): the ctypes mirrors in
graph_marl_b200/_lib.py must have the sizes and field offsets the C compiler gives include/graphmarl_b200.h."""
import ctypes as C
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PAIRS = [("gm_opt_entry", "OptEntry"), ("gm_opt_pair", "OptPair"), ("gm_opt_hparams", "OptHparams")]


def test_learner_ctypes_mirrors_match_the_header(tmp_path):
    from graph_marl_b200 import _lib

    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "graphmarl_b200.h"', "int main(void) {",
             '  printf("partials %d\\n", GM_LEARNER_PARTIALS);']
    for cname, pyname in PAIRS:
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in getattr(_lib, pyname)._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    r = subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.fail("the header does not declare a field the ctypes mirror names:\n" + r.stderr[-2000:])
    got = {}
    for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines():
        *key, v = ln.split()
        got[tuple(key)] = int(v)
    assert got[("partials",)] == _lib.GM_LEARNER_PARTIALS
    for cname, pyname in PAIRS:
        cls = getattr(_lib, pyname)
        assert C.sizeof(cls) == got[(cname, "size")], cname
        for fname, _ in cls._fields_:
            assert getattr(cls, fname).offset == got[(cname, fname)], (cname, fname)
