"""CPU checks of the device topology generator's host side: the ctypes mirror of gm_topology_tables against the header,
and Network.pick_fresh_seeds against pick_seed called once per env (the global stream must end in the same state)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_topology_tables_mirror_matches_the_header(tmp_path):
    from graph_marl_b200 import _lib

    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "graphmarl_b200.h"', "int main(void) {",
             '  printf("max_nodes %d\\n", GM_TOPOLOGY_MAX_NODES);',
             '  printf("size %zu\\n", sizeof(gm_topology_tables));']
    for fname, _ in _lib.TopologyTables._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(gm_topology_tables, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    r = subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.fail("the header does not declare a field the ctypes mirror names:\n" + r.stderr[-2000:])
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["max_nodes"]) == _lib.GM_TOPOLOGY_MAX_NODES
    assert int(got["size"]) == C.sizeof(_lib.TopologyTables)
    for fname, _ in _lib.TopologyTables._fields_:
        assert getattr(_lib.TopologyTables, fname).offset == int(got[fname]), fname


def _one_by_one(net, n):
    return [net.pick_seed(None, None, net.exclude_seeds)[0] for _ in range(n)]


def _same_state(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


@pytest.mark.parametrize("hit_exclusion", [False, True])
def test_pick_fresh_seeds_draws_like_pick_seed_per_env(hit_exclusion):
    from graph_marl_b200.env.network import Network

    n = 4096
    np.random.seed(31)
    draws = np.random.randint(2**31 - 1, size=n)
    # an exclusion list that contains two of the draws forces the call-by-call replay (pick_seed redraws an excluded seed)
    excluded = [int(draws[5]), int(draws[4000])] if hit_exclusion else [1, 2, 3]
    net = Network(20, random_topology=True, excluded_seeds=excluded)
    np.random.seed(123 if not hit_exclusion else 31)
    ref = _one_by_one(net, n)
    ref_state = np.random.get_state()
    np.random.seed(123 if not hit_exclusion else 31)
    got = net.pick_fresh_seeds(n)
    assert got.dtype == np.int64 and got.tolist() == ref
    assert _same_state(np.random.get_state(), ref_state)
    assert not set(got.tolist()) & set(excluded)
