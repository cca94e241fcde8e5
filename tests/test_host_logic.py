"""Host-side logic that needs no GPU: action packing, the network generator, the draw tables (kept identical
to the oracle's), the C-ABI library's exports, sharding + the payoff all-reduce over gloo (world_size 2)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_draw_tables_match_the_oracle_contract():
    from cygym_b200 import draw_tables as DT
    from oracle import draws as D
    for p in (0.0, 1e-9, 0.1, 0.25, 0.5, 0.999, 1.0):
        assert DT.bernoulli_threshold(p) == D.bernoulli_threshold(p)
    for lam in (0.0, 0.3, 0.7, 1.5, 4.0):
        assert DT.poisson_table(lam) == D.poisson_table(lam)
    assert DT.triangular_ceil_table(2, 5)[:7] == D.triangular_ceil_table(2, 5)
    # the integer tables reproduce the distributions: P(ceil(triangular(0,2,5)) = 1) = 0.1, <= 2 -> 0.4
    t = DT.triangular_ceil_table(2, 5)
    assert abs(t[0] / 2**32 - 0.1) < 1e-9 and abs(t[1] / 2**32 - 0.4) < 1e-9 and abs(t[3] / 2**32 - 14 / 15) < 1e-9


def test_action_pack_roundtrip_and_errors():
    from cygym_b200.vector_env import ActionBatch
    hdr, mask, order = ActionBatch.pack([(6, [1], [3, 40, 99], 7), None, (1, [0, 2], [], 0)], ["defender", "attacker", "attacker"], 100)
    assert hdr[0, 0] == (6 | (0 << 8) | (1 << 16)) and hdr[0, 2] == 3 and hdr[0, 3] == 7
    assert mask[0, 0] == 1 << 3 and mask[0, 1] == 1 << 8 and mask[0, 3] == 1 << 3
    assert hdr[1, 0] == (0x80 | (1 << 8)) and not mask[1].any()
    assert hdr[2, 0] == (1 | (1 << 8) | (2 << 16)) and hdr[2, 1] == (0 | (2 << 8))
    with pytest.raises(ValueError):
        ActionBatch.pack([(1, [0], [5, 2], 0)], 0, 100)            # unsorted needs order_form
    with pytest.raises(IndexError):
        ActionBatch.pack([(1, [0], [100], 0)], 0, 100)
    h, m, o = ActionBatch.pack([(1, [0], [5, 2, 5], 0)], 0, 100, order_form=True)
    assert list(o[0, :3]) == [5, 2, 5] and h[0, 2] == 3
    # unpack is the inverse of pack, in set form and in order form
    acts = [(6, [1], [3, 40, 99], 7), None, (1, [0, 2], [], 0), (-3, [-8, 7, 0, 5], list(range(0, 100, 7)), -500)]
    assert ActionBatch.unpack(*ActionBatch.pack(acts, 0, 100)[:2]) == acts
    acts[0] = (6, [1], [99, 3, 40, 3], 7)
    assert ActionBatch.unpack(*ActionBatch.pack(acts, 1, 100, order_form=True)) == acts


def test_compact_action_rows_roundtrip_and_ranges():
    """The 2-word header of the host-buffer rows (include/cygym_b200.h, cyg_unpack_actions) holds everything hdr[4] holds
    inside its documented ranges, and refuses what it cannot hold."""
    from cygym_b200.vector_env import ActionBatch, compact_action_rows, expand_action_rows
    rng = np.random.default_rng(5)
    acts, modes = [], []
    for b in range(400):
        if b % 17 == 0:
            acts.append(None)
        else:
            devs = sorted(int(d) for d in rng.choice(100, size=int(rng.integers(0, 100)), replace=False))
            acts.append((int(rng.integers(-3, 16)), [int(x) for x in rng.integers(-8, 8, size=int(rng.integers(0, 5)))], devs, int(rng.integers(-500, 500))))
        modes.append(int(rng.integers(0, 2)))
    hdr, mask, _ = ActionBatch.pack(acts, modes, 100)
    hdr[5, 2] |= np.uint32(77 << 16)                       # device_indices[0] + 1 as sample_action writes it
    rows = compact_action_rows(hdr, mask)
    assert rows.shape == (400, 2 + 4) and rows.dtype == np.int32
    h2, m2 = expand_action_rows(rows)
    assert np.array_equal(h2, hdr) and np.array_equal(m2, mask)
    for bad in ((1, [9], [1], 0), (1, [0], [1], 40000), (1, [-9], [1], 0)):
        h, m, _ = ActionBatch.pack([bad], 0, 100)
        with pytest.raises(ValueError):
            compact_action_rows(h, m)


@pytest.mark.parametrize("M,subnets", [(20, 1), (50, 3), (100, 8), (2000, 64)])
def test_synthetic_network_invariants(M, subnets):
    from cygym_b200 import synthetic_network
    from cygym_b200._capi import DEV_COMP, DEV_NYA, DEV_OWNED, ST_DC, ST_SERVER
    net = synthetic_network(M, n_subnets=subnets, seed=3)
    assert net.row_ptr[0] == 0 and net.row_ptr[-1] == net.E == len(net.col)
    for u in range(M):
        row = net.col[net.row_ptr[u]:net.row_ptr[u + 1]]
        assert np.all(np.diff(row) > 0) and u not in row            # ascending unique neighbours, no self loops
    assert net.mult.min() >= 1 and net.mult.max() <= 4
    st = net.dev_static
    n_dc = int((st & ST_DC).astype(bool).sum())
    assert n_dc == max(1, int(np.ceil(net.cfg["numOfDevice"] / 50)))
    assert np.all(((st & ST_SERVER) != 0) ^ ((st & ST_DC) != 0))     # every non-DC device is a server (volt:1680-1683)
    dev = net.template["dev"]
    owned = (dev & DEV_OWNED) != 0
    assert owned.sum() == max(1, round(0.05 * net.cfg["numOfDevice"])) and np.all((dev[owned] & DEV_COMP) != 0)
    assert np.all((dev[owned] & DEV_NYA) == 0)
    deg = np.zeros(M, int)
    np.add.at(deg, np.repeat(np.arange(M), np.diff(net.row_ptr)), 1)
    np.add.at(deg, net.col, 1)
    assert deg.min() >= 1                                            # the PA repair of evolve_network stays dead
    b = net.algorithmic_bytes_per_step()
    assert b == 2 * 4 * M + (net.E + 7) // 8 + 128 + 4 + (M + 7) // 8 + 12
    # CVE table has the reference's 15-column schema and the two hard-coded ids
    from cygym_b200 import cve
    assert list(net.cve_table.keys()) == cve.COLUMNS and len(cve.COLUMNS) == 15
    assert net.cve_table["matchCriteriaId"][:2] == [cve.VOLT_CVE_ID, cve.VOLT_DC_CVE_ID]


def test_shard_range_partitions():
    from cygym_b200.payoff import shard_range
    for total in (0, 1, 7, 1024, 65537):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[r][1] == spans[r + 1][0] for r in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads without a GPU and exports exactly what include/cygym_b200.h declares."""
    from cygym_b200 import _capi as K
    K.build()
    lib = C.CDLL(K.LIB_PATH)
    hdr = open(os.path.join(ROOT, "include", "cygym_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(cyg_[a-z_]+)\s*\(", hdr)))
    assert declared, "no declarations found"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert sorted(K.EXPORTS) == declared
    lib.cyg_version.restype = C.c_int
    assert lib.cyg_version() == K.ABI_VERSION


def test_product_package_never_imports_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pkg = os.path.join(ROOT, "cygym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "cyg_oracle" not in src and "tests.emu" not in src, f


_GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
from cygym_b200.payoff import shard_range, reduce_payoff
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
n_rollouts, T = 10, 20
lo, hi = shard_range(n_rollouts, rank, world)
# every rollout r of pair (i, j) contributes r + 100*i + 10*j to column 0 and 1 to column 2
part = torch.zeros(3, 2, 10, dtype=torch.float64)
for i in range(3):
    for j in range(2):
        for r in range(lo, hi):
            part[i, j, 0] += r + 100 * i + 10 * j
            part[i, j, 2] += T
out = reduce_payoff(part, n_rollouts, T)
exp0 = torch.tensor([[sum(range(n_rollouts)) / n_rollouts + 100 * i + 10 * j for j in range(2)] for i in range(3)], dtype=torch.float64)
assert torch.allclose(out[..., 0], exp0), (rank, out[..., 0])
assert torch.allclose(out[..., 2], torch.ones(3, 2, dtype=torch.float64))
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_payoff_reduce_over_gloo_world_size_2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER % {"root": ROOT})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29541", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"rank {r} ok" in o, o
