"""Copy emission of the table path (gp_decide_tables): placements copied from the per-(shape, instance group) expansion
lists with the driver's node spliced in, and the prefix-table walk for applications that need more than the list holds
(kExpandCap = 1024 entries), against the oracle through the C ABI, in both ExecutorNodes widths.  The splice cases the
CPU model (test_table_expansion_model.py) states are checked to occur here."""
import numpy as np
import pytest

from helpers import assert_same_results, res_aos

pytestmark = pytest.mark.gpu
CAP = 1024
KEYS = ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu", "count", "group")
WIDTHS = (None, dict(quantity_bits=64, node_bits=16, offsets=False))


@pytest.fixture(scope="module")
def packer(gangpack):
    p = gangpack.GangPacker()
    yield p
    p.close()


def _want(oracle, algo, cpu, mem, gpu, eoff, eorder, doff, dorder, a):
    """oracle, instance group by instance group, assembled into (driver_node, executor_nodes, off) of the whole batch"""
    count = a["count"]
    off = np.concatenate([[0], np.cumsum(count)]).astype(np.int64)
    dn = np.full(len(count), -1, np.int32)
    en = np.full(max(int(off[-1]), 1), -1, np.int32)
    for grp in range(len(eoff) - 1):
        sel = np.nonzero(a["group"] == grp)[0]
        drv = res_aos(a["drv_cpu"][sel], a["drv_mem"][sel], a["drv_gpu"][sel])
        exe = res_aos(a["exe_cpu"][sel], a["exe_mem"][sel], a["exe_gpu"][sel])
        _, wd, we, woff, _ = oracle.closed_batch(algo, 0, cpu, mem, gpu, dorder[doff[grp]:doff[grp + 1]], eorder[eoff[grp]:eoff[grp + 1]],
                                                 drv, exe, count[sel], None, n_threads=8)
        for j, i in enumerate(sel):
            dn[i] = wd[j]
            if wd[j] >= 0:
                en[off[i]:off[i + 1]] = we[woff[j]:woff[j + 1]]
    return dn, en, off


def _pack_both_widths(packer, a, algo):
    res = []
    for wire in WIDTHS:
        got = packer.pack_batch(a, algo, 0, wire=wire)
        assert packer.stats()["scan_path_apps"] == 0           # every application was decided by the tables
        res.append((got[0], np.asarray(got[1]).astype(np.int32), got[2]))
    return res


def _splice_case(cpu, mem, order, a, i, driver):
    """which part of the splice formula application i exercises (tightly-pack, no gpu)"""
    ec, em, k = a["exe_cpu"][i], a["exe_mem"][i], int(a["count"][i])
    if k == 0:
        return "k=0"
    pos = np.nonzero(order == driver)[0]
    if pos.size == 0:
        return "spare slot"
    caps = np.minimum(np.maximum(cpu[order], 0) // ec, np.maximum(mem[order], 0) // em)
    p = int(pos[0])
    sp, c0 = int(caps[:p].sum()), int(caps[p])
    if sp >= k:
        return "after the copied range"
    cd = int(min((cpu[driver] - a["drv_cpu"][i]) // ec, (mem[driver] - a["drv_mem"][i]) // em)) if c0 else 0
    if c0 == 0:
        return "no capacity"
    return "cd=0" if cd == 0 else ("cd=c0d" if cd == c0 else "0<cd<c0d")


def test_splice_cases_several_groups(oracle, packer):
    rng = np.random.default_rng(17)
    n, G = 900, 3
    cpu = ((rng.integers(0, 6, n) * 1000 + rng.choice([300, 800], n)) * (rng.random(n) < 0.7)).astype(np.int64)   # zero-capacity runs
    mem = (rng.integers(2, 40, n) << 30).astype(np.int64)
    gpu = np.zeros(n, np.int64)
    groups = rng.integers(0, G, n)
    eorder, dorder, eoff, doff = [], [], [0], [0]
    for g in range(G):
        mine = rng.permutation(np.nonzero(groups == g)[0])
        ex = mine[: int(len(mine) * 0.85)]                                     # the rest: driver-only nodes
        eorder.append(ex)
        # group 0: drivers in executor order (the driver's node is one of the first hosts); group 1: a random driver
        # order; group 2: the driver-only nodes first
        dorder.append([ex, rng.permutation(mine)[: int(len(mine) * 0.6)], np.concatenate([mine[len(ex):], ex])][g])
        eoff.append(eoff[-1] + len(ex)); doff.append(doff[-1] + len(dorder[-1]))
    eorder = np.concatenate(eorder).astype(np.int32); dorder = np.concatenate(dorder).astype(np.int32)
    eoff = np.array(eoff, np.int32); doff = np.array(doff, np.int32)
    q = 3000
    shape = rng.integers(0, 3, q)
    a = {"exe_cpu": np.array([1000, 2000, 500], np.int64)[shape], "exe_mem": np.array([1 << 30, 3 << 30, (2 << 30) + 7], np.int64)[shape],
         "exe_gpu": np.zeros(q, np.int64), "drv_gpu": np.zeros(q, np.int64),
         "drv_cpu": rng.choice([0, 250, 500, 1000, 3000], q).astype(np.int64), "drv_mem": rng.choice([1 << 30, 8 << 30], q).astype(np.int64),
         "count": rng.integers(0, 40, q).astype(np.int32), "group": rng.integers(0, G, q).astype(np.int32)}
    packer.set_snapshot(cpu, mem, gpu, eorder, dorder, eoff, doff)
    for algo in (0, 1):
        want = _want(oracle, algo, cpu, mem, gpu, eoff, eorder, doff, dorder, a)
        for got, wire in zip(_pack_both_widths(packer, a, algo), WIDTHS):
            assert_same_results(got, want, f"algo {algo} wire {wire}")
        if algo == 0:
            seen = {}
            for i in np.nonzero(want[0] >= 0)[0]:
                g = a["group"][i]
                c = _splice_case(cpu, mem, eorder[eoff[g]:eoff[g + 1]], a, i, want[0][i])
                seen[c] = seen.get(c, 0) + 1
            for c in ("k=0", "spare slot", "after the copied range", "cd=0", "0<cd<c0d", "cd=c0d"):
                assert seen.get(c, 0) > 0, (c, seen)


def test_walk_fallback_beyond_the_list(oracle, packer):
    """Counts around kExpandCap: group 0 puts the driver on the first executor node (it displaces one executor there),
    group 1 has driver-only nodes (nothing displaced).  k + displaced > 1024 takes the prefix-table walk -- still on the
    table path (no application goes to the scan) and bit-exact."""
    n0, n1 = 3000, 3002
    cpu = np.full(n0 + n1, 4000, np.int64)
    mem = np.full(n0 + n1, 64 << 30, np.int64)
    gpu = np.zeros(n0 + n1, np.int64)
    e0 = np.arange(n0, dtype=np.int32)
    e1 = np.arange(n0, n0 + n1 - 2, dtype=np.int32)
    eorder = np.concatenate([e0, e1]); eoff = np.array([0, n0, n0 + n1 - 2], np.int32)
    dorder = np.concatenate([e0[:5], np.array([n0 + n1 - 2, n0 + n1 - 1], np.int32)]); doff = np.array([0, 5, 7], np.int32)
    counts = np.array([0, 1, 1000, 1022, 1023, 1024, 1025, 1500, 2500], np.int32)
    q = 2 * len(counts) * 4                                   # >= 32: the tables are used
    a = {"exe_cpu": np.full(q, 1000, np.int64), "exe_mem": np.full(q, 1 << 30, np.int64), "exe_gpu": np.zeros(q, np.int64),
         "drv_cpu": np.full(q, 1000, np.int64), "drv_mem": np.full(q, 1 << 30, np.int64), "drv_gpu": np.zeros(q, np.int64),
         "count": np.tile(counts, q // len(counts)).astype(np.int32), "group": np.repeat([0, 1], q // 2).astype(np.int32)}
    packer.set_snapshot(cpu, mem, gpu, eorder, dorder, eoff, doff)
    for algo in (0, 1):
        want = _want(oracle, algo, cpu, mem, gpu, eoff, eorder, doff, dorder, a)
        assert (want[0] >= 0).all()
        for got, wire in zip(_pack_both_widths(packer, a, algo), WIDTHS):
            assert_same_results(got, want, f"algo {algo} wire {wire}")
