"""Executable statement of the copy emission of gp_decide_tables (csrc/gangpack_tables.cuh), on the CPU.

The table build writes, per (shape, instance group), the expansion list E: node n repeated c(n) times in priority order
(E[S[n] .. S[n+1]) = n, S the exclusive prefix of the capacities), cut at kExpandCap entries.  Every application of the
shape walks the same nodes; only the driver's node p takes cd = cap(p | driver) executors instead of c0d = c(p).  So an
application of k executors is placed by at most three copies:

    S[p] < k:  E[0, S[p]) ++ p x min(cd, k - S[p]) ++ E[S[p+1], S[p+1] + (k - S[p] - cd))
    otherwise (also a driver in a spare slot, i.e. not an executor candidate):  E[0, k)

provided the list holds k + (c0d - cd) entries; longer applications keep the prefix-table walk.  Distribute-evenly
(single round) is the same statement over c in {0, 1}.  This model mirrors the kernel's index arithmetic (a, b, skip) and
checks it against the definition (pack_tightly.go:45-61 / one round of distribute_evenly.go) on random tables."""
import numpy as np
import pytest

CAP = 1024        # kExpandCap


def expansion(caps, cap=CAP):
    """the table build's scatter: node n fills entries [S[n], S[n] + c(n)) as far as they are below cap"""
    e = np.full(cap, -1, dtype=np.int64)
    s = 0
    for n, c in enumerate(caps):
        lo, hi = s, min(s + int(c), cap)
        e[lo:max(lo, hi)] = n
        s += int(c)
    return e[:min(s, cap)]


def copy_emission(e, tab, ne, k, dslot, cd, c0d, cap=CAP):
    """the kernel's copy: None when the application needs more than the list (-> table walk)"""
    if k + (c0d - cd) > cap:
        return None
    spd = int(tab[dslot]) if dslot < ne else 0
    a = spd if (dslot < ne and spd < k) else k
    b = min(cd, k - a)
    skip = c0d - b
    return [int(e[t]) if t < a else (dslot if t < a + b else int(e[t + skip])) for t in range(k)]


def definition(caps, k, dpos, cd):
    out = []
    for n, c in enumerate(caps):
        c = cd if n == dpos else int(c)
        take = min(c, k - len(out))
        out += [n] * take
        if len(out) == k:
            break
    return out


def case(caps, k, dslot, cd, cap=CAP):
    caps = np.asarray(caps, dtype=np.int64)
    ne = len(caps)
    tab = np.concatenate([[0], np.cumsum(caps)[:-1]])
    c0d = int(caps[dslot]) if dslot < ne else 0
    got = copy_emission(expansion(caps, cap), tab, ne, k, dslot, cd, c0d, cap)
    return got, definition(caps, k, dslot if dslot < ne else -1, cd)


@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("seed", range(3))
def test_copy_equals_definition(algo, seed):
    rng = np.random.default_rng(100 * algo + seed)
    checked = copied = 0
    for _ in range(3000):
        ne = int(rng.integers(1, 80))
        caps = rng.integers(0, 6, ne) * (rng.random(ne) < rng.random())
        if algo == 1:
            caps = (caps > 0).astype(np.int64)
        total = int(caps.sum())
        if total == 0:
            continue
        dslot = int(rng.integers(0, ne + 3))                       # >= ne: a spare slot (driver-only node)
        c0d = int(caps[dslot]) if dslot < ne else 0
        cd = int(rng.integers(0, c0d + 1)) if dslot < ne else 0
        room = total - (c0d - cd) if algo == 0 else total - 1     # distribute-evenly: single round needs M[ne] >= k + 1
        if room <= 0:
            continue
        k = int(rng.integers(1, room + 1))
        cap = int(rng.choice([CAP, 8, max(1, k - 1), k + (c0d - cd)]))
        got, want = case(caps, k, dslot, cd, cap)
        checked += 1
        if got is None:
            assert k + (c0d - cd) > cap
            continue
        assert got == want
        copied += 1
    assert checked > 1500 and copied > 1000


# caps: node 0 holds 3, node 1 nothing, node 2 holds 2, node 3 holds 4 -> E = 0 0 0 2 2 3 3 3 3, S = 0 3 3 5
CAPS = [3, 0, 2, 4]


@pytest.mark.parametrize("k,dslot,cd,where", [
    (2, 3, 1, "driver after the copied range (S[p] >= k)"),
    (5, 3, 4, "driver right after the copied range"),
    (6, 2, 1, "driver inside: 0 < cd < c0d"),
    (6, 2, 0, "driver inside: cd = 0, its executors move on"),
    (6, 2, 2, "driver inside: cd = c0d"),
    (4, 0, 1, "driver before everything else"),
    (7, 0, 3, "driver first node, cd = c0d"),
    (5, 1, 0, "driver on a node without capacity"),
    (6, 6, 0, "driver in a spare slot"),
    (9, 5, 0, "spare slot, the whole list"),
])
def test_splice_cases(k, dslot, cd, where):
    got, want = case(CAPS, k, dslot, cd)
    assert got == want, where


def test_zero_executors():
    got, want = case(CAPS, 0, 2, 1)
    assert got == want == []


def test_capacity_at_and_beyond_the_list():
    caps = np.ones(3000, dtype=np.int64)
    caps[5] = 4
    # k + (c0d - cd) == CAP: copied; one more: the table walk
    got, want = case(caps, CAP - 2, 5, 2)
    assert got is not None and got == want
    got, _ = case(caps, CAP - 1, 5, 2)
    assert got is None
    got, want = case(caps, CAP, 3000, 0)                  # spare-slot driver, exactly the list
    assert got == want
    assert case(caps, CAP + 1, 3000, 0)[0] is None


def test_expansion_is_cut_at_the_cap():
    caps = np.full(10, 300, dtype=np.int64)
    e = expansion(caps)
    assert len(e) == CAP
    assert list(e[:301]) == [0] * 300 + [1] and e[-1] == CAP // 300
