"""collapse_ratio in plain Python: the reference the GPU collapse must match, and a brute-force form of the same rule.

Rows are ordered by count descending, then key bytes ascending.  Key a may be the parent of b iff both have the same
length and differ in exactly one byte, a comes first in the order and float(count(a)) >= ratio * float(count(b)).
parent(b) is the first such a in the order; every row's count goes to the end of its parent chain (its root), and
the result has one row per root.  Rows with count 0 take no part."""
from collections import defaultdict


def _order(table):
    rows = [(k, c) for k, c in table.items() if c > 0]
    rows.sort(key=lambda kc: (-kc[1], kc[0]))
    return rows


def _fold(rows, parent):
    root = {}
    for k, _ in rows:                      # rows in order: a parent's root is known before its children's
        p = parent.get(k)
        root[k] = k if p is None else root[p]
    out = {}
    for k, c in rows:
        out[root[k]] = out.get(root[k], 0) + c
    return out


def collapse_reference(table, ratio):
    """dict[bytes, int] -> dict[bytes, int], neighbours found by grouping on (len, p, key[:p], key[p+1:])."""
    rows = _order(table)
    rank = {k: i for i, (k, _) in enumerate(rows)}
    groups = defaultdict(list)
    for k, _ in rows:                      # members appended in order: a group's first member is its earliest
        for p in range(len(k)):
            groups[(len(k), p, k[:p], k[p + 1:])].append(k)
    parent = {}
    for k, c in rows:
        need = ratio * float(c)
        best = None
        for p in range(len(k)):
            a = groups[(len(k), p, k[:p], k[p + 1:])][0]
            if a != k and float(table[a]) >= need and (best is None or rank[a] < rank[best]):
                best = a
        if best is not None:
            parent[k] = best
    return _fold(rows, parent)


def collapse_brute_force(table, ratio):
    """The same rule over every pair of rows, O(n^2)."""
    rows = _order(table)
    parent = {}
    for j, (b, cb) in enumerate(rows):
        for a, ca in rows[:j]:             # the first qualifying a in the order
            if len(a) == len(b) and sum(x != y for x, y in zip(a, b)) == 1 and float(ca) >= ratio * float(cb):
                parent[b] = a
                break
    return _fold(rows, parent)


def roots(table, ratio):
    """The keys that have no parent (the keys of the collapsed table)."""
    rows = _order(table)
    rank = {k: i for i, (k, _) in enumerate(rows)}
    out = set()
    for k, c in rows:
        if not any(len(a) == len(k) and rank[a] < rank[k] and sum(x != y for x, y in zip(a, k)) == 1
                   and float(ca) >= ratio * float(c) for a, ca in rows):
            out.add(k)
    return out
