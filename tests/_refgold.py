"""Recorded outputs of the unmodified reference (tests/golden/ref_*.npz, made by tests/golden/make_ref_golden.py).

Full-size score tables are too large to store whole, so a table is kept as its scale (max |score|) and, per group,
the TOP_K best candidates with their scores; small tables are kept whole.  Large tensors are kept as a seeded sample
of their entries plus their max |value|.  The comparisons below mirror what the tests check against the live
reference: score agreement relative to the table's max, and a differing pick accepted only as a near-tie of the
reference's own table."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOP_K = 3
FULL_TABLE_MAX = 1024       # tables with at most this many entries are stored whole
SAMPLE_N = 512


# ---------------------------------------------------------------- writing (tests/golden/make_ref_golden.py)
def pack_tables(prefix, tables):
    """Score tables [eq_n, ...] (reference argmax call order) -> npz entries, concatenated over the tables."""
    tabs = [np.asarray(t, dtype=np.float32).reshape(np.shape(t)[0], -1) for t in tables]
    small = [t.size <= FULL_TABLE_MAX for t in tabs]
    tops = [np.argsort(-t, axis=0, kind="stable")[:TOP_K] for t, w in zip(tabs, small) if not w]   # first index first among equal scores
    big = [t for t, w in zip(tabs, small) if not w]
    return {prefix + "rows": np.array([t.shape[0] for t in tabs], np.int32),
            prefix + "groups": np.array([t.shape[1] for t in tabs], np.int32),
            prefix + "whole": np.array(small),
            prefix + "scale": np.array([np.abs(t).max() for t in tabs], np.float32),
            prefix + "values": np.concatenate([t.reshape(-1) for t, w in zip(tabs, small) if w] or [np.zeros(0, np.float32)]),
            prefix + "top_idx": np.concatenate(tops, 1).astype(np.int16) if tops else np.zeros((TOP_K, 0), np.int16),
            prefix + "top_val": np.concatenate([np.take_along_axis(t, o, 0) for t, o in zip(big, tops)], 1) if tops
            else np.zeros((TOP_K, 0), np.float32)}


def pack_samples(prefix, tensors, n=SAMPLE_N):
    """{name: tensor} -> a seeded sample of each tensor's entries (all of them when it is small) and its max |value|
    (float tensors) or the sums of its entries and of their squares (integer tensors)."""
    names, sizes, counts, idxs, vals, stats = [], [], [], [], [], []
    for i, (name, t) in enumerate(tensors.items()):
        a = np.asarray(t).reshape(-1)
        idx = np.arange(a.size) if a.size <= n else np.sort(np.random.default_rng(i).choice(a.size, n, replace=False))
        names.append(name); sizes.append(a.size); counts.append(idx.size); idxs.append(idx); vals.append(a[idx])
        stats.append([np.abs(a).max()] if a.dtype.kind == "f" else [a.astype(np.int64).sum(), (a.astype(np.int64) ** 2).sum()])
    return {prefix + "names": np.array(names), prefix + "size": np.array(sizes, np.int64), prefix + "count": np.array(counts, np.int32),
            prefix + "idx": np.concatenate(idxs).astype(np.int32), prefix + "val": np.concatenate(vals),
            prefix + "stats": np.array(stats)}


# ---------------------------------------------------------------- reading
def load(name):
    return np.load(os.path.join(GOLD, f"ref_{name}.npz"))


def unpack_tables(z, prefix):
    """-> per table (rows, scale, recorded row indices [k, groups], reference scores there, reference argmax per group)."""
    out, v, c = [], 0, 0
    values, top_idx, top_val = z[prefix + "values"], z[prefix + "top_idx"].astype(np.int64), z[prefix + "top_val"].astype(np.float64)
    for rows, groups, whole, scale in zip(z[prefix + "rows"], z[prefix + "groups"], z[prefix + "whole"], z[prefix + "scale"]):
        rows, groups = int(rows), int(groups)
        if whole:
            t = values[v:v + rows * groups].astype(np.float64).reshape(rows, groups); v += rows * groups
            out.append((rows, float(scale), np.broadcast_to(np.arange(rows)[:, None], t.shape), t, t.argmax(0)))
        else:
            idx = top_idx[:, c:c + groups]
            out.append((rows, float(scale), idx, top_val[:, c:c + groups], idx[0])); c += groups
    return out


def _sample(z, prefix, name, got):
    names = list(z[prefix + "names"])
    assert name in names, f"{prefix}{name} was not recorded"
    i = names.index(name)
    start = int(z[prefix + "count"][:i].sum())
    sl = slice(start, start + int(z[prefix + "count"][i]))
    a = np.asarray(got).reshape(-1)
    assert a.size == int(z[prefix + "size"][i]), f"{prefix}{name}: {a.size} entries vs {int(z[prefix + 'size'][i])} recorded"
    return a, z[prefix + "idx"][sl], z[prefix + "val"][sl], z[prefix + "stats"][i]


def compare_steps(name, got_tables, ref, group_independent_until, score_rtol, tie_eps):
    """Walk the greedy search against the recorded reference tables.  While group j has had no differing pick, its
    scores must agree with the reference's at every recorded row; a different pick must be a recorded candidate whose
    reference score is within tie_eps (relative) of the reference's best.  Steps at index >= group_independent_until
    mix all groups: the walk stops there once a pick has differed.  Returns (flips, worst score error, groups compared,
    gaps of the differing picks)."""
    assert len(got_tables) == len(ref), f"{name}: {len(got_tables)} score tables vs {len(ref)} recorded"
    flips, worst, compared, gaps = 0, 0.0, 0, []
    diverged = None
    for i, (g, (rows, scale, idx, val, best)) in enumerate(zip(got_tables, ref)):
        g = np.asarray(g, dtype=np.float64).reshape(rows, -1)
        groups = g.shape[1]
        assert idx.shape[1] == groups, f"{name} step {i}: {groups} groups vs {idx.shape[1]} recorded"
        if diverged is not None and i >= group_independent_until and diverged.any():
            break
        if diverged is None or diverged.shape[0] != groups:
            diverged = np.zeros(groups, dtype=bool)
        for j in range(groups):
            if diverged[j]:
                continue
            err = np.abs(g[idx[:, j], j] - val[:, j]).max() / (scale + 1e-300)
            worst = max(worst, err); compared += 1
            assert err < score_rtol, f"{name} step {i} group {j}: score table differs by {err:.3e} (rel. to table max)"
            bg, br = int(g[:, j].argmax()), int(best[j])
            if bg != br:
                hit = np.nonzero(idx[:, j] == bg)[0]
                assert hit.size, f"{name} step {i} group {j}: picked {bg}, not among the reference's best {list(idx[:, j])}"
                rbest = val[np.nonzero(idx[:, j] == br)[0][0], j]
                gap = (rbest - val[hit[0], j]) / (abs(rbest) + 1e-300)
                assert gap < tie_eps, f"{name} step {i} group {j}: picked {bg}, reference {br}, reference gap {gap:.3e}"
                flips += 1; diverged[j] = True; gaps.append(float(gap))
    return flips, worst, compared, gaps


def sample_rel_err(z, prefix, name, got):
    """max |got - recorded| over the recorded entries, relative to the recorded tensor's max |value|."""
    a, idx, val, stats = _sample(z, prefix, name, got)
    return float(np.abs(a[idx].astype(np.float64) - val).max() / (float(stats[0]) + 1e-300))


def assert_sample_equal(z, prefix, name, got, what):
    """Integer tensors: the recorded entries are equal and so are the sums of all entries and of their squares."""
    a, idx, val, stats = _sample(z, prefix, name, got)
    assert np.array_equal(a[idx], val), f"{what}: sampled entries differ from the reference"
    a = a.astype(np.int64)
    assert int(a.sum()) == int(stats[0]) and int((a ** 2).sum()) == int(stats[1]), \
        f"{what}: differs from the reference outside the sampled entries"
