"""tests/isocorr_reference.py (the definitions of mmseq -isocorr) against independent computations on small hand-made
cases: np.corrcoef on x and log x, a brute-force count of P(x_i > x_j) with ties, the pair order against
itertools.combinations per gene, and the shared fragments counted record by record from a .hits file."""
import itertools

import numpy as np

from mmseq_b200 import hostlib
from tests import isocorr_reference as iref


def _genes(sizes, rng):
    """a gene CSR over a permutation of the rows: gene g has sizes[g] members"""
    n = int(sum(sizes))
    members = rng.permutation(n).astype(np.int32)
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64), members


def test_pairs_follow_combinations_per_gene():
    rng = np.random.default_rng(1)
    sizes = [3, 0, 1, 2, 5, 1, 4]
    gptr, mem = _genes(sizes, rng)
    g, a, b, ma, mb, base = iref.pairs(gptr, mem)
    want = [(gi, x, y) for gi, k in enumerate(sizes) for x, y in itertools.combinations(range(k), 2)]
    assert list(zip(g.tolist(), a.tolist(), b.tolist())) == want
    assert (ma == mem[gptr[g] + a]).all() and (mb == mem[gptr[g] + b]).all()
    assert base.tolist() == np.concatenate([[0], np.cumsum([k * (k - 1) // 2 for k in sizes])])[:-1].tolist()
    k = np.diff(gptr)[g]
    assert (iref.pair_index(base, g, a, b, k) == np.arange(len(g))).all()
    gene_of, local_of = iref.gene_local(gptr, mem, len(mem))
    for gi, kk in enumerate(sizes):
        rows = mem[gptr[gi]:gptr[gi + 1]]
        assert (gene_of[rows] == (gi if kk >= 2 else -1)).all()
        assert (local_of[rows] == (np.arange(kk) if kk >= 2 else -1)).all()


def test_correlations_equal_corrcoef_and_prob_equals_brute_force():
    rng = np.random.default_rng(2)
    C, L = 4, 64
    sizes = [2, 3, 6]
    gptr, mem = _genes(sizes, rng)
    n = len(mem)
    z = rng.standard_normal((C, 1, L))
    x = np.exp(rng.normal(0.0, 1.0, (C, n, L)) + 0.8 * z * rng.choice([-1, 1], (1, n, 1)))
    x[:, mem[1]] = x[:, mem[0]]                                          # gene 0: an exact copy, all ties
    got = iref.summaries(x, gptr, mem)
    _, _, _, ma, mb, _ = iref.pairs(gptr, mem)
    flat = np.concatenate(list(x), axis=1)                               # draws of chain 0, then chain 1, ...
    for p, (i, j) in enumerate(zip(ma, mb)):
        u, v = flat[i], flat[j]
        assert abs(got["corr_mu"][p] - np.corrcoef(u, v)[0, 1]) < 1e-12
        assert abs(got["corr_log_mu"][p] - np.corrcoef(np.log(u), np.log(v))[0, 1]) < 1e-12
        gt = sum(1.0 if s > t else 0.5 if s == t else 0.0 for s, t in zip(u, v))
        assert got["prob_1_gt_2"][p] == gt / (C * L)
    assert got["corr_mu"][0] == 1.0 and got["prob_1_gt_2"][0] == 0.5     # clamped, ties count one half


def test_pooled_centring_is_not_per_chain():
    """two chains each perfectly anti-correlated within, with shifted levels: the pooled correlation is positive"""
    L = 16
    t = np.linspace(-1, 1, L)
    x = np.stack([np.stack([10 + t, 10 - t]), np.stack([20 + t, 20 - t])])
    got = iref.summaries(x, np.array([0, 2]), np.array([0, 1]))
    flat = np.concatenate(list(x), axis=1)
    assert got["corr_mu"][0] > 0.9 and abs(got["corr_mu"][0] - np.corrcoef(flat)[0, 1]) < 1e-12


def test_nan_rules():
    rng = np.random.default_rng(3)
    L = 32
    x = rng.gamma(2.0, 1.0, (1, 8, L))
    x[0, 1, 5] = np.inf
    x[0, 2, 7] = 0.0
    x[0, 3] = 3.0                                                        # constant
    x[0, 4, 9] = np.nan
    x[0, 5, 3] = -1.0
    gptr, mem = np.array([0, 8]), np.arange(8)
    got = iref.summaries(x, gptr, mem)
    _, _, _, ma, mb, _ = iref.pairs(gptr, mem)
    for p, (i, j) in enumerate(zip(ma, mb)):
        s = {i, j}
        assert np.isnan(got["corr_mu"][p]) == bool(s & {1, 3, 4}), (i, j)
        assert np.isnan(got["corr_log_mu"][p]) == bool(s & {1, 2, 3, 4, 5}), (i, j)
        assert np.isnan(got["prob_1_gt_2"][p]) == (4 in s), (i, j)


def _write_hits(path, transcripts, genes, records):
    with open(path, "w") as f:
        for t in transcripts:
            f.write(f"@TranscriptMetaData\t{t}\t1000\t1200\n")
        for g, mem in genes.items():
            f.write(f"@GeneIsoforms\t{g}\t" + "\t".join(mem) + "\n")
        for r, hits in enumerate(records):
            f.write(f">r{r}\n" + "".join(h + "\n" for h in hits))


def test_shared_fragments_counted_record_by_record(tmp_path):
    rng = np.random.default_rng(4)
    tr = [f"t{i}" for i in range(12)]
    genes = {"g0": tr[0:4], "g1": tr[4:5], "g2": tr[5:9], "g3": tr[9:12]}
    records = []
    for _ in range(400):
        k = int(rng.integers(1, 5))
        records.append(sorted(set(rng.choice(tr[:11], k).tolist()), key=tr.index))   # t11 has no hits
    path = tmp_path / "h.hits"
    _write_hits(path, tr, genes, records)
    # every gene's observed isoforms in header order, as the host program hands them to mmq_set_groups
    for layout in (hostlib.LAYOUT_COLLAPSED, hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH):
        h = hostlib.load_hits(str(path), layout)
        gptr, mem = [0], []
        for g in range(h.G):
            for t in h.gene_members[h.gene_ptr[g]:h.gene_ptr[g + 1]]:
                if h.hdr2col[t] >= 0:
                    mem.append(int(h.hdr2col[t]))
            gptr.append(len(mem))
        gptr, mem = np.array(gptr, np.int64), np.array(mem, np.int32)
        got = iref.shared(h.row_ptr, h.col, h.k if layout == hostlib.LAYOUT_COLLAPSED else None, gptr, mem)
        g, a, b, ma, mb, _ = iref.pairs(gptr, mem)
        names = [h.names[h.col2hdr[c]] for c in range(h.n)]
        want = [sum(1 for rec in records if names[i] in rec and names[j] in rec) for i, j in zip(ma, mb)]
        assert got.tolist() == want
        assert len(got) == 6 + 6 + 1 and sum(want) > 0                    # g1 has one isoform, t11 none: g3 one pair
