"""CPU oracle for weighted (schema 2) hits files — test infrastructure on top of oracle/oracle.py and
oracle/tables.py, which stay the restatement of the reference's reader and main().

Schema 2 is this package's extension of the binary format: one fp32 weight per hit after a record's
transcript indices.  The model: fragment f picks transcript t with probability proportional to
mu_t * w_ft, EM maximises sum_f log sum_{t in f} mu_t w_ft - sum_t mu_t l_t; the initial mu and the
unique hits ignore the weights; .k and .M describe the distinct sets exactly as for the same records
without weights."""
import struct
from unittest import mock

import numpy as np

from oracle import oracle as orc
from oracle import tables

_Problem = orc.Problem   # run() replaces orc.Problem while tables.run executes


class HitsFile(orc.HitsFile):
    """orc.HitsFile that also reads schema 2: `weights` holds each record's fp32 weights, aligned with its
    names (None for the other schemas)."""

    def __init__(self, path):
        self.weights = None
        super().__init__(path)

    def _binary(self, b):
        pos = b.index(b"\n") + 1
        (schema,) = struct.unpack_from("<I", b, pos)
        if schema != 2:
            return super()._binary(b)
        self.schema = 2
        self.weights = []
        pos += 4

        def line():
            nonlocal pos
            e = b.index(b"\n", pos); s = b[pos:e].decode(); pos = e + 1
            return s

        def u32v():
            nonlocal pos
            (v,) = struct.unpack_from("<I", b, pos); pos += 4
            return v

        def small():
            nonlocal pos
            v = b[pos]; pos += 1
            return u32v() if v == 255 else v

        for _ in range(u32v()):
            nm = line(); el = line(); tl = u32v()
            self.names.append(nm); self.efflen.setdefault(nm, float(el)); self.truelen.setdefault(nm, tl)
        for _ in range(u32v()):
            g = line(); c = u32v()
            self.genes.setdefault(g, [line() for _ in range(c)])
        for _ in range(u32v()):
            c = u32v()
            self.identical.append([line() for _ in range(c)])
        while pos < len(b):
            nm = line()
            if nm == "":
                small(); line(); small()
            c = u32v()
            self.records.append([self.names[u32v()] for _ in range(c)])
            self.weights.append(np.frombuffer(b, "<f4", c, pos).astype(np.float32)); pos += 4 * c


def by_length_rows(hf, cl):
    """The per-fragment rows of a weighted file as the host program hands them to the GPU (the loader's
    LAYOUT_PER_FRAGMENT_BY_LENGTH with first-appearance columns): one row per record, sets ordered by size and
    then by their member columns lexicographically, records in file order inside a set.  A record's weights follow
    its set's (ascending) columns; a transcript repeated in the record adds its weight, in fp32, to its first
    occurrence.  cl: orc.build_classes(hf).  Returns (row_ptr, col, w)."""
    sid_index = cl["sid_index"]
    rows = [tuple(int(c) for c in cl["col"][cl["row_ptr"][i]:cl["row_ptr"][i + 1]]) for i in range(cl["m"])]
    set_of = {r: i for i, r in enumerate(rows)}
    rec_set, rec_w = [], []
    for rec, wts in zip(hf.records, hf.weights):
        acc = {}
        for name, wt in zip(rec, wts):
            c = sid_index[name]
            acc[c] = np.float32(acc[c] + wt) if c in acc else np.float32(wt)
        cols = tuple(sorted(acc))
        rec_set.append(set_of[cols])
        rec_w.append([acc[c] for c in cols])
    rank = np.empty(cl["m"], np.int64)
    rank[sorted(range(cl["m"]), key=lambda i: (len(rows[i]), rows[i]))] = np.arange(cl["m"])
    order = np.argsort(rank[np.array(rec_set, np.int64)], kind="stable")
    sizes = np.array([len(rows[rec_set[r]]) for r in order], np.int64)
    row_ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    col = np.array([c for r in order for c in rows[rec_set[r]]], np.int32)
    w = np.array([x for r in order for x in rec_w[r]], np.float32)
    return row_ptr, col, w


def run(path, **kw):
    """tables.run (the reference's main() restated, same keyword arguments and result) for a weighted file.  The
    tables, .k, .M, unique hits and group sums are computed from the distinct sets exactly as tables.run does; the
    chain — initial mu, EM and the Philox Gibbs replay — runs on the weighted per-fragment rows of by_length_rows,
    which is what the host program runs on the GPU.  tables.run reads the file with orc.HitsFile and builds its
    one orc.Problem from the sets: both are substituted for the duration of the call."""
    hf = HitsFile(path)
    assert hf.schema == 2, "not a weighted hits file"
    cl = orc.build_classes(hf)
    rp, col, w = by_length_rows(hf, cl)

    class WeightedProblem(_Problem):
        def __init__(self, row_ptr, col_, k, length, alpha=0.1, beta=0.1):
            super().__init__(rp, col, None, length, weight=w, alpha=alpha, beta=beta)
            self.sets = _Problem(row_ptr, col_, k, length, alpha=alpha, beta=beta)

        def init_mu(self):
            mu0, _, cs = super().init_mu()      # the per-fragment rows, weights ignored: what the device computes
            _, uh, _ = self.sets.init_mu()      # unique hits of the sets
            return mu0, uh, cs

    with mock.patch.object(orc, "HitsFile", lambda p: hf), mock.patch.object(orc, "Problem", WeightedProblem):
        return tables.run(path, **kw)
