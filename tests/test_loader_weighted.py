"""Weighted (schema 2) hits files on the CPU: the distinct sets a per-fragment load returns next to its
rows, the CPU oracle's construction of the rows the host program hands to the GPU, and the oracle's
reader of schema 2."""
import copy

import numpy as np
import pytest

from mmseq_b200 import hostlib, synth
from oracle import oracle as orc
from tests import weighted_oracle

PER_FRAGMENT = (hostlib.LAYOUT_PER_FRAGMENT, hostlib.LAYOUT_PER_FRAGMENT_SORTED, hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)


def _with_repeats(s, every=7):
    """A copy of the sample in which every `every`-th record lists its first transcript once more (with its own weight)."""
    r = copy.copy(s)
    tid, w, ptr = [], [], [0]
    rng = np.random.default_rng(3)
    for f in range(s.N):
        b, e = int(s.frag_ptr[f]), int(s.frag_ptr[f + 1])
        t = list(s.frag_tid[b:e]); x = list(s.frag_w[b:e])
        if f % every == 3:
            t.append(t[0]); x.append(np.float32(rng.uniform(0.1, 2.0)))
        tid += t; w += x; ptr.append(len(tid))
    r.frag_ptr = np.array(ptr, np.int64); r.frag_tid = np.array(tid, np.int32); r.frag_w = np.array(w, np.float32)
    return r


@pytest.fixture(scope="module")
def weighted_sample():
    return _with_repeats(synth.Synth(41, 200, 6000, weights=True))


def _same_sets(p, c):
    """The set view of per-fragment load p equals collapsed load c field by field."""
    assert p.k is None and p.m == p.N == c.N
    assert (p.n, p.N, p.n_classes) == (c.n, c.N, c.m)
    assert np.array_equal(p.set_ptr, c.row_ptr) and np.array_equal(p.set_col, c.col) and np.array_equal(p.set_k, c.k)
    assert np.array_equal(p.hdr2col, c.hdr2col) and np.array_equal(p.col2hdr, c.col2hdr)
    assert np.array_equal(p.doublehits, c.doublehits)


@pytest.mark.parametrize("parallel", [False, True])
def test_set_view_of_weighted_file_equals_collapsed_load(tmp_path, monkeypatch, weighted_sample, parallel):
    """(parallel: the all-threads loader path, which small files do not take by default.)"""
    if parallel:
        monkeypatch.setenv("MMQ_LOADER_PAR_MIN_BYTES", "0")
    s = weighted_sample
    w2, w1 = str(tmp_path / "w2.hits"), str(tmp_path / "w1.hits")
    synth.write_hits_binary(s, w2, weights=s.frag_w)
    synth.write_hits_binary(s, w1)
    c = hostlib.load_hits(w1)
    assert c.set_ptr is None and c.doublehits.sum() > 0                 # collapsed: the rows are the sets; repeats present
    for lay in PER_FRAGMENT:
        p = hostlib.load_hits(w2, layout=lay)
        assert p.schema == 2
        _same_sets(p, c)
        _same_sets(hostlib.load_hits(w1, layout=lay), c)               # unweighted per-fragment loads too
    for lay in PER_FRAGMENT:                                            # and the in-memory records
        cm = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid)
        _same_sets(hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, frag_w=s.frag_w, layout=lay), cm)
        _same_sets(hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=lay), cm)
    with pytest.raises(RuntimeError, match="per-fragment layout"):
        hostlib.load_hits(w2)                                           # still refused collapsed


def test_set_view_in_header_order_columns(tmp_path, weighted_sample):
    s = weighted_sample
    p = str(tmp_path / "w2.hits")
    synth.write_hits_binary(s, p, weights=s.frag_w)
    lay = hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH | hostlib.LAYOUT_HEADER_ORDER_COLUMNS
    c = hostlib.from_records(s.T, s.efflen, s.frag_ptr, s.frag_tid, layout=hostlib.LAYOUT_HEADER_ORDER_COLUMNS)
    _same_sets(hostlib.load_hits(p, layout=lay), c)


@pytest.mark.parametrize("parallel", [False, True])
def test_oracle_by_length_rows_equal_the_loader(tmp_path, monkeypatch, weighted_sample, parallel):
    """weighted_oracle.by_length_rows (what the oracle runs the weighted chain on) is the loader's by-length layout exactly:
    row order, columns and weights, repeats summed into the first occurrence."""
    if parallel:
        monkeypatch.setenv("MMQ_LOADER_PAR_MIN_BYTES", "0")
    s = weighted_sample
    path = str(tmp_path / "w2.hits")
    synth.write_hits_binary(s, path, weights=s.frag_w)
    h = hostlib.load_hits(path, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH)
    hf = weighted_oracle.HitsFile(path)
    rp, col, w = weighted_oracle.by_length_rows(hf, orc.build_classes(hf))
    assert np.array_equal(rp, h.row_ptr) and np.array_equal(col, h.col)
    assert w.dtype == np.float32 and np.array_equal(w.view(np.uint32), h.w.view(np.uint32))
    assert h.first_zero_weight_record == -1


def test_oracle_reads_schema2(tmp_path, weighted_sample):
    s = weighted_sample
    path = str(tmp_path / "w2.hits")
    synth.write_hits_binary(s, path, weights=s.frag_w)
    hf = weighted_oracle.HitsFile(path)
    assert hf.schema == 2 and hf.names == [s.transcript_name(t) for t in range(s.T)]
    assert len(hf.records) == len(hf.weights) == s.N
    for f in (0, 3, 1234, s.N - 1):
        b, e = int(s.frag_ptr[f]), int(s.frag_ptr[f + 1])
        assert hf.records[f] == [s.transcript_name(int(t)) for t in s.frag_tid[b:e]]
        assert np.array_equal(hf.weights[f], s.frag_w[b:e])
    one = str(tmp_path / "w1.hits")
    synth.write_hits_binary(s, one)
    h1 = weighted_oracle.HitsFile(one)
    assert h1.schema == 1 and h1.weights is None and h1.records == hf.records


@pytest.mark.parametrize("parallel", [False, True])
def test_first_zero_weight_record(tmp_path, monkeypatch, weighted_sample, parallel):
    """A record whose weights are all zero is reported by position (0-based); a zero weight next to a positive one is not."""
    if parallel:
        monkeypatch.setenv("MMQ_LOADER_PAR_MIN_BYTES", "0")
    s = weighted_sample
    w = s.frag_w.copy()
    multi = [f for f in range(s.N) if s.frag_ptr[f + 1] - s.frag_ptr[f] >= 2]
    w[s.frag_ptr[multi[0]]] = 0.0                                       # one zero among positive weights: fine
    path = str(tmp_path / "z0.hits")
    synth.write_hits_binary(s, path, weights=w)
    assert hostlib.load_hits(path, layout=hostlib.LAYOUT_PER_FRAGMENT_BY_LENGTH).first_zero_weight_record == -1
    for f in (4000, 1711):
        w[s.frag_ptr[f]:s.frag_ptr[f + 1]] = 0.0
    path = str(tmp_path / "z.hits")
    synth.write_hits_binary(s, path, weights=w)
    for lay in PER_FRAGMENT:
        assert hostlib.load_hits(path, layout=lay).first_zero_weight_record == 1711
