"""The TMEM-assisted SSV tiles (J = 32 tiles whose first 16 words per lane are read from tensor memory, kernels_msv.cu)
against the int8-chunk tiles they replace (CKM_SSV_TMEM=0, read when a model database is loaded).  Both sweep the same int16
recurrence, so the SSV candidates, the pairs resolved in the SSV epilogue, the MSV pass set and every hit must be identical."""
import numpy as np
import pytest

from tools import synth
from conftest import CPR_HMM

pytestmark = pytest.mark.gpu


def load_both(engine, path, monkeypatch):
    out = {}
    for tm in ('0', '1'):
        monkeypatch.setenv('CKM_SSV_TMEM', tm)
        out[tm] = engine.load_models(path)
    monkeypatch.delenv('CKM_SSV_TMEM')
    return out


def same_hits(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f]), f


def stage1(engine, models, db):
    xj = engine.msv_scores(models, db)
    st = engine.stats()
    return xj, (st.n_ssv_cand, st.n_past_msv, st.n_msv_exact)


def compare(engine, ms, b, resolve, monkeypatch, min_pass):
    monkeypatch.setenv('CKM_SSV_RESOLVE', resolve)
    db = engine.seqdb(b.residues, b.offsets)
    xj0, c0 = stage1(engine, ms['0'], db)
    xj1, c1 = stage1(engine, ms['1'], db)
    assert c0 == c1
    assert np.array_equal(xj0, xj1)
    assert c1[1] >= min_pass
    h0 = engine.search(ms['0'], db)
    h1 = engine.search(ms['1'], db)
    same_hits(h0, h1)
    db.close()
    return h1


@pytest.mark.parametrize('resolve', ['1', '0'])
def test_tmem_tiles_cpr43_bench_size_bin(engine, resolve, monkeypatch):
    """One bench-size bin (2,900 ORFs) against the 43 CPR models, with and without the resolving epilogue."""
    ms = load_both(engine, CPR_HMM, monkeypatch)
    hm = synth.read_hmms(CPR_HMM)
    b = synth.make_bin('t0', hm, seed=21, n_orfs=2900, copies=(0, 1, 1, 1, 2))
    h = compare(engine, ms, b, resolve, monkeypatch, min_pass=100)
    assert len(h) > 20
    for m in ms.values():
        m.close()


def test_tmem_tiles_replica_db(engine, monkeypatch):
    """The benchmark's 5,000-model replica database (one tile group per J = 32 tile, 30 tiles per SM wave) on a 600-ORF slice
    of a bench bin, and a stable workspace footprint over repeated searches."""
    import bench
    ms = load_both(engine, bench.model_db(5000), monkeypatch)
    hm = synth.read_hmms(CPR_HMM)
    b = synth.make_bin('t1', hm, seed=22, n_orfs=600, copies=(0, 1, 1, 1, 2))
    compare(engine, ms, b, '1', monkeypatch, min_pass=1000)
    db = engine.seqdb(b.residues, b.offsets)
    first = engine.search(ms['1'], db)
    ws = engine.workspace_bytes()
    for _ in range(2):
        same_hits(first, engine.search(ms['1'], db))
        assert engine.workspace_bytes() == ws
    db.close()
    for m in ms.values():
        m.close()


def test_tmem_tiles_next_to_chained_models(engine, tmp_path, monkeypatch):
    """Models longer than a J = 32 tile (2,500 positions: a chain of J = 16 tiles, outside the TMEM path) next to J = 32 ones
    in the same database, including a subset search."""
    p = str(tmp_path / 'long.hmm')
    lm = synth.make_model_db(p, CPR_HMM, [40, 300, 700, 1100, 2047, 2048, 2500, 3000], seed=7)
    ms = load_both(engine, p, monkeypatch)
    b = synth.make_bin('t2', lm, seed=23, n_orfs=120, copies=(1,), max_len=3500, split_prob=0.0)
    compare(engine, ms, b, '1', monkeypatch, min_pass=5)
    db = engine.seqdb(b.residues, b.offsets)
    xa = engine.msv_scores(ms['0'], db, [6, 1, 4])
    xb = engine.msv_scores(ms['1'], db, [6, 1, 4])
    assert np.array_equal(xa, xb)
    db.close()
    for m in ms.values():
        m.close()
