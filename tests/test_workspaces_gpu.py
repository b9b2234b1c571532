"""The engine's device workspaces (ckm_workspace_bytes): one buffer per role, so what an engine keeps follows from the inputs
it has seen, not from the order of its calls.  Every test makes and closes its own engines, one at a time (the envelope
scratch budget is shared by the live engines)."""
import numpy as np
import pytest

from tools import synth
from conftest import CPR_HMM
from checkm_b200.engine import Engine

pytestmark = pytest.mark.gpu


def two_bins(hm):
    b1 = synth.make_bin('wa', hm, seed=61, n_orfs=150, max_len=900, tandem_prob=0.2)
    b2 = synth.make_bin('wb', hm, seed=62, n_orfs=200, max_len=900, tandem_prob=0.2)
    res = np.concatenate([b1.residues, b2.residues])
    off = np.concatenate([b1.offsets, b2.offsets[1:] + b1.offsets[-1]])
    binof = np.concatenate([np.zeros(b1.nseq, np.int32), np.ones(b2.nseq, np.int32)])
    return res, off, binof


def per_bin_subsets():
    """A quarter of the models per bin, different ones in each bin: bin_model_offsets, model_idx."""
    idx = [0, 5, 9, 13, 17, 21, 25, 29, 33, 37, 41, 2, 6, 10, 14, 18, 22, 26, 30, 34, 38, 42]
    return np.array([0, 11, 22], np.int64), np.array(idx, np.int32)


def scaffolds(seed=5, n=40):
    rng = np.random.default_rng(seed)
    seqs = []
    for _ in range(n):
        s = rng.choice(np.frombuffer(b'ACGTacgt', np.uint8), size=int(rng.integers(200, 20000)))
        for _ in range(int(rng.integers(0, 4))):
            at = int(rng.integers(0, len(s)))
            s[at:at + int(rng.integers(1, 40))] = ord('N')
        seqs.append(s)
    lens = np.array([len(s) for s in seqs], np.int64)
    padded = (lens + 63) // 64 * 64
    starts = np.concatenate([[0], np.cumsum(padded)[:-1]]).astype(np.int64)
    data = np.zeros(int(padded.sum()) + 64, np.uint8)
    for s, at in zip(seqs, starts):
        data[at:at + len(s)] = s
    return data, starts, lens


def same_hits(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f]), f


CALLS = ['search', 'search_per_bin', 'filter_scores', 'viterbi_scores', 'msv_scores', 'align', 'scaffold_stats']


@pytest.mark.parametrize('call', CALLS)
def test_second_identical_call_allocates_nothing(call):
    hm = synth.read_hmms(CPR_HMM)
    res, off, binof = two_bins(hm)
    eng = Engine(0)
    models = eng.load_models(CPR_HMM)
    db = eng.seqdb(res, off, binof, 2)
    bo, idx = per_bin_subsets()
    run = {
        'search': lambda: eng.search(models, db),
        'search_per_bin': lambda: eng.search(models, db, model_idx=idx, bin_model_offsets=bo),
        'filter_scores': lambda: eng.filter_scores(models, db, model_idx=[3, 1, 40]),
        'viterbi_scores': lambda: eng.viterbi_scores(models, db, model_idx=[3, 1, 40]),
        'msv_scores': lambda: eng.msv_scores(models, db),
        'align': lambda: eng.align(models, db, 7),
        'scaffold_stats': lambda: eng.scaffold_stats(*scaffolds()),
    }[call]
    try:
        assert eng.workspace_bytes() == 0
        run()
        first = eng.workspace_bytes()
        run()
        assert first > 0 and eng.workspace_bytes() == first
    finally:
        db.close()
        models.close()
        eng.close()


def test_footprint_and_hits_do_not_depend_on_call_order():
    """A = all 43 models over two bins, B = per-bin subsets of them.  Engine X runs A then B, engine Y B then A: the same
    workspaces, and the same hit tables as a fresh engine gives (no result depends on a stale, larger buffer).  B's pairs,
    regions and envelopes are about a quarter of A's, so each of A's workspaces is either as large as B's or more than the 25%
    growth slack above it: which call came first cannot decide its size."""
    hm = synth.read_hmms(CPR_HMM)
    res, off, binof = two_bins(hm)
    bo, idx = per_bin_subsets()

    def session(order, extra_round=False):
        eng = Engine(0)
        models = eng.load_models(CPR_HMM)
        db = eng.seqdb(res, off, binof, 2)
        run = {'A': lambda: eng.search(models, db), 'B': lambda: eng.search(models, db, model_idx=idx, bin_model_offsets=bo)}
        try:
            hits = {k: run[k]() for k in order}
            footprint = eng.workspace_bytes()
            if extra_round:
                again = {k: run[k]() for k in 'AB'}
                assert eng.workspace_bytes() == footprint
                for k in 'AB':
                    same_hits(again[k], hits[k])
            return hits, footprint
        finally:
            db.close()
            models.close()
            eng.close()

    hx, fx = session('AB', extra_round=True)
    hy, fy = session('BA')
    fresh_a, _ = session('A')
    fresh_b, _ = session('B')
    print('workspace bytes: A then B %d, B then A %d' % (fx, fy))
    assert fx == fy
    assert len(fresh_a['A']) > len(fresh_b['B']) > 0
    for k, fresh in (('A', fresh_a['A']), ('B', fresh_b['B'])):
        same_hits(hx[k], fresh)
        same_hits(hy[k], fresh)


def test_repeated_domain_phase_reuses_its_workspaces():
    """The repeat protein of test_region_with_more_domains_than_slots: its domain phase runs more than once per search, and a
    second search of it keeps the footprint of the first."""
    hm = synth.read_hmms(CPR_HMM)
    fam = min(hm, key=lambda h: h.M)
    rng = np.random.default_rng(103)
    repeats = np.concatenate([synth.emit_homolog(fam, rng, k_from=int(rng.integers(20, 25)), k_to=int(rng.integers(45, 50)), sharpen=0.6)
                              for _ in range(150)])
    b = synth.make_bin('r', hm, seed=78, n_orfs=120, max_len=900)
    seqs = [b.seq(i) for i in range(15)] + [repeats] + [b.seq(i) for i in range(15, 30)]
    residues = np.concatenate(seqs)
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.int64)
    eng = Engine(0)
    models = eng.load_models(CPR_HMM)
    db = eng.seqdb(residues, offsets)
    try:
        first = eng.search(models, db)
        assert eng.stats().n_queue_retries >= 1
        footprint = eng.workspace_bytes()
        second = eng.search(models, db)
        assert eng.stats().n_queue_retries >= 1
        assert eng.workspace_bytes() == footprint
        same_hits(first, second)
    finally:
        db.close()
        models.close()
        eng.close()
