"""Thin Python object layer over the C ABI: Engine / Models / SeqDb.  All computation happens in libckm.so."""
import ctypes as C
import numpy as np

from . import _lib
from ._lib import check, Hit, Stats, ModelInfo

ALPHABET = "ACDEFGHIKLMNPQRSTVWY-BJZOUX*~"

HIT_DTYPE = np.dtype([(n, {C.c_int32: np.int32, C.c_float: np.float32, C.c_double: np.float64}[t]) for n, t in Hit._fields_],
                     align=True)
assert HIT_DTYPE.itemsize == C.sizeof(Hit)


def digitize(text):
    """ASCII protein text -> uint8 codes (unknown symbols become X), via the library."""
    b = text.encode() if isinstance(text, str) else bytes(text)
    out = np.empty(len(b), dtype=np.uint8)
    check(_lib.lib().ckm_digitize(b, len(b), out.ctypes.data))
    return out


class Models:
    def __init__(self, engine, path):
        self.engine = engine
        self._h = C.c_void_p()
        check(_lib.lib().ckm_models_load(engine._h, path.encode(), C.byref(self._h)))
        self.path = path
        self.n = _lib.lib().ckm_models_count(self._h)
        self._info = None

    def info(self):
        if self._info is None:
            out = []
            for i in range(self.n):
                mi = ModelInfo()
                check(_lib.lib().ckm_models_info(self._h, i, C.byref(mi)))
                out.append(mi)
            self._info = out
        return self._info

    def find(self, key):
        return _lib.lib().ckm_models_find(self._h, key.encode())

    def select(self, keys):
        arr = (C.c_char_p * len(keys))(*[k.encode() for k in keys])
        idx = np.empty(max(self.n, 1), dtype=np.int32)
        n = C.c_int()
        check(_lib.lib().ckm_models_select(self._h, arr, len(keys), idx.ctypes.data, C.byref(n)))
        return idx[:n.value].copy()

    def write(self, idx, path):
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        check(_lib.lib().ckm_models_write(self._h, idx.ctypes.data, len(idx), path.encode()))

    def close(self):
        if self._h:
            _lib.lib().ckm_models_free(self._h)
            self._h = C.c_void_p()


class SeqDb:
    def __init__(self, engine, residues, offsets, bin_of_seq=None, nbins=1):
        self.engine = engine
        self.residues = np.ascontiguousarray(residues, dtype=np.uint8)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.nseq = len(self.offsets) - 1
        self.nbins = int(nbins)
        self.bin_of_seq = None if bin_of_seq is None else np.ascontiguousarray(bin_of_seq, dtype=np.int32)
        self._h = C.c_void_p()
        check(_lib.lib().ckm_seqdb_create(engine._h, self.residues.ctypes.data, self.offsets.ctypes.data, self.nseq,
                                          None if self.bin_of_seq is None else self.bin_of_seq.ctypes.data,
                                          self.nbins, C.byref(self._h)))

    def close(self):
        if self._h:
            _lib.lib().ckm_seqdb_free(self._h)
            self._h = C.c_void_p()


class Engine:
    """One engine per process per GPU (a CUDA context cannot cross fork())."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        check(_lib.lib().ckm_init(int(device), C.byref(self._h)))
        self.device = int(device)

    def device_name(self):
        buf = C.create_string_buffer(256)
        check(_lib.lib().ckm_device_name(self._h, buf, 256))
        return buf.value.decode()

    def load_models(self, path):
        return Models(self, path)

    def seqdb(self, residues, offsets, bin_of_seq=None, nbins=1):
        return SeqDb(self, residues, offsets, bin_of_seq, nbins)

    def stats(self):
        s = Stats()
        check(_lib.lib().ckm_last_stats(self._h, C.byref(s)))
        return s

    def workspace_bytes(self):
        """Device bytes the engine keeps between calls as workspaces (ckm_workspace_bytes)."""
        n = C.c_int64()
        check(_lib.lib().ckm_workspace_bytes(self._h, C.byref(n)))
        return n.value

    def msv_scores(self, models, db, model_idx=None):
        """Dense [nmodels, nseq] int32: exact MSV xJ byte for SSV candidates (256 = overflow), -1 otherwise."""
        nm = models.n if model_idx is None else len(model_idx)
        out = np.empty((nm, db.nseq), dtype=np.int32)
        mi = None if model_idx is None else np.ascontiguousarray(model_idx, dtype=np.int32)
        check(_lib.lib().ckm_msv_scores(self._h, models._h, None if mi is None else mi.ctypes.data, nm, db._h,
                                        out.ctypes.data))
        return out

    def viterbi_scores(self, models, db, model_idx=None, int32_only=False, chunked_only=False):
        """Dense [nmodels, nseq] float32 ViterbiFilter scores of every pair (packed int16x2 kernel + int32 redo list, or the
        int32 kernels alone)."""
        nm = models.n if model_idx is None else len(model_idx)
        out = np.empty((nm, db.nseq), dtype=np.float32)
        mi = None if model_idx is None else np.ascontiguousarray(model_idx, dtype=np.int32)
        check(_lib.lib().ckm_viterbi_scores(self._h, models._h, None if mi is None else mi.ctypes.data, nm, db._h,
                                            2 if chunked_only else (1 if int32_only else 0), out.ctypes.data))
        return out

    def filter_scores(self, models, db, model_idx=None):
        """Dense [nmodels, nseq] arrays: bias-filter null score, Viterbi and Forward filter scores (NaN where a stage
        was not reached) and pass flags (bit0 MSV, bit1 bias, bit2 Viterbi, bit3 Forward)."""
        nm = models.n if model_idx is None else len(model_idx)
        fs = np.empty((nm, db.nseq), dtype=np.float32)
        vs = np.empty((nm, db.nseq), dtype=np.float32)
        fw = np.empty((nm, db.nseq), dtype=np.float32)
        ps = np.empty((nm, db.nseq), dtype=np.uint8)
        mi = None if model_idx is None else np.ascontiguousarray(model_idx, dtype=np.int32)
        check(_lib.lib().ckm_filter_scores(self._h, models._h, None if mi is None else mi.ctypes.data, nm, db._h,
                                           fs.ctypes.data, vs.ctypes.data, fw.ctypes.data, ps.ctypes.data))
        return fs, vs, fw, ps

    def search(self, models, db, model_idx=None, E=0.1, domE=0.1, bin_model_offsets=None):
        """Returns a numpy structured array of ckm_hit rows (domtblout rows)."""
        hits = C.POINTER(Hit)()
        n = C.c_int64()
        mi = None if model_idx is None else np.ascontiguousarray(model_idx, dtype=np.int32)
        if bin_model_offsets is None:
            nm = models.n if mi is None else len(mi)
            check(_lib.lib().ckm_search(self._h, models._h, None if mi is None else mi.ctypes.data, nm, db._h, E, domE,
                                        C.byref(hits), C.byref(n)))
        else:
            bo = np.ascontiguousarray(bin_model_offsets, dtype=np.int64)
            check(_lib.lib().ckm_search_per_bin(self._h, models._h, mi.ctypes.data, bo.ctypes.data, db._h, E, domE,
                                                C.byref(hits), C.byref(n)))
        if n.value == 0:
            arr = np.zeros(0, dtype=HIT_DTYPE)
        else:
            buf = (C.c_char * (n.value * C.sizeof(Hit))).from_address(C.addressof(hits.contents))
            arr = np.frombuffer(buf, dtype=HIT_DTYPE).copy()
        _lib.lib().ckm_hits_free(hits)
        return arr

    def align(self, models, db, model=0):
        """Optimal-accuracy alignment of every sequence of `db` to one model (ckm_align): per-residue states (+k match,
        -k insert, 0 flank) over the unpadded residue stream, and the optimal-accuracy score of every sequence."""
        state = np.zeros(len(db.residues), dtype=np.int32)
        oasc = np.zeros(db.nseq, dtype=np.float32)
        check(_lib.lib().ckm_align(self._h, models._h, int(model), db._h, state.ctypes.data, oasc.ctypes.data))
        return state, oasc

    def scaffold_stats(self, data, starts, lens):
        """Base counts and contigs of scaffolds laid out as `seqio.scan_nt_fasta` returns them (ckm_scaffold_stats).
        Returns stats (n x 8 int64: A C G T 'N' 'n' contigs contig-bases), the scaffold index and length of every contig
        (no particular order), and the scan kernel's duration in ms."""
        n = len(lens)
        stats = np.zeros((n, 8), dtype=np.int64)
        data = np.ascontiguousarray(data, dtype=np.uint8)
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        lens = np.ascontiguousarray(lens, dtype=np.int64)
        cap = n + int(lens.sum()) // 2048 + 1024
        while True:
            cscaf = np.empty(cap, dtype=np.uint32)
            clen = np.empty(cap, dtype=np.uint32)
            found, ms = C.c_int64(), C.c_float()
            rc = _lib.lib().ckm_scaffold_stats(self._h, data.ctypes.data, data.size, starts.ctypes.data, lens.ctypes.data, n,
                                               stats.ctypes.data, cscaf.ctypes.data, clen.ctypes.data, cap, C.byref(found), C.byref(ms))
            if rc == 8 and found.value > cap:          # CKM_ECAPACITY: the count needed came back
                cap = found.value
                continue
            check(rc)
            return stats, cscaf[:found.value].astype(np.int64), clen[:found.value].astype(np.int64), float(ms.value)

    def close(self):
        if self._h:
            _lib.lib().ckm_destroy(self._h)
            self._h = C.c_void_p()
