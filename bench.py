#!/usr/bin/env python
"""bench.py -- genomes/hour of the marker-gene search hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Workloads (config["workload"]):
  --config 3 (default; BASELINE.json configs[2], the configuration the metric is quoted on): synthetic 3 Mb bins (2,900 ORFs,
      ~0.9 M residues, SURVEY.md 8d) x a 5,000-model HMM database (the 43 real, HMMER-calibrated CPR marker HMMs x 116 replicas
      under distinct accessions, sum M = 1.04 M).  One step = one batch of `bins_per_step` bins per rank; weak scaling.
  --config 2 (configs[1]): 100 synthetic 2 Mb bins (1,900 ORFs) x cpr_43_markers.hmm on one GPU.  One step = all 100 bins.
  --config 4 (configs[3] stand-in): a FIXED set of 512 bins with log-normal genome sizes (median 3.2 Mb, 0.6-10 Mb) x the
      5,000-model database, partitioned over the ranks by longest-processing-time (checkm_b200.sharding.partition_bins);
      one step = the whole set, the time is that of the last rank; QA rows gathered with ckm_allgather_qa.  Strong scaling.

One "step" = the whole hot path (SSV/MSV -> bias -> Viterbi -> Forward -> domain definition -> hit table -> marker-set
reduction -> QA rows) over the step's bins.

value : inputs (digitised ORFs, models) resident in HBM before the timed region.
e2e   : the same through the C ABI with HOST buffers -- H2D of the step's residues and D2H of its hit table and QA rows
        inside the timed region.
plugin: (config 3, N = 1) the drop-in path itself: FASTA files on disk -> MarkerGeneFinder.find -> domtblout + side-car
        files -> ResultsParser.analyseResults -> printSummary, per step, everything inside the timed region.
--impl reference : the CPU arm.  `hmmsearch` itself when it is on PATH (kind "hmmer"); otherwise the CPU restatement of its
        pipeline (oracle/, SSE2 striped MSV/Viterbi filters, every host core; kind "port") followed by the REFERENCE's own
        ResultsParser (oracle/_ref, byte-compiled from /root/reference) -- one full bin x all models per step, no scaling.
--dump-outputs DIR : after the timed steps, the hit table and QA rows of the last timed step, one .npy per field
        (dump_outputs).  The workload is generated from fixed seeds, so two builds can be compared output for output.
"""
import argparse
import ctypes as C
import io
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
CPR = os.path.join(ROOT, 'tests', 'golden', 'cpr_43_markers.hmm')

N_MODELS = 5000
BINS_PER_STEP = 32
CFG = {2: dict(orfs=1900, n_models=43, total_bins=100), 3: dict(orfs=2900, n_models=N_MODELS, total_bins=None),
       4: dict(orfs=None, n_models=N_MODELS, total_bins=512)}


def rank_info():
    return int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))


def diverse_model_db(n_models=N_MODELS):
    """A second 5,000-model database for the realism check (`--db diverse`): model lengths log-normal around the Pfam/TIGRFAM
    mean (30-1,500 positions, tools/synth.perturbed_model_lengths), rows stitched from windows of the real models, STATS from
    the least-squares fit of the 43 calibrated ones.  Not the headline: stitched models are not calibrated by HMMER, so the
    cascade's pass rates are only approximately the nominal ones."""
    from tools import synth
    path = '/tmp/ckm_bench_db_diverse_%d.hmm' % n_models
    if not os.path.exists(path):
        lengths = synth.perturbed_model_lengths(np.random.default_rng(11), n_models)
        synth.make_model_db_fast(path + '.tmp', CPR, lengths, seed=12)
        os.replace(path + '.tmp', path)
    return path


def model_db(n_models=N_MODELS):
    """HMM database file.  43 models: the reference's fixture itself.  5,000 models: written once per box under /tmp -- every
    one of the 43 real, HMMER-calibrated CPR marker HMMs repeated under distinct names/accessions (sum M = 1.04 M).  Replicas
    are separate models to the engine (own tiles, own tables, own hits); real models keep the STATS lines -- and with them
    the filter pass rates of the cascade (2% / 0.1% / 1e-5) -- those of a real search."""
    if n_models == 43:
        return CPR
    path = '/tmp/ckm_bench_db_%d.hmm' % n_models
    if not os.path.exists(path):
        recs = [r + '//\n' for r in open(CPR).read().split('//\n') if r.strip()]
        tmp = path + '.%d.tmp' % os.getpid()
        with open(tmp, 'w') as out:
            n = rep = 0
            while n < n_models:
                for r in recs:
                    if n >= n_models:
                        break
                    if rep == 0:
                        out.write(r)
                    else:
                        lines = r.split('\n')
                        for i, ln in enumerate(lines[:6]):
                            if ln.startswith('NAME '):
                                lines[i] = ln + '_r%d' % rep
                            elif ln.startswith('ACC '):
                                acc = ln.split()[1]
                                lines[i] = 'ACC   %s' % ((acc.split('.')[0] + 'r%d.' % rep + acc.split('.')[1]) if '.' in acc else acc + 'r%d' % rep)
                        out.write('\n'.join(lines))
                    n += 1
                rep += 1
        os.replace(tmp, path)
    return path


class Batch(object):
    """A set of bins searched together: concatenated residues, CSR offsets, bin of every ORF, names."""

    def __init__(self, bins):
        self.bins = bins
        self.res = np.concatenate([b.residues for b in bins])
        lens = np.concatenate([np.diff(b.offsets) for b in bins])
        self.off = np.zeros(len(lens) + 1, dtype=np.int64)
        self.off[1:] = np.cumsum(lens)
        self.binof = np.repeat(np.arange(len(bins), dtype=np.int32), [b.nseq for b in bins])
        self.db = None                  # resident copies, one per pipeline slot
        self.meta = None


def make_bins(n, seed0, orfs):
    from tools import synth
    hm = synth.read_hmms(CPR)
    return [synth.make_bin('bin%d' % (seed0 + i), hm, seed=seed0 + i, n_orfs=orfs, copies=(0, 1, 1, 1, 2)) for i in range(n)]


def heterogeneous_bins(total, seed=4):
    """The fixed bin set of config 4: genome sizes log-normal (median 3.2 Mb, clipped to 0.6-10 Mb; ~1 ORF per kb), ORFs taken
    from a pool of 24 generated 3 Mb bins (generating 512 genomes residue by residue would take longer than the benchmark)."""
    from tools import synth
    pool = make_bins(24, 7000, 2900)
    rng = np.random.default_rng(seed)
    sizes = np.clip(rng.lognormal(np.log(3.2e6), 0.55, size=total), 0.6e6, 10e6)
    out = []
    for j, sz in enumerate(sizes):
        n = int(sz / 1000.0 * 0.93)
        take, k = [], int(rng.integers(len(pool)))
        while n > 0:
            p = pool[k % len(pool)]
            m = min(n, p.nseq)
            take.append((p, m))
            n -= m
            k += 1
        res = np.concatenate([p.residues[:p.offsets[m]] for p, m in take])
        lens = np.concatenate([np.diff(p.offsets[:m + 1]) for p, m in take])
        off = np.zeros(len(lens) + 1, dtype=np.int64)
        off[1:] = np.cumsum(lens)
        names, descs = [], []
        for t, (p, m) in enumerate(take):
            names += ['s%d%s' % (t, nm) for nm in p.names[:m]]
            descs += p.descs[:m]
        out.append(synth.Bin('het%04d' % j, res, off, names, descs, []))
    return out


class ClockSampler(threading.Thread):
    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p)), 'measured'
    return {"hbm_gbs": 6650.0}, 'fallback'


def ssv_traffic():
    """DRAM bytes per SSV launch from the committed `ncu --set full` capture, or None."""
    for name in ('r2_ssv32_traffic.json', 'r1_ssv32_traffic.json'):
        try:
            return json.load(open(os.path.join(ROOT, 'profiles', name)))
        except Exception:
            continue
    return None


def total_model_positions(db_path):
    tot = 0
    with open(db_path) as f:
        for line in f:
            if line.startswith('LENG'):
                tot += int(line.split()[1])
    return tot


DUMP_BYTES = 60 * 1000 * 1000                 # array data; the .npy headers stay well inside 64 MB


def dump_outputs(out_dir, tables, prefix=''):
    """Writes every field of the structured arrays `tables` ({name: array}) as out_dir/<prefix><name>_<field>.npy: float32
    fields as float32, all others as float64, with the row indices as <name>_row.npy.  Smallest table first, each takes
    at most an equal share of what is left of DUMP_BYTES; a table with more rows than that is written as a fixed, seeded
    sample of its rows, in row order."""
    os.makedirs(out_dir, exist_ok=True)
    kinds = {name: {f: (np.float32 if arr.dtype[f].base == np.float32 else np.float64) for f in arr.dtype.names}
             for name, arr in tables.items()}
    row_bytes = {name: 8 + sum(np.dtype(k).itemsize * max(1, int(np.prod(tables[name].dtype[f].shape))) for f, k in kinds[name].items())
                 for name in tables}
    left = DUMP_BYTES
    for z, name in enumerate(sorted(tables, key=lambda n: len(tables[n]) * row_bytes[n])):
        arr = tables[name]
        cap = left // (len(tables) - z) // row_bytes[name]
        rows = np.arange(len(arr))
        if len(arr) > cap:
            rows = np.sort(np.random.default_rng(0).choice(len(arr), cap, replace=False))
        left -= len(rows) * row_bytes[name]
        np.save(os.path.join(out_dir, '%s%s_row.npy' % (prefix, name)), rows.astype(np.float64))
        for f, kind in kinds[name].items():
            np.save(os.path.join(out_dir, '%s%s_%s.npy' % (prefix, name, f)), np.ascontiguousarray(arr[f][rows], dtype=kind))


def workload_name(cfg, sumM):
    if cfg == 2:
        return "configs[1]: 100 synthetic 2 Mb bins (1,900 ORFs, ~0.59 M residues each) x cpr_43_markers.hmm (43 HMMs, sum M = %d)" % sumM
    if cfg == 4:
        return ("configs[3] stand-in, strong scaling: a fixed set of 512 synthetic bins with log-normal genome sizes (median 3.2 Mb, "
                "0.6-10 Mb) x 5,000 HMMs (sum M = %d), LPT-partitioned over the ranks" % sumM)
    return ("configs[2] stand-in: synthetic 3 Mb bins (2,900 ORFs, ~0.9 M residues, 0-2 planted homologs per CPR family) x 5,000 HMMs "
            "(the 43 real HMMER-calibrated CPR models x 116 replicas under distinct accessions, sum M = %d)" % sumM)


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm
# ----------------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm starts: the CPUs this process may run on, capped by the cgroup CPU quota when there is one (a
    container that sees 128 CPUs but is granted 12 CPU-seconds per second gains nothing from 128 threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()                       # cgroup v2
        if quota != 'max':
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        try:
            quota = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())                  # cgroup v1
            period = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if quota > 0:
                n = min(n, max(1, -(-quota // period)))
        except Exception:
            pass
    return n


def cpu_seconds():
    t = os.times()
    return t.user + t.system


def cpu_arm_setup(db_path):
    """Oracle model file with the SSE2 filters enabled; the reference's reduction if oracle/_ref was built."""
    from oracle import pyoracle as po
    from oracle import build_ref
    hf = po.HmmFile(db_path)
    hf.enable_simd()
    ref = None
    data = '/tmp/ckm_bench_cpu_data'
    os.makedirs(os.path.join(data, 'pfam'), exist_ok=True)
    with open(os.path.join(data, 'pfam', 'Pfam-A.hmm.dat'), 'w') as f:
        f.write('# STOCKHOLM 1.0\n//\n')
    if build_ref.available():
        try:
            HmmModelParser, MarkerSetParser, ResultsParser = build_ref.import_reference(data)
            ref = dict(models=HmmModelParser(db_path).models(), ResultsParser=ResultsParser, MarkerSetParser=MarkerSetParser, db_path=db_path)
        except Exception as exc:              # the baseline then stops at the hit table, and says so
            ref = None
            sys.stderr.write('reference reduction unavailable: %r\n' % (exc,))
    return po, hf, ref


def cpu_arm_step(po, hf, ref, bins, nthreads, workdir):
    """The CPU path over `bins`: search every bin on all cores, write domtblout, run the reference's reduction.  Returns
    (seconds search, seconds reduce, rows)."""
    shutil.rmtree(workdir, ignore_errors=True)
    os.makedirs(os.path.join(workdir, 'storage'))
    with open(os.path.join(workdir, 'storage', 'bin_stats.analyze.tsv'), 'w') as f:
        for b in bins:
            f.write("%s\t{'GC': 0.5, 'Genome size': 1000}\n" % b.bin_id)
    t0 = time.perf_counter()
    rows = 0
    hmmsearch = shutil.which('hmmsearch')
    for b in bins:
        bdir = os.path.join(workdir, 'bins', b.bin_id)
        os.makedirs(bdir)
        table = os.path.join(bdir, 'hmmer.analyze.txt')
        if hmmsearch:
            faa = os.path.join(bdir, 'genes.faa')
            with open(faa, 'w') as f:
                f.write(b.fasta())
            subprocess.check_call([hmmsearch, '--domtblout', table, '--noali', '--notextw', '-E', '0.1', '--domE', '0.1', '--cpu', str(nthreads),
                                   hf.path if hasattr(hf, 'path') else ref['db_path'], faa], stdout=subprocess.DEVNULL)
        else:
            rp = po.search(hf, b.residues, b.offsets, nthreads=nthreads)
            po.write_domtblout(rp, hf, b.names, b.descs, table)
            rows += rp.contents.nhits
            po.free_results(rp)
    t1 = time.perf_counter()
    if ref is not None:
        import warnings
        RP = ref['ResultsParser']({b.bin_id: ref['models'] for b in bins})
        old = sys.stderr
        sys.stderr = io.StringIO()
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                RP.analyseResults(workdir, 'bin_stats.analyze.tsv', 'hmmer.analyze.txt')
                ms = ref['MarkerSetParser']().getMarkerSets(workdir, [b.bin_id for b in bins], ref['db_path'])
                for b in bins:
                    RP.results[b.bin_id].geneCountsForSelectedMarkerSet(ms[b.bin_id], False)
        finally:
            sys.stderr = old
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, rows, ('hmmer' if hmmsearch else 'port')


def run_reference(args):
    rank, local, world = rank_info()
    if rank != 0:
        return
    cfg = args.config
    spec = CFG[cfg]
    db_path = model_db(spec['n_models'])
    nper = 1 if cfg != 2 else 4                               # bins per step: a bounded sample of the workload, never scaled
    bins = make_bins(nper, 1000, spec['orfs'] or 2900)
    cores = host_threads()
    sumM = total_model_positions(db_path)
    po, hf, ref = cpu_arm_setup(db_path)
    work = '/tmp/ckm_bench_cpu_run'
    for _ in range(1 if args.warmup > 0 else 0):               # one warm-up step is enough for a CPU path (page cache, threads)
        cpu_arm_step(po, hf, ref, bins[:1], cores, work)
    ts = tr = 0.0
    kind = 'port'
    c0 = cpu_seconds()
    for _ in range(args.steps):
        a, b, _, kind = cpu_arm_step(po, hf, ref, bins, cores, work)
        ts += a
        tr += b
    cpu_s = cpu_seconds() - c0
    t = ts + tr
    gph = nper * args.steps / t * 3600.0
    cells = float(sum(len(b.residues) for b in bins)) * sumM * args.steps
    sample = ("%d full bin(s) (%d ORFs each) x all %d models per step, %d steps: search %.1f s on %d threads (%s), reduction %.1f s (%s); "
              "no extrapolation" % (nper, bins[0].nseq, spec['n_models'], args.steps, ts, cores,
                                    'hmmsearch' if kind == 'hmmer' else 'CPU restatement with SSE2 striped MSV/Viterbi filters',
                                    tr, "the reference's own ResultsParser, one process" if ref is not None else 'not available'))
    line = {"metric": "genomes/hour", "value": gph, "unit": "genomes/hour", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * t / args.steps, "higher_is_better": True, "scaling": "weak" if cfg != 4 else "strong", "vs_baseline": None,
            "dtype": "u8/int16/f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(cfg, sumM), "bins_per_step": args.bins_per_step, "orfs_per_bin": bins[0].nseq, "n_models": spec['n_models'],
                       "per_gpu_bins_per_step": args.bins_per_step, "parallelism": "CPU: all host cores on one bin at a time",
                       "sample_per_step": sample},
            "cpu_baseline": {"value": gph, "unit": "genomes/hour", "cores": cores, "kind": kind, "sample": sample,
                             "cores_visible": os.cpu_count(), "cores_busy": cpu_s / t, "cpu_seconds_per_bin": cpu_s / (nper * args.steps),
                             "gcups_per_core": cells / cpu_s / 1e9, "search_s_per_bin": ts / (nper * args.steps),
                             "reduce_s_per_bin": tr / (nper * args.steps),
                             "note": "gcups_per_core = DP cells of the step / CPU-seconds consumed, whole pipeline (HMMER's published MSV filter speed is "
                                     "~10 GCUPS per core); cores_busy = CPU-seconds / wall seconds, i.e. the host cores this run really had"},
            "e2e": {"value": gph, "unit": "genomes/hour", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ckm')
    ap.add_argument('--config', type=int, default=3, choices=(2, 3, 4))
    ap.add_argument('--bins-per-step', type=int, default=BINS_PER_STEP)
    ap.add_argument('--db', default='replicas', choices=('replicas', 'diverse'), help='config 3/4 model database: 116 replicas of the 43 calibrated models (default) or 5,000 stitched models of diverse length')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-plugin', action='store_true', help='skip the files-on-disk plug-in path measurement')
    ap.add_argument('--profile-plugin', action='store_true', help='cProfile of the plug-in path host code (stderr)')
    ap.add_argument('--pipeline', type=int, default=2, help='batches in flight per GPU (one engine + host thread each)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the hit table and QA rows of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
        return
    rank, local, world = rank_info()
    cfg = args.config
    spec = CFG[cfg]
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    os.environ['CKM_DEVICE'] = str(local)
    from checkm_b200 import _lib, runtime, sharding
    from checkm_b200.resultsParser import QA_DTYPE
    B = args.bins_per_step
    get_db = diverse_model_db if (args.db == 'diverse' and spec['n_models'] != 43) else model_db
    if rank == 0:
        get_db(spec['n_models'])
    if world > 1:
        dist.barrier()
    db_path = get_db(spec['n_models'])
    NP = max(1, args.pipeline)
    engs = runtime.engines(NP)
    t0 = time.perf_counter()
    models = runtime.models_for(db_path)
    t_load = time.perf_counter() - t0
    info = models.info()
    nm = models.n
    sumM_all = sum(int(mi.M) for mi in info)

    # ---- the rank's batches, and which batches make up step i ----
    t0 = time.perf_counter()
    total_bins = None
    if cfg == 3:
        batches = [Batch(make_bins(B, 10000 * (rank + 1) + 100 * z, spec['orfs'])) for z in range(2)]
        step_batches = lambda i: [i % 2]                      # noqa: E731
        bins_per_step_rank = B
    else:
        if cfg == 2:
            allbins = make_bins(spec['total_bins'], 0, spec['orfs'])
        else:
            allbins = heterogeneous_bins(spec['total_bins'])
        total_bins = len(allbins)
        costs = [float(len(b.residues)) * sumM_all for b in allbins]
        mine = sharding.partition_bins(costs, world)[rank]
        mybins = [allbins[int(j)] for j in mine]
        # batches of at most B bins and ~32 M residues, largest bins first (the tail of the step is then made of small batches)
        mybins.sort(key=lambda b: -len(b.residues))
        batches, cur, cur_res = [], [], 0
        for b in mybins:
            if cur and (len(cur) >= B or cur_res + len(b.residues) > 32 * 1024 * 1024):
                batches.append(Batch(cur))
                cur, cur_res = [], 0
            cur.append(b)
            cur_res += len(b.residues)
        if cur:
            batches.append(Batch(cur))
        step_batches = lambda i: list(range(len(batches)))    # noqa: E731
        bins_per_step_rank = len(mybins)
        del allbins
    t_gen = time.perf_counter() - t0
    for bt in batches:
        bt.db = [e_.seqdb(bt.res, bt.off, bt.binof, len(bt.bins)) for e_ in engs]

    # ---- reduction metadata: one marker set per bin = all models (HMM-file semantics), no clans ----
    acc_is_tigr = np.asarray([1 if b'TIGR' in mi.acc else 0 for mi in info], dtype=np.uint8)
    is_pfam = np.asarray([1 if mi.acc.startswith(b'PF') else 0 for mi in info], dtype=np.uint8)
    clan = np.full(nm, -1, dtype=np.int32)
    nest_off = np.zeros(nm + 1, dtype=np.int64)
    has = np.zeros((nm, 3), dtype=np.int32)
    cut = np.zeros((nm, 6), dtype=np.float64)
    for i, mi in enumerate(info):
        has[i] = (mi.has_ga, mi.has_tc, mi.has_nc)
        cut[i] = (mi.ga_d[0], mi.ga_d[1], mi.tc_d[0], mi.tc_d[1], mi.nc_d[0], mi.nc_d[1])
    opts = _lib.ReduceOpts()
    opts.evalue_threshold, opts.evalue_exp10, opts.evalue_mant = 1e-10, -10, 10.0
    opts.length_threshold, opts.pseudogene_length = 0.7, 0.3

    def batch_meta(bt):
        if bt.meta is None:
            scaf, num, rank_ = [], [], []
            scaf_ids = {}                              # the same ids on every run (str hashes change with the process)
            for bi, b in enumerate(bt.bins):
                order = {n: r for r, n in enumerate(sorted(b.names))}
                for n in b.names:
                    c = n.rfind('_')
                    scaf.append(scaf_ids.setdefault((bi, n[:c]), len(scaf_ids)))
                    num.append(int(n[c + 1:]))
                    rank_.append(order[n])
            nb = len(bt.bins)
            bt.meta = tuple(np.asarray(a, dtype=np.int32) for a in (scaf, num, rank_)) + \
                (np.arange(nb + 1, dtype=np.int64), np.arange(nb + 1, dtype=np.int64) * nm, np.tile(np.arange(nm, dtype=np.int32), nb))
        return bt.meta

    def reduce_hits(bt, hits, eng):
        scaf, num, rank_, bin_set_off, set_marker_off, set_marker_idx = batch_meta(bt)
        meta = _lib.ReduceMeta()
        meta.is_pfam, meta.is_tigr, meta.clan = is_pfam.ctypes.data, acc_is_tigr.ctypes.data, clan.ctypes.data
        meta.nest_off, meta.nest_idx = nest_off.ctypes.data, None
        meta.has_cut, meta.cutoffs = has.ctypes.data, cut.ctypes.data
        meta.scaffold_id, meta.orf_num, meta.name_rank = scaf.ctypes.data, num.ctypes.data, rank_.ctypes.data
        meta.bin_set_off, meta.set_marker_off, meta.set_marker_idx = bin_set_off.ctypes.data, set_marker_off.ctypes.data, set_marker_idx.ctypes.data
        qa = C.POINTER(_lib.QaRow)()
        nqa = C.c_int32()
        mh = C.POINTER(_lib.MarkerHit)()
        nmh = C.c_int64()
        harr = np.ascontiguousarray(hits)
        _lib.check(_lib.lib().ckm_reduce(eng._h, nm, len(scaf), len(bt.bins), harr.ctypes.data_as(C.POINTER(_lib.Hit)), len(harr), C.byref(opts),
                                         C.byref(meta), C.byref(qa), C.byref(nqa), C.byref(mh), C.byref(nmh)))
        buf = (C.c_char * (nqa.value * C.sizeof(_lib.QaRow))).from_address(C.addressof(qa.contents))
        rows = np.frombuffer(buf, dtype=QA_DTYPE).copy()
        _lib.lib().ckm_free(qa)
        _lib.lib().ckm_free(mh)
        return rows, nmh.value

    for bt in batches:
        batch_meta(bt)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device='cuda')

    # ---- QA-row gather: NCCL all-gather through the library's own entry point (ckm_allgather_qa) ----
    comm = None
    max_rows = max(1, bins_per_step_rank)
    if world > 1:
        mr = torch.tensor([max_rows], dtype=torch.int64, device='cuda')
        dist.all_reduce(mr, op=dist.ReduceOp.MAX)
        max_rows = int(mr.item())
        uid = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            _lib.check(_lib.lib().ckm_nccl_unique_id(uid.ctypes.data, 128))
        ut = torch.from_numpy(uid).cuda()
        dist.broadcast(ut, 0)
        uid = ut.cpu().numpy()
        comm = C.c_void_p()
        _lib.check(_lib.lib().ckm_nccl_comm_init(engs[0]._h, world, rank, uid.ctypes.data, C.byref(comm)))
    gathered = np.zeros(world * max_rows, dtype=QA_DTYPE)
    counts = np.zeros(world, dtype=np.int32)
    gather_lock = threading.Lock()

    def gather(rows):
        """All ranks' QA rows of a step on every rank (config #4's "NCCL gather of qa table")."""
        if world == 1:
            return rows
        with gather_lock:
            r = np.ascontiguousarray(rows)
            _lib.check(_lib.lib().ckm_allgather_qa(engs[0]._h, comm, r.ctypes.data, len(r), max_rows, world, gathered.ctypes.data, counts.ctypes.data))
        return gathered

    host_ms = {'search': 0.0, 'reduce': 0.0}

    def do_batch(bt, w, resident):
        e_ = engs[w]
        flush_buf.zero_()                              # 256 MiB write, asynchronous to the engine streams
        t1 = time.perf_counter()
        if resident:
            hits = e_.search(models, bt.db[w])
            st = e_.stats()
        else:
            db = e_.seqdb(bt.res, bt.off, bt.binof, len(bt.bins))          # host buffers -> HBM
            try:
                hits = e_.search(models, db)                                # hit table back on the host
                st = e_.stats()
            finally:
                db.close()
        t2 = time.perf_counter()
        rows, nmh = reduce_hits(bt, hits, e_)
        t3 = time.perf_counter()
        return hits, st, rows, (1e3 * (t2 - t1), 1e3 * (t3 - t2))

    def run_steps(nsteps, resident):
        """nsteps steps; the batches of all steps form one work list that the NP pipeline slots take in order.  The QA rows of
        a step are gathered when its last batch is done.  Returns the per-batch records."""
        work = [(i, b) for i in range(nsteps) for b in step_batches(i)]
        out = [None] * len(work)
        errs = []
        remaining = {}
        for i, _ in work:
            remaining[i] = remaining.get(i, 0) + 1
        rows_of = {i: [] for i in remaining}
        lock = threading.Lock()

        def worker(w):
            try:
                torch.cuda.set_device(local)           # the current device is per host thread
                for z in range(w, len(work), NP):
                    i, b = work[z]
                    rec = do_batch(batches[b], w, resident)
                    out[z] = rec
                    with lock:
                        rows_of[i].append(rec[2])
                        remaining[i] -= 1
                        last = remaining[i] == 0
                    if last and world == 1:
                        gather(np.concatenate(rows_of[i]))
            except BaseException as ex:                # surfaced on the main thread
                errs.append(ex)
        if NP == 1:
            worker(0)
        else:
            ths = [threading.Thread(target=worker, args=(w,)) for w in range(NP)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        if errs:
            raise errs[0]
        if world > 1:                                  # collectives from one thread, in step order, on every rank
            for i in sorted(rows_of):
                gather(np.concatenate(rows_of[i]) if rows_of[i] else np.zeros(0, dtype=QA_DTYPE))
        return out

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(nsteps, resident):
        """nsteps steps between two device-wide synchronisations (+ barrier), timed on the device with CUDA events recorded
        right after the first and right after the second synchronisation (the engines launch on their own streams, so the
        events bracket the region rather than ride one stream); the host wall clock is kept as a cross-check."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        ev0.record()
        t0_ = time.perf_counter()
        recs_ = run_steps(nsteps, resident)
        sync()
        ev1.record()
        ev1.synchronize()
        return recs_, ev0.elapsed_time(ev1) / 1e3, time.perf_counter() - t0_

    run_steps(max(args.warmup, 0) if cfg == 3 else min(1, args.warmup), True)
    sampler = ClockSampler(local)
    sampler.start()
    recs, t_res, t_res_wall = timed(args.steps, True)
    if args.dump_outputs:
        last = recs[-len(step_batches(args.steps - 1)):]      # the batches of the last timed step, in work order
        dump_outputs(args.dump_outputs, {'hits': np.concatenate([r[0] for r in last]), 'qa': np.concatenate([r[2] for r in last])},
                     '' if world == 1 else 'rank%d_' % rank)
    ssv_ms = msv_ms = other_ms = 0.0
    launches = cells = pairs = 0
    for hits, st, rows, hm in recs:
        ssv_ms += st.ms_ssv
        msv_ms += st.ms_msv
        other_ms += st.ms_bias + st.ms_vit + st.ms_fwd + st.ms_domdef
        launches += st.kernel_launches + 5
        cells += st.n_cells
        pairs += st.n_pairs
        host_ms['search'] += hm[0]
        host_ms['reduce'] += hm[1]
    hits, st, rows = recs[-1][:3]
    d2h = int(sum(r[0].nbytes + r[2].nbytes for r in recs) / args.steps)
    recs_e, t_e2e, t_e2e_wall = timed(args.steps, False)
    # one batch at a time on one engine: the stage times of an undisturbed search (the SSV roofline is quoted on both)
    iso = [do_batch(batches[step_batches(i)[0]], 0, True)[1] for i in range(2)]
    sync()
    iso_ssv_ms = sum(s_.ms_ssv for s_ in iso) / len(iso)
    iso_st = iso[-1]
    iso_bins = len(batches[step_batches(1)[0]].bins)

    # ---- the plug-in path itself (config 3, one GPU): files on disk -> find -> domtblout/side-car -> analyseResults -> QA table ----
    plugin = None
    if cfg == 3 and world == 1 and not args.no_plugin:
        plugin = plugin_path(args, batches, db_path, models)

    sampler.stop_flag = True
    sampler.join(timeout=2)
    if world > 1:
        tt = torch.tensor([t_res, t_e2e], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_res, t_e2e = float(tt[0]), float(tt[1])
        nb = torch.tensor([bins_per_step_rank], dtype=torch.int64, device='cuda')
        dist.all_reduce(nb, op=dist.ReduceOp.SUM)
        bins_per_step_all = int(nb.item())
    else:
        bins_per_step_all = bins_per_step_rank
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    genomes = bins_per_step_all * args.steps
    value = genomes / t_res * 3600.0
    e2e = genomes / t_e2e * 3600.0
    # roofline of the dominant kernel (SSV pre-filter): algorithmic bytes = sum over pairs of (L + 4) (SURVEY.md 8d)
    nsteps_batches = float(len(recs)) / args.steps
    resid_step = float(sum(len(batches[b].res) for b in step_batches(0)))
    alg_bytes_per_step = resid_step * nm + 4.0 * (pairs / args.steps)
    peaks, peak_kind = measured_peaks()
    traffic = ssv_traffic()
    ssv_s = (ssv_ms / args.steps) / 1000.0
    achieved = alg_bytes_per_step / ssv_s / 1e9
    real_cells = resid_step * sumM_all
    h2d = int(sum(batches[b].res.nbytes + batches[b].off.nbytes + batches[b].binof.nbytes for b in step_batches(0)))
    line = {"metric": "genomes/hour", "value": value, "unit": "genomes/hour", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * t_res / args.steps, "higher_is_better": True, "scaling": "strong" if cfg == 4 else "weak", "vs_baseline": None,
            "dtype": "int16 (SSV) / u8 (MSV) / int16 (Viterbi) / f32 (Forward, domain definition)", "data": "synthetic",
            "config": {"workload": workload_name(cfg, sumM_all) + (" [--db diverse: 5,000 stitched models, lengths log-normal 30-1,500]" if args.db == 'diverse' else ""), "config": cfg,
                       "bins_per_step": bins_per_step_all, "orfs_per_bin": spec['orfs'], "n_models": nm, "per_gpu_bins_per_step": bins_per_step_rank,
                       "batches_per_step_per_gpu": nsteps_batches, "parallelism": "bins sharded, 1 process/GPU" + (", LPT partition of a fixed set" if cfg == 4 else ""),
                       "batches_in_flight_per_gpu": NP,
                       "l2": "256 MiB flush write issued before every batch; the model tables alone (> 200 MB for 5,000 models) exceed L2",
                       "model_load_s": t_load, "workload_generation_s": t_gen},
            "e2e": {"value": e2e, "unit": "genomes/hour", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "C ABI with host buffers: ckm_seqdb_create (H2D) + ckm_search (D2H hit table) + ckm_reduce (D2H QA rows) per batch"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks.get("hbm_gbs"), "unit": "GB/s", "frac": achieved / peaks.get("hbm_gbs"),
                         "traffic": (traffic["dram_bytes_per_bin"] * bins_per_step_rank) if (traffic and cfg != 2) else None,
                         "traffic_source": (traffic or {}).get("source"), "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == 'measured' else 'fallback 6650',
                         "kernel": "ssv_kernel<J> (SSV pre-filter, all pairs)", "kernel_ms_per_step": ssv_ms / args.steps,
                         "isolated": {"kernel_ms": iso_ssv_ms, "bins": iso_bins, "what": "same kernel, one batch in flight (no other stream on the SMs)"},
                         "note": "the stage is DP-cell bound, not HBM bound (SURVEY.md 8d): see gcups"},
            "gcups": {"real_cells_per_step": real_cells, "tile_cells_per_step": cells / args.steps, "ssv_gcups_real": real_cells / ssv_s / 1e9,
                      "ssv_gcups_tile": cells / args.steps / ssv_s / 1e9, "smem_bound_gcups": 148 * (2048.0 / 31.0) * 1.965,
                      "smem_bound_note": "J=32 tile row = 7 LDS.128 (1 int8 chunk + 6 int16 quads = 28 wavefronts) + 1 SHFL (3) per 2048 cells at 1 wavefront/clk/SM, 148 SMs, 1.965 GHz",
                      "ssv_frac_of_smem_bound": (cells / args.steps / ssv_s / 1e9) / (148 * (2048.0 / 31.0) * 1.965),
                      "stage_ms_per_step": {"ssv": ssv_ms / args.steps, "msv_exact": msv_ms / args.steps, "bias+vit+fwd+domdef": other_ms / args.steps,
                                            "wall_ms_per_step": {k_: v_ / args.steps for k_, v_ in host_ms.items()},
                                            "isolated_batch": {"bins": iso_bins, "ssv": iso_st.ms_ssv, "msv_exact": iso_st.ms_msv, "bias": iso_st.ms_bias, "vit": iso_st.ms_vit,
                                                               "fwd": iso_st.ms_fwd, "domdef": iso_st.ms_domdef, "total": iso_st.ms_total}}},
            "cascade": {"pairs": int(st.n_pairs), "ssv_cand": int(st.n_ssv_cand), "past_msv": int(st.n_past_msv), "past_bias": int(st.n_past_bias),
                        "past_vit": int(st.n_past_vit), "past_fwd": int(st.n_past_fwd), "rows": int(st.n_reported), "vit_int32_redo": int(st.n_vit_redo),
                        "what": "last batch of the timed region"},
            "timing": {"how": "CUDA events around the K timed steps (after barrier + device synchronize on both sides), max over ranks", "host_wall_s": t_res_wall, "host_wall_e2e_s": t_e2e_wall},
            "clocks": sampler.summary()}
    if plugin is not None:
        line["plugin"] = plugin
    if not args.no_cpu_baseline and world == 1:
        cores = host_threads()
        po, hf, ref = cpu_arm_setup(db_path)
        sample_bins = batches[0].bins[:1] if cfg != 2 else batches[0].bins[:4]
        c0 = cpu_seconds()
        ts_, tr_, _, kind = cpu_arm_step(po, hf, ref, sample_bins, cores, '/tmp/ckm_bench_cpu_run')
        cpu_s = cpu_seconds() - c0
        cb = float(sum(len(b.residues) for b in sample_bins)) * sumM_all
        line["cpu_baseline"] = {"value": len(sample_bins) / (ts_ + tr_) * 3600.0, "unit": "genomes/hour", "cores": cores, "kind": kind,
                                "cores_visible": os.cpu_count(), "cores_busy": cpu_s / (ts_ + tr_), "cpu_seconds_per_bin": cpu_s / len(sample_bins),
                                "gcups_per_core": cb / cpu_s / 1e9, "search_s_per_bin": ts_ / len(sample_bins), "reduce_s_per_bin": tr_ / len(sample_bins),
                                "sample": "%d full bin(s) x all %d models: search %.1f s on %d threads (%s) + reduction %.1f s (%s); no extrapolation"
                                          % (len(sample_bins), nm, ts_, cores, 'hmmsearch' if kind == 'hmmer' else 'CPU restatement, SSE2 striped filters', tr_,
                                             "the reference's ResultsParser" if ref is not None else 'not available')}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def plugin_path(args, batches, db_path, models):
    """FASTA files on disk -> MarkerGeneFinder.find -> domtblout + side-car -> ResultsParser.analyseResults -> printSummary(1):
    what `checkm analyze --genes` + `checkm qa` run, per step of bins_per_step bins, all inside the timed region."""
    import logging
    import torch
    from checkm_b200.markerGeneFinder import MarkerGeneFinder
    from checkm_b200.markerSets import MarkerSetParser
    from checkm_b200.resultsParser import ResultsParser
    from checkm_b200.defaultValues import DefaultValues
    logging.getLogger('timestamp').setLevel(logging.ERROR)
    root = '/tmp/ckm_bench_plugin_%d' % os.getpid()
    shutil.rmtree(root, ignore_errors=True)
    data = os.path.join(root, 'data')
    os.makedirs(os.path.join(data, 'pfam'))
    with open(os.path.join(data, 'pfam', 'Pfam-A.hmm.dat'), 'w') as f:
        f.write('# STOCKHOLM 1.0\n//\n')
    DefaultValues.set_data_root(data)
    # args.steps x bins_per_step distinct bins (hard links to the two batches' files under distinct bin ids): ONE find() call and
    # ONE analyseResults over all of them, as `checkm analyze` / `checkm qa` run on a directory of bins
    src = []
    for z, bt in enumerate(batches):
        d = os.path.join(root, 'src%d' % z)
        os.makedirs(d)
        for b in bt.bins:
            p_ = os.path.join(d, b.bin_id + '.faa')
            with open(p_, 'w') as f:
                f.write(b.fasta())
            src.append(p_)

    def bin_files(tag, nsteps):
        d = os.path.join(root, 'in_' + tag)
        os.makedirs(d)
        out_ = []
        for i in range(nsteps * len(batches[0].bins)):
            p_ = os.path.join(d, 'g%s_%04d.faa' % (tag, i))
            os.link(src[i % len(src)], p_)
            out_.append(p_)
        return out_

    class _AAI:
        aaiMeanBinHetero = {}
    stage = {'find': 0.0, 'marker_sets': 0.0, 'analyse': 0.0, 'summary': 0.0}

    def run(tag, nsteps):
        out = os.path.join(root, 'out_' + tag)
        os.makedirs(os.path.join(out, 'storage'))
        binFiles = bin_files(tag, nsteps)
        t0 = time.perf_counter()
        binIdToModels = MarkerGeneFinder(1).find(binFiles, out, 'hmmer.analyze.txt', 'hmmer.analyze.ali.txt', db_path, False, False, True)
        t1 = time.perf_counter()
        binIds = sorted(binIdToModels.keys())
        with open(os.path.join(out, 'storage', 'bin_stats.analyze.tsv'), 'w') as f:
            for b in binIds:
                f.write("%s\t{'GC': 0.5, 'Genome size': 1000}\n" % b)
        ms = MarkerSetParser(1).getMarkerSets(out, binIds, db_path)
        t2 = time.perf_counter()
        RP = ResultsParser(binIdToModels)
        RP.analyseResults(out, 'bin_stats.analyze.tsv', 'hmmer.analyze.txt')
        t3 = time.perf_counter()
        RP.printSummary(1, _AAI(), ms, False, None, True, os.path.join(out, 'qa.tsv'), out)
        t4 = time.perf_counter()
        for k, v in zip(('find', 'marker_sets', 'analyse', 'summary'), (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            stage[k] += v
        for k, v in getattr(RP, 'timing', {}).items():
            stage['analyse.' + k] = stage.get('analyse.' + k, 0.0) + v
        return len(binIds)
    run('warm', 1)
    for k in [k for k in stage if k.startswith('analyse.')]:
        del stage[k]
    if args.profile_plugin:
        import cProfile
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        run('prof', 1)
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats('cumulative').print_stats(28)
    for k in stage:
        stage[k] = 0.0
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t0 = time.perf_counter()
    n = run('timed', args.steps)
    torch.cuda.synchronize()
    ev1.record()
    ev1.synchronize()
    wall = time.perf_counter() - t0
    dev = ev0.elapsed_time(ev1) / 1e3
    shutil.rmtree(root, ignore_errors=True)
    return {"value": n / dev * 3600.0, "unit": "genomes/hour", "bins": n, "seconds": dev, "host_wall_s": wall,
            "ms_per_bin": {k: 1e3 * v / n for k, v in stage.items()},
            "what": "files on disk -> ONE MarkerGeneFinder.find over all bins (reader / 2 searchers / writer threads) -> domtblout + side-car "
                    "per bin -> ONE ResultsParser.analyseResults -> printSummary(1) to a file: what `checkm analyze --genes` + `checkm qa` run"}


if __name__ == '__main__':
    main()
