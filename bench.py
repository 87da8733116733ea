#!/usr/bin/env python3
"""
bench.py -- BASELINE.json metric on B200: reads/s (+ GCUPS) of the adapter-alignment hot path.

Main line (default --workload endtrim = BASELINE.json configs[1]): 1 M synthetic ~8 kb ONT reads (seed 20260923, SURVEY
8(d)), adapter set SQK-NSK007 (= the LSK109 Y-adapter), end-trim only: per read the 150-nt start window vs Y_Top (28 nt)
and the 150-nt end window vs Y_Bottom (22 nt) -> 2 alignments, 7 500 DP cells, 372 algorithmic bytes per read.  A "step"
is one pass of the hot path over the whole batch.

The same JSON line carries a `configs` block with a reduced-step run of the other BASELINE configs (each with its own
value / e2e / roofline / parity gate / cpu_baseline):
  demux   configs[2]  1 M reads x 356 adapter sequences (all 119 sets + 12 native-full + 96 rapid-full), end windows
  middle  configs[3]  full-read middle-adapter scan, 5 % chimeras: 10 M reads over 8 GPUs = 1.25 M reads per GPU
  sweep   configs[4]  read-length sweep 500 bp - 100 kb x the 192 forward-barcode sequences, 2.5e8 bases per length and GPU
(--configs none skips them, --workload X makes X the main line.)

  value   reads/s with the inputs already resident in HBM (adapterAlignmentBatchDevice), CUDA-event timed
  e2e     reads/s through the host-buffer C-ABI call (adapterAlignmentBatchMulti, pinned host buffers): H2D + kernels +
          D2H inside the timed region, every rank on its own shard and PCIe link; `e2e_with_gather` (N > 1) adds the NCCL
          gather of all records to rank 0 and rank 0's copy to its host memory
  roofline      dominant DP kernel: algorithmic bytes / CUDA-event duration vs the measured HBM peak (the north star asks
                for it; the kernel is integer-issue bound, so `roofline_alu` is the binding one)
  roofline_alu  cells/s of the dominant kernel vs the int16x2 issue peak: SMs x 4 schedulers x 32 lanes x clock x 2 cells
                / instructions per row-step (counted from SASS, profiles/sass_counts.json)
  cpu_baseline / --impl reference   the reference's own C++ (oracle/_ref/cpp_functions.so, else the oracle port) timed
          by the native harness on the host cores: 1 thread and a sweep over {nproc/4, nproc/2, nproc} threads and nproc
          processes (separate heaps), best kept, on a bounded sample of the same pair list

Launch: python bench.py [--gpus N --steps K --warmup W]; for N>1 via torchrun (one rank per GPU).  --scaling weak
(default): every rank processes its own full-size batch; --scaling strong: the batch is split over the ranks.
--dump-outputs DIR writes the main workload's records of the last timed step as .npy files; the inputs are seeded, so two
builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_READS = {'endtrim': 1000000, 'demux': 1000000, 'middle': 1250000, 'sweep': 0}
SWEEP_LENGTHS = '500,1000,2000,5000,10000,20000,50000,100000'
OUT_CAP_BYTES = 320 << 20          # e2e: records copied back per call (larger batches go through the ABI in read chunks)
DUMP_CAP_BYTES = 60000000          # --dump-outputs: all files together stay below 64 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='endtrim', choices=['endtrim', 'demux', 'middle', 'sweep'])
    ap.add_argument('--configs', default='all', help="other BASELINE configs measured into the line's `configs` block: "
                                                     "all | none | comma list of demux,middle,sweep")
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--sweep-lengths', default=SWEEP_LENGTHS)
    ap.add_argument('--sweep-bases', type=float, default=2.5e8, help='sweep: bases per length point and rank')
    ap.add_argument('--reads', type=int, default=0, help='reads of the main workload (per rank if weak, total if strong)')
    ap.add_argument('--config-reads', default='', help='reads of the `configs` entries, e.g. demux=65536,middle=131072')
    ap.add_argument('--cpu-sample-reads', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--e2e-decisions', action='store_true',
                    help='e2e (endtrim / demux): adapterEndDecisions -- trim amounts + barcode score pairs decided on the '
                         'device, 4 + 4*adapters bytes per window come back instead of 36 per alignment')
    ap.add_argument('--opt', action='append', default=[], metavar='NAME=VALUE',
                    help='engine option for this run (pb200SetOption), e.g. --opt scratch_mb=72')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='write the records of the last timed step of the main workload to DIR/*.npy (float64, at most '
                         '%d MB in all: a fixed seeded sample of rows where larger), to compare two builds output for output'
                         % (DUMP_CAP_BYTES // 1000000))
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed regions (NVML; nvidia-smi as fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self.stop_flag = False
        self.active = False
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40, 'hw_power_brake': 0x80,
                 'sw_power_cap': 0x4}
        while not self.stop_flag:
            if self.active:
                try:
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    try:
                        r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(0.01)

    def summary(self):
        if not self.samples:
            try:
                out = subprocess.check_output(['nvidia-smi', '--query-gpu=clocks.sm,clocks.max.sm', '--format=csv,noheader,nounits',
                                               '-i', str(self.index)], timeout=20).decode().strip().split(',')
                return {'sm_mhz': float(out[0]), 'sm_max_mhz': float(out[1]), 'reasons': ['not sampled under load']}
            except Exception:
                return {'sm_mhz': None, 'sm_max_mhz': self.sm_max, 'reasons': ['unavailable']}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.sm_max, 'reasons': sorted(self.reasons),
                'samples': len(self.samples)}

    def take(self):
        """summary of the samples since the last take()"""
        s = self.summary()
        self.samples, self.reasons = [], set()
        return s


# ------------------------------------------------------------------------------------------------------------------
class Workload:
    """name, desc (nominal, arm-independent), n reads on this rank, batches = [(name, buf uint8, off int64, adapters)]"""

    def __init__(self, name, desc, n, nominal_reads, batches):
        self.name, self.desc, self.n, self.nominal_reads, self.batches = name, desc, n, nominal_reads, batches
        self.cells = sum(int(off[-1] - off[0]) * sum(len(a) for a in ads) for _, _, off, ads in batches)
        self.alg_bytes = sum(int(off[-1] - off[0]) + sum(len(a) for a in ads) + 36 * (len(off) - 1) * len(ads)
                             for _, _, off, ads in batches)
        self.alignments_per_read = sum(len(ads) for _, _, _, ads in batches) if name != 'sweep' else len(batches[0][3])

    def config(self, scaling):
        """identical in both arms (the driver compares the dicts): nominal parameters only"""
        return {'workload': self.desc, 'reads_per_gpu' if scaling == 'weak' else 'reads_total': self.nominal_reads,
                'alignments_per_read': self.alignments_per_read, 'scoring': list(_wl().DEFAULT_SCORING), 'scaling': scaling}


def _wl():
    from porechop_b200 import workloads
    return workloads


def nominal_reads(name, args, main):
    if main and args.reads:
        return args.reads
    for kv in args.config_reads.split(','):
        k, _, v = kv.partition('=')
        if k == name and v:
            return int(v)
    return DEFAULT_READS[name]


def make_workload(name, args, rank, world, main, limit=None, alloc=None):
    """The batch of `rank`.  limit: only the first `limit` reads (the generators are prefix-consistent: the CPU arm times a
    prefix of exactly the batch the GPU arm aligns).  alloc(nbytes) -> uint8 array to generate large buffers into."""
    wl = _wl()
    seed = wl.SEED + rank
    nom = nominal_reads(name, args, main)
    n = nom if args.scaling == 'weak' else (nom // world + (1 if rank < nom % world else 0))
    if args.scaling == 'strong':
        seed = wl.SEED + 1000 + rank
    if limit is not None:
        n = min(n, limit)
    big = (lambda nbytes: alloc(nbytes)) if alloc else (lambda nbytes: None)
    if name == 'endtrim':
        yt, yb = wl.nsk007()
        L, sw, ew = wl.synth_end_windows(n, yt, yb, seed=seed)
        batches = [('start',) + wl.windows_to_batch(sw) + ([yt],), ('end',) + wl.windows_to_batch(ew) + ([yb],)]
        desc = '%d synthetic ~8kb reads (lognormal, seed %d+rank), SQK-NSK007 (LSK109 Y-adapter), end-trim: 150x28 + 150x22 per read' % (nom, wl.SEED)
    elif name == 'demux':
        starts, ends = wl.demux_adapters()
        L, sw, ew = wl.synth_end_windows(n, starts[100], ends[100], seed=seed)
        batches = [('start',) + wl.windows_to_batch(sw) + (starts,), ('end',) + wl.windows_to_batch(ew) + (ends,)]
        desc = '%d synthetic reads x 356 adapter sequences (119 sets + 12 native-full + 96 rapid-full: 227 start + 129 end), demux end windows' % nom
    elif name == 'sweep':
        bcs = wl.forward_barcode_sequences()
        lengths = [int(x) for x in args.sweep_lengths.split(',')]
        batches, n, nom = [], 0, 0
        for Ln in lengths:
            k_nom = max(1, int(args.sweep_bases // Ln))
            k = k_nom if args.scaling == 'weak' else max(1, k_nom // world)
            if limit is not None:
                k = min(k, max(1, int(limit * 8000 // Ln)))          # `limit` is given in 8-kb read equivalents
            buf, off = wl.synth_fixed_length_reads(k, Ln, bcs, seed=seed + Ln, out=big(k * Ln))
            batches.append(('L%d' % Ln, buf, off, bcs))
            n += k
            nom += k_nom
        desc = 'read-length sweep %s x 192 forward barcode sequences (24 nt), %.1e bases per length, full-read scan' % (
            args.sweep_lengths, args.sweep_bases)
    else:
        yt, yb = wl.nsk007()
        buf, off = wl.synth_reads_fast(n, yt, yb, seed=seed, chimera_p=0.05, out=big(n * 8400 + (4 << 20)) if n > 50000 else None)
        batches = [('middle', buf, off, [yt, yb])]
        desc = '%d synthetic full reads (~8 kb lognormal, 5%% chimeras) x {Y_Top, Y_Bottom}, middle-adapter scan' % nom
    return Workload(name, desc, n, nom, batches)


def cgroup_cpu_limit():
    """CPUs the cgroup lets this process use at once (cpu.max = "quota period", v1: cfs_quota_us / cfs_period_us), or None.
    Round 2: the GPU boxes show nproc = 128 under a quota of 16 CPUs -- threads beyond the quota only get throttled."""
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            q, p = f.read().split()[:2]
        return None if q == 'max' else max(1, int(-(-int(q) // int(p))))
    except (OSError, ValueError):
        pass
    try:
        with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
            q = int(f.read())
        with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
            p = int(f.read())
        return None if q <= 0 else max(1, -(-q // p))
    except (OSError, ValueError):
        return None


def host_cores():
    """host cores this process can really use: the affinity mask, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    lim = cgroup_cpu_limit()
    return max(1, min(n, lim)) if lim else n


def cpu_info():
    model, quota = None, None
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.startswith('model name'):
                    model = line.split(':', 1)[1].strip()
                    break
    except OSError:
        pass
    for p in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            with open(p) as f:
                quota = f.read().strip()
                break
        except OSError:
            pass
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count()
    return {'model': model, 'nproc': os.cpu_count(), 'affinity': aff, 'cgroup_cpu_max': quota, 'usable_cores': host_cores()}


# ------------------------------------------------------------------------------------------------------------------
def harness_paths():
    lib = os.path.join(ROOT, 'oracle', '_ref', 'cpp_functions.so')
    kind = 'reference'
    if not os.path.exists(lib):
        lib = os.path.join(ROOT, 'oracle', 'liboracle.so')
        kind = 'port'
    harness = os.path.join(ROOT, 'oracle', '_ref', 'ref_harness')
    if not os.path.exists(harness) or not os.path.exists(lib):
        subprocess.check_call(['make', '-s', '-C', os.path.join(ROOT, 'oracle'), 'liboracle.so', 'harness', 'ref'])
    return harness, lib, kind


class HarnessFiles:
    """The first `reads` reads of every batch of a workload, written once as harness input files."""

    def __init__(self, workload, reads_per_batch):
        wl = _wl()
        self.dir = tempfile.TemporaryDirectory()
        self.files, self.reads, self.cells = [], 0, 0
        for (name, buf, off, ads), k in zip(workload.batches, reads_per_batch):
            k = min(int(k), len(off) - 1)
            abuf, aoff = wl.pack_adapters(ads)
            p = os.path.join(self.dir.name, name + '.bin')
            base = int(off[0])
            wl.write_harness_file(p, buf[base:int(off[k])], off[:k + 1] - base, abuf, aoff, wl.DEFAULT_SCORING)
            self.files.append((name, p, k))
            self.reads += k
            self.cells += int(off[k] - off[0]) * sum(len(a) for a in ads)

    def run(self, threads, procs=1, answers=None):
        """-> seconds over all batches.  answers: list that receives, per batch, the result strings (pair order)."""
        harness, lib, kind = harness_paths()
        sec = 0.0
        env = dict(os.environ)
        if procs > 1:
            env['REF_HARNESS_PROCS'] = str(procs)
        for name, p, k in self.files:
            cmd = [harness, lib, p, str(threads)]
            if answers is not None:
                cmd.append(p + '.answers')
            info = json.loads(subprocess.check_output(cmd, env=env).decode())
            sec += info['seconds']
            if answers is not None:
                with open(cmd[-1]) as f:
                    answers.append(f.read().split('\n')[:-1])
        return sec


def sample_sizes(workload, cores, seconds, per_core_gcups=0.06):
    """reads per batch such that the all-core run takes about `seconds` (the reference runs ~0.08 GCUPS per core alone)."""
    out = []
    total_cells = max(workload.cells, 1)
    for name, buf, off, ads in workload.batches:
        n = len(off) - 1
        cells_per_read = max(1.0, (int(off[-1] - off[0]) / max(n, 1)) * sum(len(a) for a in ads))
        share = (int(off[-1] - off[0]) * sum(len(a) for a in ads)) / total_cells
        out.append(int(max(8, min(n, share * seconds * per_core_gcups * 1e9 * cores / cells_per_read))))
    return out


def cpu_baseline(workload, sample_reads=0, sweep=True, seconds=3.0, want_answers=True):
    """1-thread and all-core numbers of the reference CPU path on a bounded sample (SURVEY 8(d), BASELINE.md section 3).
    Returns (dict, answers per batch or None, reads per batch)."""
    cores = host_cores()
    harness, lib, kind = harness_paths()
    sizes = [min(sample_reads, len(off) - 1) for _, _, off, _ in workload.batches] if sample_reads else sample_sizes(workload, cores, seconds)
    files = HarnessFiles(workload, sizes)
    # reads/s of the WORKLOAD: a sample may hold different fractions of the batches, so scale by cells
    cells_per_read = workload.cells / max(workload.n, 1)
    answers = [] if want_answers else None
    runs = []
    if sweep or cores < 2:
        sec = files.run(cores, 1, answers)
        runs.append({'threads': cores, 'procs': 1, 'seconds': sec})
    if sweep and cores >= 4:
        over = min(2 * cores, os.cpu_count() or cores)      # under a cgroup quota, 2x the quota was the best mode on the round-2 box
        for t in sorted({max(1, cores // 2), over} - {cores}):
            runs.append({'threads': t, 'procs': 1, 'seconds': files.run(t)})
    if cores >= 2:
        # one process per core (separate heaps): the mode that does not depend on the allocator's arena behaviour; the side
        # configs time only this one (and take the parity answers from a small threaded run)
        runs.append({'threads': 1, 'procs': cores, 'seconds': files.run(1, cores)})
        if not sweep and want_answers:
            small = HarnessFiles(workload, [min(k, 512) for k in sizes])
            small.run(min(cores, 16), 1, answers)
    for r in runs:
        r['gcups'] = files.cells / r['seconds'] / 1e9
        r['reads_per_s'] = files.cells / r['seconds'] / cells_per_read
    best = max(runs, key=lambda r: r['gcups'])
    # one thread: a 1/cores share of the sample (about the same wall time)
    one = HarnessFiles(workload, [max(1, k // max(cores // 2, 1)) for k in sizes])
    sec1 = one.run(1)
    d = {'value': best['reads_per_s'], 'unit': 'reads/s', 'cores': best['threads'] * best['procs'], 'kind': kind,
         'gcups': best['gcups'], 'mode': '%d threads x %d processes' % (best['threads'], best['procs']),
         'one_thread': {'value': one.cells / sec1 / cells_per_read, 'unit': 'reads/s', 'gcups': one.cells / sec1 / 1e9,
                        'sample_reads': one.reads},
         'sweep': runs, 'host': cpu_info(),
         'sample': 'first %s reads of the batches (%d alignment cells x 1e6), native harness over the reference C-ABI '
                   '(adapterAlignment+freeCString); reads/s scaled by cells to the whole workload' % (sizes, files.cells // 1000000)}
    return d, answers, sizes


def parity_gate(records_per_batch, answers_per_batch, format_record):
    """SURVEY 8(d) parity gate: the engine's records of the sampled pairs, rendered as the reference's result string,
    must equal the CPU reference's strings.  (An empty alignment is compared on its first field only: the reference
    leaves the others uninitialised.)  Returns {'checked': n, 'mismatches': k}."""
    checked = bad = 0
    for rec, ans in zip(records_per_batch, answers_per_batch):
        assert len(rec) >= len(ans), 'parity sample larger than the kept records'
        for r, a in zip(rec[:len(ans)], ans):
            g = format_record(r)
            ok = (g == a) or (a.startswith('-1,') and g.startswith('-1,'))
            checked += 1
            bad += 0 if ok else 1
    return {'checked': checked, 'mismatches': bad}


# ------------------------------------------------------------------------------------------------------------------
def sass_counts():
    p = os.path.join(ROOT, 'profiles', 'sass_counts.json')
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return {}


def measure_gpu(workload, args, ctx, K, Wm, main):
    """value / e2e / roofline of one workload on this rank's GPU; rank 0 gets the complete dict."""
    import torch
    import torch.distributed as dist
    W, wl, world, rank, sampler = ctx['W'], _wl(), ctx['world'], ctx['rank'], ctx['sampler']
    scoring = wl.DEFAULT_SCORING
    keep = ctx['keep']

    def pinned(shape, dtype):
        t = torch.empty(shape, dtype=dtype, pin_memory=True)
        keep.append(t)
        return t

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- host (pinned) and device copies of the inputs ----
    host, dev = [], []
    for name, buf, off, ads in workload.batches:
        abuf, aoff = wl.pack_adapters(ads)
        hb = torch.from_numpy(buf)
        if not hb.is_pinned():
            hb = pinned(len(buf), torch.uint8)
            hb.numpy()[:] = buf
        ho = pinned(len(off), torch.int64)
        ho.numpy()[:] = off
        n_reads = len(off) - 1
        chunk = max(1, min(n_reads, OUT_CAP_BYTES // (36 * len(ads))))
        out0 = pinned((chunk * len(ads), 9), torch.int32)                # records of the first chunk are kept (parity gate)
        out1 = pinned((chunk * len(ads), 9), torch.int32) if chunk < n_reads else out0
        host.append((hb, ho, abuf, aoff, chunk, out0, out1))
        db, do = hb.cuda(non_blocking=True), ho.cuda(non_blocking=True)
        dout = torch.empty((n_reads * len(ads), 9), dtype=torch.int32, device='cuda')
        max_len = int(np.max(np.diff(off))) if n_reads else 0
        dev.append((db, do, abuf, aoff, dout, max_len))
    torch.cuda.synchronize()
    in_bytes = sum(h[0].numel() + h[1].numel() * 8 + len(h[2]) + len(h[3]) * 4 for h in host)
    # bytes that really cross PCIe: with the packed upload (h2d_pack, "auto" resolves per host) the sequences travel as 4-bit codes
    # (a submit = one chunk of every batch; the engine packs submits of >= 32 MB)
    per_submit = sum(h[0].numel() * min(1.0, h[4] / max(h[1].numel() - 1, 1)) for h in host)
    packed_upload = W.get_option('h2d_pack') == 1 or (bool(W.get_option('h2d_pack_large_submit')) and per_submit >= (32 << 20))
    h2d_bytes = in_bytes - sum(h[0].numel() // 2 for h in host) if packed_upload else in_bytes
    for h in host:      # equally long sequences (the 150-base end windows): the engine makes their offsets on the device
        lens = h[1][1:] - h[1][:-1]
        if lens.numel() and int(lens.min()) == int(lens.max()):
            h2d_bytes -= h[1].numel() * 8
    out_bytes = sum((h[1].numel() - 1) * (len(h[3]) - 1) * 36 for h in host)

    bench_stream = ctx['stream']

    def step_device():
        s = bench_stream.cuda_stream
        assert s != 0
        for db, do, abuf, aoff, dout, max_len in dev:
            W.adapter_alignment_batch_device(db.data_ptr(), do.data_ptr(), do.numel() - 1, db.numel(), max_len, abuf, aoff,
                                             scoring, dout.data_ptr(), s)

    # e2e: one Multi submit per step when everything fits the record cap, else read chunks per batch
    calls = []
    single = all(h[4] >= h[1].numel() - 1 for h in host)
    if single:
        calls.append([(hb.numpy(), ho.numpy(), abuf, aoff, out0.numpy()) for hb, ho, abuf, aoff, chunk, out0, out1 in host])
    else:
        for hb, ho, abuf, aoff, chunk, out0, out1 in host:
            n_reads = ho.numel() - 1
            for s0 in range(0, n_reads, chunk):
                s1 = min(n_reads, s0 + chunk)
                o = (out0 if s0 == 0 else out1).numpy()[:(s1 - s0) * (len(aoff) - 1)]
                calls.append([(hb.numpy(), ho.numpy()[s0:s1 + 1], abuf, aoff, o)])

    dec_out = None
    if args.e2e_decisions and workload.name in ('endtrim', 'demux'):
        dec_out = [(pinned(h[1].numel() - 1, torch.int32), pinned((h[1].numel() - 1, len(h[3]) - 1, 2), torch.uint16)) for h in host]

    def step_e2e():
        if dec_out is not None:
            W.adapter_end_decisions([(h[0].numpy(), h[1].numpy(), h[2], h[3], b[0] == 'start', list(range(len(b[3]))))
                                     for b, h in zip(workload.batches, host)], scoring, wl.END_SIZE, 2, 75.0, 4,
                                    out_arrays=[(t.numpy(), p.numpy(), None) for t, p in dec_out])
            return
        for c in calls:
            W.adapter_alignment_batch_multi(c, scoring)

    # ---- value: device-resident ----
    for _ in range(max(Wm, 1)):
        step_device()
    barrier()
    W.synchronize()
    W.timing_enable(True)
    W.timing_read(reset=True)
    l0 = W.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.take()
    sampler.active = True
    barrier()
    ev0.record(bench_stream)
    for _ in range(K):
        step_device()
    ev1.record(bench_stream)
    barrier()
    sampler.active = False
    launches = W.kernel_launches() - l0
    dev_ms = ev0.elapsed_time(ev1)
    W.synchronize()
    kinds = W.timing_read_kinds(reset=True)
    W.timing_enable(False)
    clocks_value = sampler.take()

    # ---- e2e: host buffers through the C-ABI ----
    for _ in range(max(Wm, 1)):
        step_e2e()
    barrier()
    sampler.active = True
    t0 = time.perf_counter()
    for _ in range(K):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    sampler.active = False
    clocks_e2e = sampler.take()
    if dec_out is not None:
        out_bytes = sum(t.numel() * 4 + p.numel() * 2 for t, p in dec_out)
        for c in calls:                                   # the parity gate needs the records: one untimed record step
            W.adapter_alignment_batch_multi(c, scoring)

    # ---- e2e with the NCCL re-gather of every rank's records to rank 0 (north star: "re-gather the output stream") ----
    gather_ms = None
    if world > 1 and main:
        from porechop_b200.distributed import gather_records
        counts = []
        for d in dev:
            c = [None] * world
            dist.all_gather_object(c, int(d[4].shape[0]))
            counts.append(c)
        hall = [pinned((sum(c), 9), torch.int32) if rank == 0 else None for c in counts]
        G = max(1, min(K, 3))

        def step_gather():
            with torch.cuda.stream(bench_stream):
                for (hb, ho, *_), (db, do, abuf, aoff, dout, max_len), c, ha in zip(host, dev, counts, hall):
                    db.copy_(hb, non_blocking=True)
                    do.copy_(ho, non_blocking=True)
                    W.adapter_alignment_batch_device(db.data_ptr(), do.data_ptr(), do.numel() - 1, db.numel(), max_len, abuf,
                                                     aoff, scoring, dout.data_ptr(), bench_stream.cuda_stream)
                    allrec = gather_records(dout, c, dst=0)
                    if allrec is not None:
                        ha.copy_(allrec, non_blocking=True)
            bench_stream.synchronize()
        step_gather()
        barrier()
        t0 = time.perf_counter()
        for _ in range(G):
            step_gather()
        barrier()
        gather_ms = (time.perf_counter() - t0) * 1e3 / G

    t = torch.tensor([dev_ms, e2e_s * 1e3, gather_ms or 0.0, float(workload.n), float(workload.cells), float(workload.alg_bytes),
                      float(in_bytes), float(out_bytes)], dtype=torch.float64, device='cuda')
    if world > 1:
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone()
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, gather_ms = float(tm[0]), float(tm[1]), float(tm[2])
        total_reads, total_cells = float(ts[3]), float(ts[4])
    else:
        e2e_ms = e2e_s * 1e3
        total_reads, total_cells = float(workload.n), float(workload.cells)
    res = {'host': host, 'dev': dev}
    if rank != 0:
        return None, res

    value = total_reads * K / (dev_ms / 1e3)
    e2e_value = total_reads * K / (e2e_ms / 1e3)
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    # dominant DP kernel of the step = the kind with the largest CUDA-event time (events recorded by the library around
    # every DP launch on the launching stream)
    dom = max(kinds, key=lambda k: kinds[k]['ms']) if kinds else None
    roof, alu = None, None
    sm_mhz = clocks_value.get('sm_mhz') or 1965.0
    if dom and kinds[dom]['n']:
        kd = kinds[dom]
        per_step_ms = kd['ms'] / K
        launch_ms = kd['ms'] / kd['n']
        launches_per_step = kd['n'] / K
        # what the dominant kind really processes: sequences up to direct_max take the single-pass trace kernel, longer ones
        # the score pass (+ a bounded window pass that reports its own cells) -- a mixed workload (the length sweep) must not
        # credit one kernel with the whole step
        dmax = W.get_option('direct_max')
        share_cells = share_bytes = 0.0
        for _, _, off, ads in workload.batches:
            lens = np.diff(np.asarray(off))
            sel = lens <= dmax if dom == 'trace_kernel' else lens > dmax
            if dom not in ('trace_kernel', 'score_kernel'):
                sel = np.ones(len(lens), dtype=bool)
            ad_bases = sum(len(a) for a in ads)
            share_cells += float(lens[sel].sum()) * ad_bases
            share_bytes += float(lens[sel].sum()) + (ad_bases if sel.any() else 0) + 36.0 * float(sel.sum()) * len(ads)
        frac_cells = share_cells / max(workload.cells, 1)
        bytes_per_launch = (share_bytes if share_cells else workload.alg_bytes) / launches_per_step
        achieved = bytes_per_launch / (launch_ms / 1e3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get(workload.name)
        except Exception:
            pass
        roof = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                'peak_source': peak_src, 'kernel': dom, 'launch_ms': launch_ms, 'launches_per_step': launches_per_step,
                'algorithmic_bytes_per_launch': bytes_per_launch,
                'kernels_ms_per_step': {k: v['ms'] / K for k, v in kinds.items()},
                'note': 'algorithmic bytes of the step (sum|H| + sum|V| + 36 B per alignment) / launches of the dominant kernel; '
                        'the kernel is integer-issue bound by construction (SURVEY 0.7): see roofline_alu'}
        sc = sass_counts().get(dom, {})
        cells_kernel = kd.get('cells') or workload.cells * K * (frac_cells if share_cells else 1.0)   # full-sweep kernels: every cell of their share
        cps = cells_kernel / (kd['ms'] / 1e3)
        if sc.get('instr_per_cell'):
            peak_cells = 148 * 4 * 32 * sm_mhz * 1e6 / sc['instr_per_cell']
            alu = {'kernel': dom, 'instr_per_cell': sc['instr_per_cell'], 'source': sc.get('source'),
                   'achieved_cells_per_s': cps, 'peak_cells_per_s': peak_cells, 'frac': cps / peak_cells, 'sm_mhz': sm_mhz,
                   'gcups_kernel': cps / 1e9, 'ms_per_step': per_step_ms}
        else:
            alu = {'kernel': dom, 'achieved_cells_per_s': cps, 'gcups_kernel': cps / 1e9, 'sm_mhz': sm_mhz,
                   'lane_instr_peak_per_s': 148 * 4 * 32 * sm_mhz * 1e6, 'ms_per_step': per_step_ms}
    line = {
        'metric': 'reads/sec', 'value': value, 'unit': 'reads/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': dev_ms / K, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
        'dtype': 'int16 (s16x2 DPX)', 'data': 'synthetic',
        'gcups': total_cells * K / (dev_ms / 1e3) / 1e9,
        'config': workload.config(args.scaling),
        'cells_per_read': workload.cells / max(workload.n, 1),
        'timing': {'l2': 'inputs %.0f MB per step and rank exceed the 126 MB L2' % (in_bytes / 1e6) if in_bytes > 126e6 else
                         'inputs %.0f MB per step' % (in_bytes / 1e6), 'clock': 'CUDA events on the launching stream (value), '
                   'host clock around synchronous C-ABI calls (e2e); max over ranks'},
        'e2e': {'value': e2e_value, 'unit': 'reads/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': out_bytes,
                'host_input_bytes_per_step': in_bytes,
                'upload': ('4-bit codes packed by %d host threads (h2d_pack=%d)' % (W.get_option('pack_threads'), W.get_option('h2d_pack')))
                          if packed_upload else 'ASCII bytes as they cross the ABI (h2d_pack=%d)' % W.get_option('h2d_pack'),
                'ms_per_step': e2e_ms / K, 'gcups': total_cells * K / (e2e_ms / 1e3) / 1e9,
                'path': ('adapterEndDecisions (host buffers, pinned), decisions come back' if dec_out is not None else
                         'adapterAlignmentBatchMulti (host buffers, pinned), %d submit(s) per step per rank' % len(calls)) +
                        '; records stay rank-local',
                'options': args.opt, 'ratio_to_value': e2e_value / value},
        'gpu_launches': int(launches),
        'roofline': roof, 'roofline_alu': alu,
        'clocks': clocks_value, 'clocks_e2e': clocks_e2e,
    }
    if gather_ms:
        line['e2e_with_gather'] = {'value': total_reads / (gather_ms / 1e3), 'unit': 'reads/s', 'ms_per_step': gather_ms,
                                   'path': 'per rank: pinned host -> device copy, adapterAlignmentBatchDevice, NCCL gather of the '
                                           '36-byte records to rank 0, rank 0 device -> host copy of all ranks\' records'}
    return line, res


def dump_outputs(out_dir, workload, dev):
    """The 9-int records the timed device-resident path left in its output buffers after its last step, one pair of
    float64 files per batch: <workload>_<batch>_records.npy [rows, 9] and <workload>_<batch>_rows.npy (the pair index of
    each row).  A batch larger than its share of DUMP_CAP_BYTES keeps a sample of rows drawn with a fixed seed."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    keep = DUMP_CAP_BYTES // len(dev) // (10 * 8)
    for (name, _, _, _), d in zip(workload.batches, dev):
        rec = d[4]
        n = rec.shape[0]
        rows = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        sel = rec.index_select(0, torch.from_numpy(rows).to(rec.device)).cpu().numpy()
        base = os.path.join(out_dir, '%s_%s' % (workload.name, name))
        np.save(base + '_records.npy', sel.astype(np.float64))
        np.save(base + '_rows.npy', rows.astype(np.float64))


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    from porechop_b200 import distributed as D
    numa = None
    all_cpus = os.sched_getaffinity(0)
    try:
        numa = D.bind_host_to_gpu(_pci_bus_id(local_rank), int(os.environ.get('LOCAL_WORLD_SIZE', world)), local_rank)
    except Exception:
        numa = None
    gpu_cpus = os.sched_getaffinity(0)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from porechop_b200 import cpp_function_wrappers as W
    for kv in args.opt:
        name, _, val = kv.partition('=')
        W.set_option(name, val)
    sampler = ClockSampler(local_rank)
    sampler.start()
    keep = []
    ctx = {'W': W, 'world': world, 'rank': rank, 'sampler': sampler, 'keep': keep, 'stream': torch.cuda.Stream()}

    def alloc(nbytes):
        t = torch.empty(int(nbytes), dtype=torch.uint8, pin_memory=True)
        keep.append(t)
        return t.numpy()

    def one(name, K, Wm, main):
        w = make_workload(name, args, rank, world, main, alloc=alloc)
        line, res = measure_gpu(w, args, ctx, K, Wm, main)
        if main and rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, w, res['dev'])
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                os.sched_setaffinity(0, all_cpus)          # the CPU baseline runs on ALL host cores, not the GPU's NUMA node
                try:
                    cb, answers, sizes = cpu_baseline(w, args.cpu_sample_reads if main else 0, sweep=main,
                                                      seconds=3.0 if main else 2.0)
                finally:
                    os.sched_setaffinity(0, gpu_cpus)
                line['cpu_baseline'] = cb
                # parity gate: the records the timed e2e steps left in the first output chunk vs the reference's strings
                recs = [h[5].numpy() for h in res['host']]
                line['parity'] = parity_gate(recs, answers, W.format_record)
                line['parity']['against'] = cb['kind']
            except Exception as e:
                line['parity'] = {'error': repr(e)}
        del res
        keep.clear()
        torch.cuda.empty_cache()
        return line

    line = one(args.workload, args.steps, args.warmup, True)
    others = [] if args.configs == 'none' else [c for c in (['demux', 'middle', 'sweep'] if args.configs == 'all' else args.configs.split(','))
                                                 if c and c != args.workload]
    cfgs = {}
    for name in others:
        try:
            sub = one(name, 2 if name != 'demux' else 1, 1, False)
        except Exception as e:                      # a failing side config must not lose the headline
            sub = {'error': repr(e)}
        if rank == 0:
            cfgs[name] = sub
    sampler.stop_flag = True
    if rank == 0:
        line['configs'] = cfgs
        line['numa'] = numa
        bad = [k for k, v in [('main', line)] + list(cfgs.items()) if isinstance(v, dict) and
               (v.get('parity', {}).get('mismatches') or 'error' in v.get('parity', {}) or 'error' in v)]
        if bad:
            line['invalid'] = 'parity gate failed / errored for: %s' % bad
        print(json.dumps(line))
        rc = 1 if bad else 0
    else:
        rc = 0
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return rc


def _pci_bus_id(index):
    import torch
    p = torch.cuda.get_device_properties(index)
    if hasattr(p, 'pci_bus_id') and hasattr(p, 'pci_device_id'):
        return '%04x:%02x:%02x.0' % (getattr(p, 'pci_domain_id', 0), p.pci_bus_id, p.pci_device_id)
    out = subprocess.check_output(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i', str(index)], timeout=20)
    return out.decode().strip()


# ------------------------------------------------------------------------------------------------------------------
def reference_cli_anchor():
    """BASELINE configs[0]: the unmodified reference CLI (staged copy baseline/_ref, oracle/Makefile `stage`) on
    test/test_one_adapter_set.fastq, --threads 1: wall seconds (correctness anchor; 9 reads)."""
    ref = os.path.join(ROOT, 'baseline', '_ref')
    runner, fq = os.path.join(ref, 'porechop-runner.py'), os.path.join(ref, 'test', 'test_one_adapter_set.fastq')
    if not (os.path.exists(runner) and os.path.exists(fq)):
        return {'unavailable': 'baseline/_ref not staged (make -C oracle stage, authoring container)'}
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, 'out.fastq')
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, runner, '-i', fq, '-o', out, '--threads', '1'], stdout=subprocess.DEVNULL,
                               stderr=subprocess.DEVNULL, env=dict(os.environ, PYTHONWARNINGS='ignore'))
            times.append(time.perf_counter() - t0)
            if r.returncode != 0:
                return {'unavailable': 'reference CLI exited %d' % r.returncode}
        n_out = sum(1 for _ in open(out)) // 4
    return {'workload': 'reference CLI, test/test_one_adapter_set.fastq, defaults, --threads 1', 'wall_s': min(times),
            'reads_in': 9, 'reads_out': n_out, 'reads_per_s': 9 / min(times)}


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return 0
    wl = _wl()
    cores = host_cores()
    harness, lib, kind = harness_paths()

    def one(name, K, Wm, main):
        # ~2 s of all-core work per step; the generators are prefix-consistent, so this is a prefix of the GPU arm's batch
        per_read = {'endtrim': 7500.0, 'demux': 150.0 * 17975, 'middle': 8040.0 * 50, 'sweep': 8000.0 * 4608}[name]
        limit = args.cpu_sample_reads or int(max(64, min(nominal_reads(name, args, main) or 1 << 30, 2.0 * 0.06e9 * cores / per_read)))
        w = make_workload(name, args, 0, 1, main, limit=limit)
        sizes = [len(off) - 1 for _, _, off, _ in w.batches]
        files = HarnessFiles(w, sizes)
        cells_per_read = w.cells / max(w.n, 1)
        # mode: threads in one process vs one process per core (separate heaps), best of a warm-up pair
        modes = [(cores, 1)] + ([(1, cores)] if cores >= 2 else []) + \
                ([(min(2 * cores, os.cpu_count() or cores), 1)] if 2 * cores <= (os.cpu_count() or cores) else [])
        trial = {m: files.run(*m) for m in modes}
        mode = min(trial, key=trial.get)
        times = []
        for s in range(Wm + K):
            sec = files.run(*mode)
            if s >= Wm:
                times.append(sec)
        t = float(np.mean(times))
        value = files.cells / t / cells_per_read
        nominal = make_nominal_config(name, args, main)
        one_t = HarnessFiles(w, [max(1, k // max(cores // 2, 1)) for k in sizes])
        sec1 = one_t.run(1)
        return {'impl': 'reference', 'metric': 'reads/sec', 'value': value, 'unit': 'reads/s', 'n_gpus': args.gpus,
                'steps': K, 'warmup': Wm, 'ms_per_step': t * 1e3, 'higher_is_better': True,
                'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'int32', 'data': 'synthetic',
                'gcups': files.cells / t / 1e9, 'config': nominal, 'cells_per_read': cells_per_read,
                'cpu_baseline': {'value': value, 'unit': 'reads/s', 'cores': mode[0] * mode[1], 'kind': kind,
                                 'mode': '%d threads x %d processes' % mode,
                                 'trial_seconds': {'%dx%d' % m: v for m, v in trial.items()},
                                 'one_thread': {'value': one_t.cells / sec1 / cells_per_read, 'unit': 'reads/s',
                                                'gcups': one_t.cells / sec1 / 1e9},
                                 'host': cpu_info(),
                                 'sample': 'first %s reads of the batches per step (%d alignments), native harness over the '
                                           'reference C-ABI' % (sizes, sum(k * len(b[3]) for k, b in zip(sizes, w.batches)))},
                'e2e': {'value': value, 'unit': 'reads/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}

    line = one(args.workload, args.steps, args.warmup, True)
    others = [] if args.configs == 'none' else [c for c in (['demux', 'middle', 'sweep'] if args.configs == 'all' else args.configs.split(','))
                                                 if c and c != args.workload]
    line['configs'] = {}
    for name in others:
        try:
            line['configs'][name] = one(name, 2, 1, False)
        except Exception as e:
            line['configs'][name] = {'error': repr(e)}
    line['configs']['cli_anchor'] = reference_cli_anchor()
    print(json.dumps(line))
    return 0


def make_nominal_config(name, args, main):
    """The `config` dict of Workload.config() without generating the batch (both arms must print identical dicts)."""
    wl = _wl()
    nom = nominal_reads(name, args, main)
    if name == 'endtrim':
        desc = '%d synthetic ~8kb reads (lognormal, seed %d+rank), SQK-NSK007 (LSK109 Y-adapter), end-trim: 150x28 + 150x22 per read' % (nom, wl.SEED)
        apr = 2
    elif name == 'demux':
        desc = '%d synthetic reads x 356 adapter sequences (119 sets + 12 native-full + 96 rapid-full: 227 start + 129 end), demux end windows' % nom
        apr = 356
    elif name == 'sweep':
        desc = 'read-length sweep %s x 192 forward barcode sequences (24 nt), %.1e bases per length, full-read scan' % (
            args.sweep_lengths, args.sweep_bases)
        apr = 192
        nom = sum(max(1, int(args.sweep_bases // int(x))) for x in args.sweep_lengths.split(','))
    else:
        desc = '%d synthetic full reads (~8 kb lognormal, 5%% chimeras) x {Y_Top, Y_Bottom}, middle-adapter scan' % nom
        apr = 2
    return {'workload': desc, 'reads_per_gpu' if args.scaling == 'weak' else 'reads_total': nom,
            'alignments_per_read': apr, 'scoring': list(wl.DEFAULT_SCORING), 'scaling': args.scaling}


def main():
    args = parse_args()
    if args.impl == 'reference':
        return run_reference(args)
    return run_b200(args)


if __name__ == '__main__':
    sys.exit(main())
