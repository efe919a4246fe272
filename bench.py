#!/usr/bin/env python3
"""bench.py -- mpileup reference positions/sec on the BASELINE workloads.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--region-mb M] [--modes a,b,...] [--dump-outputs DIR]
  (N>1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

ONE JSON line.  Its top-level keys are the headline workload; `modes` holds one sub-record per further
BASELINE configuration, each with its own value / roofline / cpu_baseline:

  (headline)     BASELINE config 2 shape x8: M Mb (default 8), 30x, 150 bp pairs, `mpileup -a`, no FASTA -> no BAQ
  mpileup_f_baq  the same window with its FASTA: `mpileup -f` = BAQ on every read (config 3's mode; bam_plcmd.c:1086,451)
  depth_a        `depth -a` over the same window                                     (config 5; bam2depth.c:209-477)
  coverage       `coverage` over the same window                                     (config 5; coverage.c:589-661)
  gl_c4          config 4 shape: 500 x 2 kb targets at 200x + 20 hotspots at 2000x -> genotype likelihoods per column
                 (bcf_call_glfgen + errmod_cal, bam2bcf.c:65-123)

A "step" is one pass of the hot path over one staged batch; inputs (0.05 GB/Mb) and outputs (0.08 GB/Mb) of a
step are far larger than the 126 MB L2, so successive steps cannot be served from cache.  With N GPUs every
rank owns its own region (weak scaling, no data-path collective; the one collective is the all_gather of the
per-region column summaries rank 0 needs to emit shards in genome order, issued once for all timed steps).
Every workload runs K timed steps.  Inputs are generated from fixed seeds, so the same arguments give the same
inputs on every run, and --dump-outputs lets two builds be compared output for output.

value  device-resident: inputs already staged in HBM; K x (read stage + column stage), max over ranks.
e2e    through the C ABI with HOST buffers: pinned-host SoA -> b200_stage (H2D + read stage) ->
       b200_mpileup_text -> pinned-host text (D2H), every step.
roofline  algorithmic bytes (SURVEY 8d) / CUDA-event time of the dominant kernel; BAQ: algorithmic non-fused
       FP64 operations (l_qseq x (2bw+1) x 53 per read) / CUDA-event time of the BAQ kernels.
cpu_baseline / --impl reference: the CPU oracle (the reference cannot be built here: htslib is absent,
       DESIGN.md) on the box's host cores -- as many processes as the scheduler affinity AND the cgroup CPU
       quota allow; the per-process and the single-process rates are reported next to the total so that a
       starved box is visible.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

METRIC = 'mpileup reference positions/sec'
UNIT = 'positions/s'
ALL_MODES = ('mpileup_f_baq', 'depth_a', 'coverage', 'gl_c4')
# nominal non-fused FP64 rate of a B200: 148 SMs x 64 FP64 lanes x 1.965 GHz (an FMA counts as ONE issue slot here
# because BAQ must not contract a*b+c); no driver-measured figure exists for this pipe
FP64_NONFMA_PEAK = 148 * 64 * 1.965e9


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def measured_traffic(kernels):
    """DRAM bytes per launch of the named kernels from the round's ncu capture (profiles/r02_traffic.json, written by
    tools/ncu_traffic.py) -- only while the kernel sources are the ones the capture was taken from; otherwise None."""
    p = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    try:
        import hashlib
        rec = json.load(open(p))
        h = hashlib.sha256()
        for s_ in rec['sources']:
            h.update(open(os.path.join(ROOT, s_), 'rb').read())
        if h.hexdigest() != rec['sources_sha256']:
            return None
        return float(sum(rec['dram_bytes_per_launch'][k] for k in kernels))
    except Exception:
        return None


def usable_cores():
    """CPUs this process may really use: scheduler affinity capped by the cgroup CPU quota."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()[:2]          # cgroup v2
        if q != 'max':
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())       # cgroup v1
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(quota)))
    return n, {'os_cpu_count': os.cpu_count(), 'sched_affinity': aff, 'cgroup_quota_cpus': quota}


def bind_to_gpu_numa(local):
    """Keep this rank's host threads -- and, by first touch, the pinned buffers they allocate -- on the NUMA node its GPU hangs
    off (8 ranks x 4 handles share two root complexes otherwise: the e2e leg of the 1->8 curve is PCIe/host-memory bound).
    Best effort: any missing piece (NVML, sysfs NUMA info, a cpuset that excludes the node) leaves the affinity untouched."""
    info = {'bound': False}
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        phys = int(vis.split(',')[local]) if vis and vis.split(',')[local].strip().isdigit() else local
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(':', 1)
        dev = os.path.join('/sys/bus/pci/devices', (dom[-4:] + ':' + rest).lower())
        node = int(open(os.path.join(dev, 'numa_node')).read())
        info['node'] = node
        if node < 0:
            return info
        cpus = set()
        for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        target = os.sched_getaffinity(0) & cpus
        info['cpus'] = len(target)
        if len(target) >= 8:
            os.sched_setaffinity(0, target)
            info['bound'] = True
    except Exception as e:                                      # noqa: BLE001 -- measurement aid only
        info['note'] = str(e)[:100]
    return info


class ClockSampler:
    """SM clock + throttle reasons of one GPU, polled through NVML every few ms while the timed
    regions run (the recipe's nvidia-smi query, without the process start-up latency)."""
    REASONS = (('hw_slowdown', 0x8), ('sw_power_cap', 0x4), ('sw_thermal_slowdown', 0x20), ('hw_thermal_slowdown', 0x40))

    def __init__(self, index, period=0.004):
        self.index, self.period, self.rows, self.stop = index, period, [], False
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[index]) if vis and vis.split(',')[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while not self.stop:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.h is not None:
            self.t = threading.Thread(target=self._poll, daemon=True); self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.h is not None:
            self.t.join(timeout=2)

    def summary(self):
        sm = [r[0] for r in self.rows]
        reasons = sorted({name for _, bits in self.rows for name, mask in self.REASONS if bits & mask})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': getattr(self, 'max_mhz', None), 'reasons': reasons,
                'samples': len(sm), 'source': 'nvml, polled during the timed regions'}


# ------------------------------------------------------------------------------------------------ CPU arm
def oracle_path():
    exe = os.path.join(ROOT, 'oracle', '_build', 'plp_oracle')
    if not os.path.exists(exe):
        subprocess.run(['make', '-s', '-C', os.path.join(ROOT, 'oracle')], check=True)
    return exe


class CpuSample:
    """A bounded sample of each workload for the CPU legs: a BGZF-compressed BAM (what `samtools mpileup` really reads,
    so the CPU arm pays BGZF inflate + BAM decode like the real tool) plus its FASTA."""

    def __init__(self, td, sample_mb=1.0):
        from samtools_b200 import synth
        self.td, self.mb = td, sample_mb
        n = int(sample_mb * 1e6)
        soa = synth.make_region(n, seed=99, chunk=500_000, with_ref=True)
        self.bam = os.path.join(td, 'sample.bam'); self.fa = os.path.join(td, 'sample.fa')
        synth.write_bam(self.bam, soa); synth.write_fasta(self.fa, soa['tid_name'], soa['ref_full'])
        self.ncols = n
        self.n_reads = len(soa['pos'])
        self._panel = None

    def panel(self):
        if self._panel is None:
            from samtools_b200 import synth
            p = synth.make_panel(n_targets=25, n_hot=1, seed=98)
            bam = os.path.join(self.td, 'panel.bam'); fa = os.path.join(self.td, 'panel.fa')
            synth.write_bam(bam, p); synth.write_fasta(fa, p['tid_name'], p['ref_full'])
            self._panel = (bam, fa, panel_columns(p))
        return self._panel

    def command(self, mode):
        """(argv after the oracle binary, units of work per run, description)"""
        if mode == 'mpileup_a':
            return ['mpileup', '-a', self.bam], self.ncols, f'`mpileup -a` over a {self.mb:g} Mb 30x/150bp BAM window'
        if mode == 'mpileup_f_baq':
            return ['mpileup', '-a', '-f', self.fa, self.bam], self.ncols, f'`mpileup -a -f` (BAQ) over a {self.mb:g} Mb 30x/150bp BAM window'
        if mode == 'depth_a':
            return ['depth', '-a', self.bam], self.ncols, f'`depth -a` over a {self.mb:g} Mb 30x/150bp BAM window'
        if mode == 'coverage':
            return ['coverage', self.bam], self.ncols, f'`coverage` over a {self.mb:g} Mb 30x/150bp BAM window'
        if mode == 'gl_c4':
            bam, fa, ncol = self.panel()
            return ['gl', '-B', '-f', fa, bam], ncol, 'genotype likelihoods (`gl -B -f`: glfgen + errmod_cal per column) over a 25-target 200x panel with one 2000x hotspot'
        raise ValueError(mode)


def panel_columns(p):
    """covered columns of a panel batch (what the GL path emits one record for): union of the reads' reference spans"""
    from samtools_b200 import synth
    pos = p['pos']; end = pos + synth.ref_span(p)
    hi = np.maximum.accumulate(end)
    starts = np.concatenate([[True], pos[1:] > hi[:-1]])
    seg_beg = pos[starts]
    seg_end = np.concatenate([hi[:-1][starts[1:]], hi[-1:]])
    return int((seg_end - seg_beg).sum())


def text_arrays(name, text, seed, runs=32, run_len=1 << 16, block=1 << 20):
    """A text output as arrays small enough to store: its length; two checksums per MiB over all of it (the byte sum and the
    sum weighted by the position in the MiB, both exact in float64); `runs` stretches of `run_len` bytes at seeded offsets,
    byte values as float32."""
    a = np.frombuffer(text, np.uint8)
    w = 1 + np.arange(block, dtype=np.int64) % 65521
    sums = np.zeros((-(-len(a) // block), 2), np.float64)
    for i in range(len(sums)):
        seg = a[i * block:(i + 1) * block].astype(np.int64)
        sums[i] = seg.sum(), seg @ w[:len(seg)]
    starts = np.sort(np.random.default_rng(seed).integers(0, max(1, len(a) - run_len + 1), runs))
    sample = np.concatenate([a[s:s + run_len] for s in starts]).astype(np.float32)
    return {f'{name}_length': np.array([len(a)], np.float64), f'{name}_checksums': sums, f'{name}_sample': sample}


def gl_arrays(name, pos, n, qs, p25, seed, rows=1 << 15):
    """Genotype-likelihood columns as arrays: per-field sums over every column (float64) and a seeded sample of columns."""
    k = len(pos)
    idx = np.sort(np.random.default_rng(seed).choice(k, min(k, rows), replace=False))
    sums = np.concatenate([[k, n.sum()], qs.reshape(k, -1).sum(0, dtype=np.float64), p25.reshape(k, -1).sum(0, dtype=np.float64)])
    return {f'{name}_sums': sums.astype(np.float64), f'{name}_pos': pos[idx].astype(np.float64), f'{name}_n': n[idx].astype(np.float64),
            f'{name}_qsum': qs[idx].astype(np.float32), f'{name}_p25': p25[idx].astype(np.float32)}


def write_dump(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(d, name + '.npy'), a)


def run_oracle_parallel(exe, argv, procs):
    t0 = time.perf_counter()
    ps = [subprocess.Popen([exe] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for _ in range(procs)]
    for p in ps:
        if p.wait() != 0:
            raise RuntimeError('oracle failed: ' + ' '.join(argv))
    return time.perf_counter() - t0


def cpu_leg(exe, sample, mode, procs, reps, warm):
    """`procs` concurrent single-threaded oracle processes (the reference pileup is single-threaded, bam_plcmd.c:1098; an
    all-cores run is region-sharded processes, SURVEY 8d), each over the whole sample; returns the cpu_baseline record."""
    argv, units, what = sample.command(mode)
    t1 = run_oracle_parallel(exe, argv, 1)                     # one process alone: the un-contended per-core rate
    for _ in range(warm):
        run_oracle_parallel(exe, argv, procs)
    t = [run_oracle_parallel(exe, argv, procs) for _ in range(reps)]
    total = sum(t)
    val = procs * units * reps / total
    return {'value': val, 'unit': UNIT, 'cores': procs, 'kind': 'port',
            'per_process': val / procs, 'one_process_alone': units / t1, 'parallel_efficiency': (val / procs) / (units / t1),
            'sample': f'{procs} concurrent single-threaded oracle processes, each {what} (BGZF inflate + BAM decode included) to /dev/null, '
                      f'{reps} timed rounds', 'seconds_per_round': total / reps}, total / reps


def reference_arm(args):
    """--impl reference: the CPU implementation of the path on all usable host cores (oracle port)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    exe = oracle_path()
    cores, how = usable_cores()
    modes = parse_modes(args)
    with tempfile.TemporaryDirectory() as td:
        sample = CpuSample(td, 1.0)
        head, sec = cpu_leg(exe, sample, 'mpileup_a', cores, args.steps, min(args.warmup, 1))
        sub = {}
        for m in modes:
            rec, _ = cpu_leg(exe, sample, m, cores, 2, 0)
            sub[m] = {'value': rec['value'], 'unit': UNIT, 'cpu_baseline': rec}
    head['core_accounting'] = how
    val = head['value']
    line = {'metric': METRIC, 'value': val, 'unit': UNIT, 'impl': 'reference', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1e3 * sec, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8',
            'data': 'synthetic', 'config': workload_config(args),
            'cpu_baseline': head,
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0, 'modes': sub}
    print(json.dumps(line))


def workload_config(args):
    return {'workload': f'BASELINE C2 shape x{args.region_mb:g}: synthetic {args.region_mb:g} Mb region per GPU, 30x depth, 150 bp paired reads, '
                        f'`mpileup -a` (no FASTA -> no BAQ, overlap removal on, -Q13, -d 8000)',
            'region_mb_per_gpu': args.region_mb, 'depth': 30, 'read_len': 150,
            'l2_policy': 'inputs (0.05 GB/Mb) and outputs (0.08 GB/Mb) per step exceed the 126 MB L2; no explicit flush',
            'parallelism': f'region-shard x{args.gpus}',
            'modes': 'sub-records: mpileup_f_baq (same window + FASTA, BAQ on), depth_a, coverage (same window), gl_c4 (200x panel with 2000x hotspots)'}


def parse_modes(args):
    if args.modes in ('', 'none'):
        return []
    if args.modes == 'all':
        return list(ALL_MODES)
    ms = [m for m in args.modes.split(',') if m]
    for m in ms:
        if m not in ALL_MODES:
            raise SystemExit(f'unknown mode {m}; choose from {ALL_MODES}')
    return ms


def pin(soa):
    """Keep the SoA arrays in pinned host memory so cudaMemcpyAsync runs at PCIe speed."""
    import torch
    out = dict(soa)
    for k, v in soa.items():
        if isinstance(v, np.ndarray) and v.nbytes > 0:
            t = torch.from_numpy(np.ascontiguousarray(v)).pin_memory()
            out[k] = t.numpy()
            out['_pin_' + k] = t
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--region-mb', type=float, default=8.0)
    ap.add_argument('--modes', default='all', help="comma list of extra workloads (%s), 'all' or 'none'" % ', '.join(ALL_MODES))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--e2e-handles', type=int, default=4,
                    help='engine handles (one host thread each) used by the end-to-end loop; handles are per-thread objects like the htslib iterators they replace')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last step of each workload returned to its caller as DIR/<name>.npy '
                         '(float32/float64; text outputs as length, per-MiB checksums and a seeded sample; rank 0 only)')
    args = ap.parse_args()
    if args.impl == 'reference':
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from samtools_b200 import engine, synth, shard

    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    numa = bind_to_gpu_numa(local) if world > 1 else {'bound': False, 'note': 'single rank: not bound'}
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the pileup engine has no CPU fallback)')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)
    modes = parse_modes(args)

    ncols = int(args.region_mb * 1e6)
    soa_ref = synth.make_region(ncols, seed=2 + rank, with_ref=True)          # this rank's region
    ref_arr = soa_ref['ref']
    soa = dict(soa_ref); soa['ref'] = None
    soa = pin(soa)
    n_reads = len(soa['pos'])
    h2d = int(sum(soa[k].nbytes for k in ('pos', 'flag', 'mapq', 'l_qseq', 'n_cigar', 'cigar_off', 'qual_off', 'mtid', 'mpos', 'isize',
                                          'prev_same_name', 'rbits', 'cigar', 'seq4', 'qual')))
    bytes_in = synth.algorithmic_bytes_in(soa, overlap=True)

    eng = engine.Engine(local)
    sconf = engine.default_stage_conf(engine.MODE_MPILEUP)
    mconf = engine.mpileup_conf(all=1)
    eng.stage(soa, sconf)
    out_len = eng.mpileup_text(mconf, fetch=False)
    out_host_t = torch.empty(out_len + 4096, dtype=torch.uint8).pin_memory()
    out_host = out_host_t.numpy()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # device-resident measurement: its own handle, with pristine qualities / mapq kept resident so that the read stage
    # (which edits them in place) can be repeated without the PCIe copies
    eng_dev = engine.Engine(local)
    eng_dev.set_keep_raw(True)
    eng_dev.stage(soa, sconf)
    stage_ms = []
    summaries = []

    def step_device():
        """the whole hot path on resident inputs: read stage (filters, overlap tweak, descriptors, read slices) + column stage"""
        eng_dev.restage()
        stage_ms.append(eng_dev.last_stage_device_ms)
        n = eng_dev.mpileup_text(mconf, fetch=False)
        summaries.append([n, ncols, n_reads])
        return n

    def exchange_summaries():
        """the path's one collective: per-region column summaries (bytes, columns, reads) of every step to every rank, so
        that rank 0 can emit the shards in genome order -- one all_gather for all the steps, not one per step"""
        if world > 1 and summaries:
            flat = [x for s in summaries for x in s]
            shard.gather_summaries(flat, device=dev)
        summaries.clear()

    # end-to-end: the caller owns a stream of windows; like htslib handles, an engine handle serves one
    # thread, so a pipeline uses one handle per host thread (H2D of one window overlaps kernels / D2H of another)
    import ctypes as C
    import threading as _th
    n_h = max(1, args.e2e_handles)
    handles = [eng] + [engine.Engine(local) for _ in range(n_h - 1)]
    outs = [out_host] + [torch.empty(out_len + 4096, dtype=torch.uint8).pin_memory().numpy() for _ in range(n_h - 1)]

    def one_window(h, buf):
        h.stage(soa, sconf)
        n = C.c_size_t(0)
        if h.lib.b200_mpileup_text(h.h, C.byref(mconf), buf.ctypes.data_as(C.c_void_p), buf.nbytes, C.byref(n)) != 0:
            raise RuntimeError(h.lib.b200_last_error(h.h).decode())
        return n.value

    def run_e2e(k_steps):
        """k_steps windows through n_h handles; returns the text bytes of each handle's last window"""
        res = [0] * n_h
        def worker(j):
            for s_ in range(j, k_steps, n_h):
                res[j] = one_window(handles[j], outs[j])
                summaries.append([res[j], ncols, n_reads])
        ths = [_th.Thread(target=worker, args=(j,)) for j in range(n_h)]
        [t.start() for t in ths]; [t.join() for t in ths]
        exchange_summaries()
        return res

    for _ in range(args.warmup):
        run_e2e(n_h); step_device()
    exchange_summaries()

    # ---- device-resident: K passes of read stage + column stage
    kernel_ms, parts_ms = [], []
    stage_ms.clear()
    with ClockSampler(local) as clk:
        sync_all()
        l0 = eng_dev.launches
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_device()
            kernel_ms.append(eng_dev.last_kernel_ms)
            parts_ms.append(eng_dev.last_mpileup_parts_ms)
        exchange_summaries()
        sync_all()
        dt = time.perf_counter() - t0
        launches = eng_dev.launches - l0
        # ---- end to end through the C ABI with host buffers
        sync_all()
        t0 = time.perf_counter()
        e2e_bytes = run_e2e(args.steps)
        sync_all()
        dt_e2e = time.perf_counter() - t0
    dump = {}
    if args.dump_outputs and rank == 0:
        last = (args.steps - 1) % n_h                 # the handle that ran the last timed window
        dump.update(text_arrays('mpileup_a_text', outs[last][:e2e_bytes[last]], seed=1))
    dt = shard.max_over_ranks(dt, dev); dt_e2e = shard.max_over_ranks(dt_e2e, dev)
    clocks = clk.summary()
    for h in handles[1:]:
        h.close()

    peak, peak_src = peaks()
    line = None
    if rank == 0:
        kms = float(np.mean(kernel_ms))
        size_ms, scan_ms, write_ms = [float(x) for x in np.mean(np.array(parts_ms), axis=0)]
        # column stage = entry pass (read-major: every read's bases -> 16-bit entries + the line-length sums) + tile scan + gather
        # (column-major: entries -> text).  The roofline names the slower of the two passes.  Algorithmic bytes (SURVEY 8d): the
        # gather consumes every read base once and writes every text byte once -> bytes_in + bytes_out; the entry pass reads the
        # staged reads once -> bytes_in (its entry strings are an intermediate, not algorithmic traffic)
        if write_ms >= size_ms:
            dom, alg, dom_ms, dom_k = 'k_mp_gather (entry strings -> text)', bytes_in + out_len, write_ms, ['k_mp_gather']
        else:
            dom, alg, dom_ms, dom_k = 'k_mp_entries + k_ss_scan + k_ss_cols (reads -> entry strings, line sizes)', bytes_in, size_ms, ['k_mp_entries', 'k_ss_scan', 'k_ss_cols']
        achieved = alg / (dom_ms * 1e-3) / 1e9
        traffic = measured_traffic(dom_k)                # from the round's ncu capture while the kernel sources are unchanged, else null
        value = world * ncols * args.steps / dt
        e2e = world * ncols * args.steps / dt_e2e
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8',
                'data': 'synthetic', 'config': workload_config(args), 'clocks': clocks,
                'e2e': {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': int(out_len), 'ms_per_step': 1e3 * dt_e2e / args.steps,
                        'handles': n_h},
                'gpu_launches': int(launches),
                'roofline': {'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                             'traffic': traffic, 'peak_source': peak_src, 'algorithmic_bytes_per_launch': int(alg),
                             'bytes_in': int(bytes_in), 'bytes_out': int(out_len), 'kernel_ms': dom_ms,
                             'step_kernels_ms': {'read_stage': float(np.mean(stage_ms)), 'entry_pass': size_ms, 'tile_offset_scan': scan_ms,
                                                 'gather': write_ms, 'column_stage_total': kms, 'total': kms + float(np.mean(stage_ms))},
                             'step_frac': (bytes_in + out_len) / ((kms + float(np.mean(stage_ms))) * 1e-3) / 1e9 / peak},
                'reads_per_step_per_gpu': n_reads, 'numa': numa}

    # ------------------------------------------------------------------------------------ further BASELINE configurations
    sub = {}
    msteps = args.steps

    def timed(fn, k, w=2):
        for _ in range(w):
            fn()
        sync_all()
        t0_ = time.perf_counter()
        for _ in range(k):
            fn()
        sync_all()
        return shard.max_over_ranks(time.perf_counter() - t0_, dev)

    if 'mpileup_f_baq' in modes:
        soa_b = dict(soa); soa_b['ref'] = ref_arr
        e = engine.Engine(local); e.set_keep_raw(True)
        bconf = engine.default_stage_conf(engine.MODE_MPILEUP)
        e.stage(soa_b, bconf)
        blen = e.mpileup_text(mconf, fetch=False)
        baq_ms, st_ms, k_ms = [], [], []

        def step_baq():
            e.restage(); baq_ms.append(e.last_baq_ms); st_ms.append(e.last_stage_device_ms)
            e.mpileup_text(mconf, fetch=False); k_ms.append(e.last_kernel_ms)
        dtb = timed(step_baq, msteps, w=1)
        l = soa['l_qseq'].astype(np.int64)
        ops = float((l * 15 * 53).sum())                       # SURVEY 8d: l_qseq x (2bw+1) x (fwd 22 + bwd 25 + MAP 6), bw = 7
        bms = float(np.mean(baq_ms[-msteps:]))
        ach = ops / (bms * 1e-3)
        sub['mpileup_f_baq'] = {
            'workload': f'same {args.region_mb:g} Mb window with its FASTA: `mpileup -a -f` (BAQ = sam_prob_realn on every read, overlap removal, -Q13)',
            'value': world * ncols * msteps / dtb, 'unit': UNIT, 'ms_per_step': 1e3 * dtb / msteps, 'steps': msteps, 'bytes_out': int(blen),
            'reads_per_s_baq_kernels': n_reads / (bms * 1e-3),
            'roofline': {'bound': 'fp64 (non-fused: BAQ must not contract a*b+c)', 'kernel': 'BAQ kernels (k_baq_plan + k_baq_reg)', 'achieved': ach / 1e12,
                         'peak': FP64_NONFMA_PEAK / 1e12, 'unit': 'Top/s (FP64, non-FMA)', 'frac': ach / FP64_NONFMA_PEAK,
                         'peak_source': 'nominal: 148 SMs x 64 FP64 lanes x 1.965 GHz (no measured FP64 figure in MEASURED_PEAKS.json)',
                         'algorithmic_ops_per_launch': ops, 'kernel_ms': bms, 'traffic': None,
                         'step_kernels_ms': {'read_stage_total': float(np.mean(st_ms[-msteps:])), 'of_which_baq': bms, 'column_stage': float(np.mean(k_ms[-msteps:]))}}}
        if args.dump_outputs and rank == 0:           # the column stage again on the last step's staged reads: same bytes
            dump.update(text_arrays('mpileup_f_baq_text', e.mpileup_text(mconf), seed=2))
        e.close()

    if 'depth_a' in modes or 'coverage' in modes:
        e = engine.Engine(local); e.set_keep_raw(True)
        if 'depth_a' in modes:
            dconf = engine.default_stage_conf(engine.MODE_DEPTH)
            e.stage(soa, dconf)
            dlen = e.depth_text(all=1, fetch=False)
            k_ms, st_ms = [], []

            def step_depth():
                e.restage(); st_ms.append(e.last_stage_device_ms)
                e.depth_text(all=1, fetch=False); k_ms.append(e.last_kernel_ms)
            dtd = timed(step_depth, msteps)
            din = int((4 * soa['n_cigar'].astype(np.int64) + 24).sum())          # SURVEY 8d: depth needs no bases / qualities at -q 0
            kd = float(np.mean(k_ms[-msteps:]))
            sub['depth_a'] = {'workload': f'`depth -a` over the same {args.region_mb:g} Mb window (BASELINE config 5)',
                              'value': world * ncols * msteps / dtd, 'unit': UNIT, 'ms_per_step': 1e3 * dtd / msteps, 'steps': msteps, 'bytes_out': int(dlen),
                              'roofline': {'bound': 'hbm', 'kernel': 'k_depth_size + scan + k_depth_write', 'achieved': (din + dlen) / (kd * 1e-3) / 1e9, 'peak': peak,
                                           'unit': 'GB/s', 'frac': (din + dlen) / (kd * 1e-3) / 1e9 / peak, 'peak_source': peak_src,
                                           'algorithmic_bytes_per_launch': int(din + dlen), 'kernel_ms': kd, 'traffic': None,
                                           'step_kernels_ms': {'read_stage': float(np.mean(st_ms[-msteps:])), 'column_stage': kd}}}
            if args.dump_outputs and rank == 0:
                dump.update(text_arrays('depth_a_text', e.depth_text(all=1), seed=3))
        if 'coverage' in modes:
            cconf = engine.default_stage_conf(engine.MODE_COVERAGE, rflag_filter=4 | 256 | 512 | 1024, end=ncols)
            e.stage(soa, cconf)
            k_ms, st_ms = [], []
            cov = {}

            def step_cov():
                st = e.restage(); st_ms.append(e.last_stage_device_ms)
                cov.update(e.coverage(min_baseQ=0, min_depth=1), n_selected_reads=st.n_selected_reads, summed_mapq=st.summed_mapq)
                k_ms.append(e.last_kernel_ms)
            dtc = timed(step_cov, msteps)
            if args.dump_outputs and rank == 0:
                dump['coverage_sums'] = np.array(list(cov.values()), np.float64)
            cin = int((soa['l_qseq'].astype(np.int64) + 4 * soa['n_cigar'].astype(np.int64) + 24).sum())   # qualities + cigar + core fields
            kc = float(np.mean(k_ms[-msteps:]))
            sub['coverage'] = {'workload': f'`coverage` over the same {args.region_mb:g} Mb window (BASELINE config 5)',
                               'value': world * ncols * msteps / dtc, 'unit': UNIT, 'ms_per_step': 1e3 * dtc / msteps, 'steps': msteps,
                               'roofline': {'bound': 'hbm', 'kernel': 'k_coverage', 'achieved': cin / (kc * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                                            'frac': cin / (kc * 1e-3) / 1e9 / peak, 'peak_source': peak_src, 'algorithmic_bytes_per_launch': cin, 'kernel_ms': kc,
                                            'traffic': None, 'step_kernels_ms': {'read_stage': float(np.mean(st_ms[-msteps:])), 'column_stage': kc}}}
        e.close()

    if 'gl_c4' in modes:
        panel = synth.make_panel(seed=4 + rank)                   # 500 x 2 kb at 200x, 20 hotspots at 2000x
        pcols = panel_columns(panel)
        pp = pin(panel)
        e = engine.Engine(local); e.set_keep_raw(True)
        gconf = engine.default_stage_conf(engine.MODE_MPILEUP, baq=0)
        e.stage(pp, gconf)
        k_ms, st_ms = [], []

        def step_gl():
            e.restage(); st_ms.append(e.last_stage_device_ms)
            e.glf(13, 0, fetch=False); k_ms.append(e.last_kernel_ms)
        dtg = timed(step_gl, msteps, w=1)
        gin = synth.algorithmic_bytes_in(panel, overlap=True)
        gout = pcols * (25 * 4 + 16)
        kg = float(np.mean(k_ms[-msteps:]))
        sub['gl_c4'] = {'workload': 'BASELINE config 4 shape: 500 targets x 2 kb at 200x, 20 hotspots at 2000x (%d reads, %d covered columns), '
                                    '`mpileup -B` read stage -> bcf_call_glfgen + errmod_cal per column, likelihoods left in HBM' % (len(panel['pos']), pcols),
                        'value': world * pcols * msteps / dtg, 'unit': 'columns/s', 'ms_per_step': 1e3 * dtg / msteps, 'steps': msteps,
                        'roofline': {'bound': 'hbm', 'kernel': 'k_gl_count + scan + k_gl', 'achieved': (gin + gout) / (kg * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                                     'frac': (gin + gout) / (kg * 1e-3) / 1e9 / peak, 'peak_source': peak_src, 'algorithmic_bytes_per_launch': int(gin + gout),
                                     'kernel_ms': kg, 'traffic': None, 'step_kernels_ms': {'read_stage': float(np.mean(st_ms[-msteps:])), 'column_stage': kg}}}
        e.close()
        if args.dump_outputs and rank == 0:
            # errmod_cal's shuffle draws from one random stream that runs on across calls, so a fresh handle makes as many calls
            # as preceded the last timed step (one warm-up, msteps - 1 timed) before it fetches that step's columns
            r = engine.Engine(local); r.set_keep_raw(True)
            st = r.stage(pp, gconf)
            for _ in range(msteps):
                r.restage(); r.glf(13, 0, fetch=False)
            r.restage()
            dump.update(gl_arrays('gl_c4', *r.glf(13, int(st.n_cols) + 16), seed=4))
            r.close()

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            exe = oracle_path()
            with tempfile.TemporaryDirectory() as td:
                sample = CpuSample(td, 1.0)
                rec, _ = cpu_leg(exe, sample, 'mpileup_a', 1, 4, 0)
                line['cpu_baseline'] = rec
                for m in sub:
                    rec, _ = cpu_leg(exe, sample, m, 1, 1, 0)
                    sub[m]['cpu_baseline'] = rec
        line['modes'] = sub
        if args.dump_outputs:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line))
    eng.close(); eng_dev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
