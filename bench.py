#!/usr/bin/env python
"""bench.py -- resquiggle throughput of the B200-native hot path.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W

One step = one pass of the hot path (normalise -> segment -> banded DP -> skipped
bases -> Theil-Sen rescale -> score, incl. the iterate / rescue policy) over one
batch of synthetic reads.  Headline workload at N = 1: BASELINE.json configs[1] (100k
synthetic DNA reads, ~4k samples, bandwidth 200, default start parameters -> every
read takes the static-band path, W ~ 748).  For N > 1 every rank runs its own batch
of the same size (reads shard with no collective; "scaling": "weak").

Printed JSON (rank 0): `value` = reads/s with inputs resident in HBM (device time, CUDA
events on the library's stream), `e2e` = the same through tb2_resquiggle_batch with pinned
HOST buffers (H2D + D2H inside the timed region), `roofline` for the dominant kernel
(k_align, the banded DP), `cpu_baseline` = the reference's own code (oracle/_ref) -- or the
C port when that is absent -- timed in a clean interpreter BEFORE any CUDA call, single
process and all cores, `parity` = a random sample of the timed batch bit-compared with the
oracle after the timed regions, and (N = 1) `extra_configs`: the same fields for the other
BASELINE.json shapes (configs[2] mixed 2k-20k / bw 400 + rescue, configs[3] direct RNA 8k +
5mC LLR + per-position counts, configs[4] 50k samples / bw 1200 + forced-rescue subset).

    python bench.py --workload mixed --queue --reads R       strong scaling over a shared
                                                             NCCL-free queue of length buckets

`--dump-outputs DIR` writes what the last resident timed step computed for every workload run
(a seeded sample of its reads) as DIR/<workload>_<field>.npy in float64; the inputs depend only
on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the tree may be read-only and is never written: no bytecode caches next to the sources
sys.dont_write_bytecode = True

# the CPU arms run one single-threaded worker process per host thread (the reference's
# --processes model): keep BLAS / OpenMP pools from oversubscribing the cores
for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMEXPR_NUM_THREADS'):
    os.environ.setdefault(_v, '1')

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

ALN_DNA = (4.2, 4.2, 200, 1500, 20.0, 40, 750, 2500, 250)     # configs[1]: bandwidth = 200
ALN_MIXED = (4.2, 4.2, 400, 1500, 20.0, 40, 750, 2500, 250)   # configs[2]: bandwidth = 400
ALN_C5 = (4.2, 4.2, 1200, 1500, 20.0, 40, 750, 2500, 250)     # configs[4]: bandwidth = 1200
ALN_RNA = (6, 4, 500, 1500, 20.0, 50, 1000, 3000, 250)        # RNA defaults
SEG_DNA = (5, 3, 1, 5)
SEG_RNA = (12, 6, 2, 15)
N_BASES = 444          # ~4k raw samples at 9 samples / base (+150 leader)
METRIC = 'resquiggle_reads_per_sec'

CONFIGS = {
    'c1': dict(kind='DNA', aln=ALN_DNA, seg=SEG_DNA, nbases=N_BASES, reads=100000, parity=1024,
               cpu_single=48, cpu_pool_per_core=96,
               label='configs[1]: %d synthetic DNA reads/GPU x ~4k samples (444 bases, 6-mer '
                     'model), bandwidth=200, default start params => static-band path W~748, '
                     'float64 raw'),
    'mixed': dict(kind='DNA', aln=ALN_MIXED, seg=SEG_DNA, nbases='mixed', reads=40000, parity=512,
                  cpu_single=8, cpu_pool_per_core=4,
                  label='configs[2]-like: %d synthetic DNA reads/GPU, 2k-20k samples (222-2222 '
                        'bases), bandwidth=400 adaptive band + save-bandwidth rescue, float64 raw'),
    'rna': dict(kind='RNA', aln=ALN_RNA, seg=SEG_RNA, nbases=270, reads=20000, parity=512, llr=True,
                cpu_single=8, cpu_pool_per_core=8,
                label='configs[3]: %d synthetic direct-RNA reads/GPU x ~8k samples (270 bases, '
                      '5-mer model), RNA defaults (bw 500, t-test segmentation, stalls) + 5mC '
                      'alt-model per-read LLR + per-position counts, float64 raw'),
    'c5': dict(kind='DNA', aln=ALN_C5, seg=SEG_DNA, nbases=5555, reads=6000, parity=64,
               stall_every=20, stall_extra=11000, cpu_single=2, cpu_pool_per_core=1,
               label='configs[4]: %d synthetic DNA reads/GPU x ~50k samples (5555 bases), '
                     'bandwidth=1200, every 20th read carries an 11k-sample stall (forced '
                     'save-bandwidth rescue), float64 raw'),
}


class RP(object):
    def __init__(self, aln=ALN_DNA, seg=SEG_DNA, save=False, rna=False):
        (self.match_evalue, self.skip_pen, bw, sbw, self.max_half_z_score,
         self.band_bound_thresh, self.start_bw, self.start_save_bw, self.start_n_bases) = aln
        self.bandwidth = sbw if save else bw
        (self.running_stat_width, self.min_obs_per_base, self.raw_min_obs_per_base,
         self.mean_obs_per_event) = seg
        self.z_shift = float(np.sqrt(2.0 / np.pi)) + self.match_evalue
        self.stay_pen = self.match_evalue
        self.use_t_test_seg = rna


def host_info():
    """what the CPU numbers were measured on: affinity, cgroup quota, physical cores, load"""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    for p in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(p).read().split()
            if p.endswith('cpu.max'):
                if txt[0] != 'max':
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            break
        except Exception:
            continue
    phys, model = None, None
    try:
        pairs, pid = set(), None
        for line in open('/proc/cpuinfo'):
            if line.startswith('physical id'):
                pid = line.split(':')[1].strip()
            elif line.startswith('core id'):
                pairs.add((pid, line.split(':')[1].strip()))
            elif line.startswith('model name') and model is None:
                model = line.split(':', 1)[1].strip()
        phys = len(pairs) or None
    except Exception:
        pass
    try:
        load = list(os.getloadavg())
    except Exception:
        load = None
    usable = aff if quota is None else max(1, min(aff, int(quota)))
    return {'affinity_cpus': aff, 'cgroup_cpu_quota': quota, 'physical_cores': phys,
            'cpu_model': model, 'loadavg': load, 'usable': usable}


def host_cores():
    return host_info()['usable']


def peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, device):
        self.device = device
        self.samples = []
        self.err = ''
        self._nvml = self._nvml_open()
        self._stop = threading.Event()
        self._t = None

    def _nvml_open(self):
        """NVML handle of this rank's GPU (opened before the timed region); None if unavailable"""
        for attempt in range(3):
            try:
                import pynvml as nv
                nv.nvmlInit()
                vis = os.environ.get('CUDA_VISIBLE_DEVICES')
                h = None
                if vis:
                    ents = [e.strip() for e in vis.split(',')]
                    ent = ents[self.device] if self.device < len(ents) else ''
                    try:
                        h = nv.nvmlDeviceGetHandleByIndex(int(ent))
                    except Exception:
                        try:
                            h = nv.nvmlDeviceGetHandleByUUID(ent.encode())
                        except Exception:
                            h = None
                if h is None:
                    h = nv.nvmlDeviceGetHandleByIndex(self.device)
                mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
                get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                    getattr(nv, 'nvmlDeviceGetCurrentClocksThrottleReasons')
                nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                get_reasons(h)
                return nv, h, mx, get_reasons
            except Exception as e:
                self.err = 'nvml: %r' % (e,)
                time.sleep(0.05 * (attempt + 1))
        return None

    def _run_nvml(self):
        """NVML in-process (tens of samples per timed region); False if unavailable"""
        if self._nvml is None:
            return False
        nv, h, mx, get_reasons = self._nvml
        bits = ((0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5))   # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = int(get_reasons(h))
                rec = [sm, mx, 'Not Active', 'Not Active', 'Not Active', 'Not Active']
                for bit, pos in bits:
                    if r & bit:
                        rec[pos] = 'Active'
                self.samples.append(tuple(rec))
            except Exception as e:
                self.err = 'nvml sample: %r' % (e,)
            self._stop.wait(0.02)
        return bool(self.samples)

    def _run(self):
        if self._run_nvml():
            return
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        while not self._stop.is_set():
            try:
                o = subprocess.run(['nvidia-smi', '-i', str(self.device), '--query-gpu=' + q,
                                    '--format=csv,noheader,nounits'], capture_output=True,
                                   text=True, timeout=5).stdout.strip().split('\n')[0]
                f = [x.strip() for x in o.split(',')]
                self.samples.append((float(f[0]), float(f[1]), f[2], f[3], f[4], f[5]))
            except Exception as e:
                self.err += ' nvidia-smi: %r' % (e,)
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable'], 'error': self.err[:300]}
        sm = sorted(s[0] for s in self.samples)
        reasons = []
        for name, idx in (('hw_slowdown', 2), ('hw_thermal_slowdown', 3),
                          ('sw_thermal_slowdown', 4), ('sw_power_cap', 5)):
            if any(s[idx] == 'Active' for s in self.samples):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': self.samples[0][1],
                'reasons': reasons, 'samples': len(self.samples)}


# ---------------------------------------------------------------------------
# synthetic workload
# ---------------------------------------------------------------------------
def workload_nbases(cfg, n, seed, ci):
    if cfg['nbases'] == 'mixed':          # configs[2]: 2k-20k raw samples per read
        return np.random.RandomState((seed * 7919 + ci) % (2 ** 32)).randint(222, 2223, n)
    return cfg['nbases']


def make_workload(cfg, n_reads, seed, pinned_factory=None):
    from tombo_b200 import synthetic as syn
    kmer_ref, cpos = syn.make_kmer_ref(cfg['kind'], 0)
    chunks, offs, seqs, soffs = [], [0], [], [0]
    done, ci = 0, 0
    per = 10000 if cfg['nbases'] != 5555 else 500
    while done < n_reads:
        m = min(per, n_reads - done)
        raw, ro, codes, so = syn.make_read_batch(
            kmer_ref, m, workload_nbases(cfg, m, seed, ci), seed * 1000 + ci, kind=cfg['kind'],
            stall_every=cfg.get('stall_every', 0), stall_extra=cfg.get('stall_extra', 0))
        chunks.append(raw); seqs.append(codes)
        offs.extend((ro[1:] + offs[-1]).tolist())
        soffs.extend((so[1:] + soffs[-1]).tolist())
        done += m; ci += 1
    raw_off = np.array(offs, dtype=np.int64)
    seq_off = np.array(soffs, dtype=np.int64)
    total = int(raw_off[-1])
    raw = pinned_factory(total, np.float64) if pinned_factory is not None else np.empty(total)
    p = 0
    for c in chunks:
        raw[p:p + c.shape[0]] = c
        p += c.shape[0]
    seq = np.concatenate(seqs)
    return kmer_ref, cpos, raw, raw_off, seq, seq_off


def dp_algorithmic_bytes(raw_off, seq_off, k, rp):
    """SURVEY.md 8(d): A_dp = 8*E + 16*B + 8*B + 8*(B+1) + ceil(2*C/8) per read
    (event means in, levels in, band starts + traceback out, 2-bit moves leaving
    the chip); C = band cells of the read's path."""
    s = (raw_off[1:] - raw_off[:-1]).astype(np.int64)
    b = (seq_off[1:] - seq_off[:-1]).astype(np.int64) - (k - 1)
    e = np.maximum(s // rp.mean_obs_per_event, (b * 1.1).astype(np.int64))
    n_em = e - 1
    mask = np.minimum(b, n_em) // 4
    w = n_em - mask
    short = (n_em < rp.start_bw + rp.start_n_bases) | (b < rp.start_n_bases)
    # long reads: start search (start_n_bases x start_bw) + one band row per base
    cells = np.where(short, b * w, rp.start_n_bases * rp.start_bw + b * rp.bandwidth)
    a = 8 * e + 16 * b + 8 * b + 8 * (b + 1) + (2 * cells + 7) // 8
    return a.astype(np.float64), cells.astype(np.float64)


def alt_table(kmer_ref):
    from tombo_b200 import synthetic as syn
    k = len(kmer_ref[0][0])
    alt = np.full((4 ** k, k), np.nan)
    code = {'A': 0, 'C': 1, 'G': 2, 'T': 3}
    for km, pos, m, sd in syn.make_alt_kmer_ref(kmer_ref, 'C', seed=1):
        idx = 0
        for b in km:
            idx = idx * 4 + code[b]
        alt[idx, pos] = m
    return alt


# ---------------------------------------------------------------------------
# CPU baseline: the reference's own implementation on the host cores, in a clean
# interpreter (no CUDA context, no pinned memory in the parent to fork)
# ---------------------------------------------------------------------------
_W = {}


def _cpu_init(kind, names):
    sys.path.insert(0, os.path.join(REPO, 'oracle'))
    from tombo_b200 import synthetic as syn
    _W['kind'] = kind
    for name in names:
        cfg = CONFIGS[name]
        kmer_ref, cpos = syn.make_kmer_ref(cfg['kind'], 0)
        w = {'kmer_ref': kmer_ref, 'cpos': cpos}
        rna = cfg['kind'] == 'RNA'
        if kind == 'reference':
            import ref_harness as rh
            w['rh'] = rh
            w['std_ref'], _ = rh.make_models(kmer_ref, cpos)
            w['sst'], w['p'], w['sp'] = rh.make_params(cfg['kind'], cfg['aln'])
        else:
            import oracle as orc
            w['orc'] = orc
            w['means'], w['sds'] = syn.kmer_table(kmer_ref)
            w['p'] = RP(cfg['aln'], cfg['seg'], rna=rna)
            w['sp'] = RP(cfg['aln'], cfg['seg'], save=True, rna=rna)
            w['pol'] = orc.policy(cfg['kind'])
        _W[name] = w


def _cpu_one(job):
    name, seed = job
    from tombo_b200 import synthetic as syn
    cfg, w = CONFIGS[name], _W[name]
    nb = workload_nbases(cfg, 1, seed, 0)
    nb = int(nb[0]) if not np.isscalar(nb) else int(nb)
    stall = None
    if cfg.get('stall_every') and seed % cfg['stall_every'] == cfg['stall_every'] - 1:
        stall = (nb // 2, cfg['stall_extra'])
    r = syn.make_read(w['kmer_ref'], w['cpos'], nb, seed, kind=cfg['kind'], stall=stall)
    t0 = time.perf_counter()
    if _W['kind'] == 'reference':
        res, err, info = w['rh'].run_read(r.raw, r.genome_seq, w['std_ref'], w['sst'], w['p'],
                                          w['sp'], read_index=seed)
        ok = res is not None
    else:
        k = len(w['kmer_ref'][0][0])
        rm, rs = w['orc'].levels_from_codes(syn.seq_to_codes(r.genome_seq), w['means'], w['sds'], k)
        o = w['orc'].run_read(np.asarray(r.raw, dtype=np.float64), rm, rs, w['p'], w['sp'],
                              w['pol'], read_index=seed)
        ok = o['status'] == 0
    return time.perf_counter() - t0, r.raw.shape[0], ok


def cpu_baseline_kind():
    sys.path.insert(0, os.path.join(REPO, 'oracle'))
    try:
        import ref_harness as rh
        if rh.available():
            return 'reference'
    except Exception:
        pass
    return 'port'


def _summ(out, wall, n):
    samples = sum(o[1] for o in out)
    return {'reads_per_s': n / wall, 'samples_per_s': samples / wall, 'wall_s': wall,
            'ok': int(sum(o[2] for o in out)), 'n': n,
            'per_read_core_ms': 1e3 * sum(o[0] for o in out) / n}


def cpu_leg(names, cores, kind, steps=1, warmup_reads=2, scale=1.0):
    """single-process and Pool(cores) reads/s of the CPU implementation for each config
    (multiprocessing.Pool == the compute half of the reference's --processes)."""
    import multiprocessing as mp
    res = {'host': host_info(), 'kind': kind, 'cores': cores}
    _cpu_init(kind, names)
    for name in names:                       # single process: BASELINE.json configs[0] style
        cfg = CONFIGS[name]
        for s in range(warmup_reads):
            _cpu_one((name, 898000 + s))
        n = max(1, int(cfg['cpu_single'] * scale))
        t0 = time.perf_counter()
        out = [_cpu_one((name, 899000 + i)) for i in range(n)]
        res.setdefault(name, {})['single'] = _summ(out, time.perf_counter() - t0, n)
    pool = mp.get_context('fork').Pool(cores, initializer=_cpu_init, initargs=(kind, names))
    try:
        pool.map(_cpu_one, [(names[0], 897000 + i) for i in range(cores)])      # import + warm-up
        for name in names:
            cfg = CONFIGS[name]
            n = max(cores, int(cores * cfg['cpu_pool_per_core'] * scale))
            runs = []
            for st in range(steps):
                jobs = [(name, 900000 + 7919 * st + i) for i in range(n)]
                t0 = time.perf_counter()
                out = pool.map(_cpu_one, jobs, chunksize=max(1, n // (cores * 8)))
                runs.append(_summ(out, time.perf_counter() - t0, n))
            tot_n = sum(r['n'] for r in runs)
            tot_w = sum(r['wall_s'] for r in runs)
            agg = {'reads_per_s': tot_n / tot_w,
                   'samples_per_s': sum(r['samples_per_s'] * r['wall_s'] for r in runs) / tot_w,
                   'wall_s': tot_w, 'ok': sum(r['ok'] for r in runs), 'n': tot_n,
                   'per_read_core_ms': sum(r['per_read_core_ms'] * r['n'] for r in runs) / tot_n,
                   'steps': steps}
            res[name]['pool'] = agg
    finally:
        pool.close(); pool.join()
    res['host_after'] = host_info()
    return res


def cpu_leg_subprocess(names, steps=1, scale=1.0):
    """run cpu_leg in a fresh interpreter: no CUDA context or pinned pages in the process
    that forks the worker pool (round 1's in-process leg was 3-10x slower than the
    --impl reference arm on the same box for that reason)"""
    cmd = [sys.executable, os.path.abspath(__file__), '--cpu-leg', ','.join(names),
           '--steps', str(steps), '--cpu-scale', str(scale)]
    o = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    for line in reversed(o.stdout.strip().splitlines()):
        if line.startswith('{'):
            return json.loads(line)
    raise RuntimeError('cpu leg failed: ' + o.stderr[-800:])


def cpu_baseline_obj(leg, name):
    c = leg[name]
    h = leg['host']
    return {'value': c['pool']['reads_per_s'], 'unit': 'reads/s', 'cores': leg['cores'],
            'kind': leg['kind'], 'samples_per_sec': c['pool']['samples_per_s'],
            'per_read_core_ms': c['pool']['per_read_core_ms'],
            'single_process': {'value': c['single']['reads_per_s'], 'unit': 'reads/s',
                               'per_read_ms': c['single']['per_read_core_ms'],
                               'n': c['single']['n']},
            'host': {k: h[k] for k in ('affinity_cpus', 'cgroup_cpu_quota', 'physical_cores',
                                       'cpu_model', 'loadavg')},
            'sample': '%d reads of the same workload, Pool(%d) over resquiggle_read + '
                      'iterate/rescue policy, %.1f s wall; single process: %d reads; clean '
                      'interpreter before any CUDA call'
                      % (c['pool']['n'], leg['cores'], c['pool']['wall_s'], c['single']['n'])}


# ---------------------------------------------------------------------------
def dist_setup(n_gpus):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist_mod.init_process_group(backend='gloo', rank=rank, world_size=world)
        dist = dist_mod
    return rank, world, local, dist


def barrier(dist):
    if dist is not None:
        dist.barrier()


def reduce_max(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def reduce_sum(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t[0])


def traffic_per_read():
    """measured DRAM bytes per read of the dominant kernel from this round's ncu capture
    (profiles/k_align_traffic.json); None when the capture predates the current kernel source
    (the file stores a hash of csrc/dp_*.cuh), so a stale constant never reaches the line"""
    import hashlib
    tp = os.path.join(REPO, 'profiles', 'k_align_traffic.json')
    try:
        t = json.load(open(tp))
    except Exception:
        return None, 'no capture'
    h = hashlib.sha256()
    for f in ('dp_row.cuh', 'dp_align.cuh', 'dp_align_kernel.cuh', 'dp_row2.cuh', 'common.cuh'):
        p = os.path.join(REPO, 'tombo_b200', 'csrc', f)
        if os.path.exists(p):
            h.update(open(p, 'rb').read())
    if t.get('source_sha16') != h.hexdigest()[:16]:
        return None, 'capture predates the current kernel source'
    return t.get('dram_bytes_per_read'), t.get('capture', 'ncu --set full')


DUMP_VALUES_PER_CONFIG = 1 << 20     # per workload; at most 4 workloads stay under 64 MB
DUMP_MAX_READS = 16384
DUMP_MAX_POSITIONS = 65536


def dump_outputs(directory, name, ctx, out, llr):
    """Write a seeded sample of what the last batch_compute returned as float64 .npy files
    DIR/<name>_<field>.npy: whole reads, drawn in a fixed order until DUMP_VALUES_PER_CONFIG
    values (their per-read fields, segs, norm_mean and LLR sites), and for the LLR workload a
    fixed sample of the finalized region statistics.  read_index holds the sampled reads.
    Values the library leaves undefined are written as 0 so that every file is finite: the
    float fields of a failed read (status != 0; its score is NaN) and frac / damp_frac of a
    position without valid calls (valid_cov == 0; NaN as in the reference).  A NaN anywhere
    else is kept."""
    seg_off, base_off = out['seg_off'], out['base_off']
    n = seg_off.shape[0] - 1
    cost = np.diff(seg_off) + np.diff(base_off) + 11      # + read_index and 10 per-read values
    if llr:
        llr_val, llr_pos, site_off = ctx.batch_llr_download()
        cost = cost + 2 * np.diff(site_off)
    order = np.random.RandomState(2024).permutation(n)
    take = np.sort(order[np.cumsum(cost[order]) <= DUMP_VALUES_PER_CONFIG][:DUMP_MAX_READS])

    def ragged(a, off):
        return np.concatenate([a[:0]] + [a[off[i]:off[i + 1]] for i in take])
    arrays = {'read_index': take}
    for f in ('status', 'n_iters', 'flags', 'read_start_rel_to_raw', 'sig_match_score',
              'scale_values'):
        arrays[f] = out[f][take]
    arrays['segs'] = ragged(out['segs'], seg_off)
    arrays['norm_mean'] = ragged(out['norm_mean'], base_off)
    failed = arrays['status'] != 0
    arrays['sig_match_score'][failed] = 0.0
    arrays['scale_values'][failed] = 0.0
    arrays['norm_mean'][np.repeat(failed, np.diff(base_off)[take])] = 0.0
    if llr:
        arrays['llr'] = ragged(llr_val, site_off)
        arrays['llr_pos'] = ragged(llr_pos, site_off)
        reg = ctx.region_stats_finalize(2, 0)
        m = reg['pos'].shape[0]
        pick = np.sort(np.random.RandomState(2025).choice(m, min(m, DUMP_MAX_POSITIONS),
                                                          replace=False))
        for f, v in reg.items():
            arrays['region_' + f] = v[pick]
        no_valid = arrays['region_valid_cov'] == 0
        arrays['region_frac'][no_valid] = 0.0
        arrays['region_damp_frac'][no_valid] = 0.0
    os.makedirs(directory, exist_ok=True)
    for f, a in arrays.items():
        np.save(os.path.join(directory, '%s_%s.npy' % (name, f)), np.asarray(a, dtype=np.float64))


def run_config(name, n_reads, steps, warmup, ctx, rank, local, dist, n_gpus, pin, do_parity=True,
               int16_e2e=False, dump_dir=None):
    """warm-up, timed resident region (device clock), timed end-to-end region (host buffers),
    parity sample -- for one workload.  Returns the fields of the JSON line."""
    from tombo_b200 import _lib, synthetic as syn
    cfg = CONFIGS[name]
    rna = cfg['kind'] == 'RNA'
    kmer_ref, cpos, raw, raw_off, seq, seq_off = make_workload(cfg, n_reads, 1 + rank, pin)
    if os.environ.get('TB2_BENCH_ROUND_RAW'):
        # diagnostic: integer-valued signal (what the int16 DAC dtype holds) through the f64 path
        np.round(raw, out=raw)
    k = len(kmer_ref[0][0])
    means, sds = syn.kmer_table(kmer_ref)
    ctx.set_model(means, sds, k, cpos)
    llr = bool(cfg.get('llr'))
    if llr:
        ctx.set_alt_model(alt_table(kmer_ref), k)
    rp = RP(cfg['aln'], cfg['seg'], rna=rna)
    sp = RP(cfg['aln'], cfg['seg'], save=True, rna=rna)
    pol = _lib.make_policy(cfg['kind'], subsample_seed=rank)
    n_samples = int(raw_off[-1])
    nb_tot = int(seq_off[-1] - (k - 1) * n_reads)
    out = {'segs': pin(nb_tot + n_reads, np.int64), 'read_start_rel_to_raw': pin(n_reads, np.int64),
           'scale_values': pin(n_reads * 5, np.float64).reshape(n_reads, 5),
           'sig_match_score': pin(n_reads, np.float64), 'norm_mean': pin(nb_tot, np.float64),
           'status': pin(n_reads, np.int32), 'n_iters': pin(n_reads, np.int32),
           'flags': pin(n_reads, np.int32)}
    h2d = raw.nbytes + seq.nbytes + raw_off.nbytes + seq_off.nbytes
    d2h = sum(v.nbytes for v in out.values())
    # per-position statistics of the LLR stage: reads tile a 1 Mb region
    read_start = ((np.arange(n_reads, dtype=np.int64) * 7919) % 1000000) if llr else None
    llr_thresh = (2.5, -2.5) if rna else (2.5, -1.5)             # LLR_THRESH

    def stats_stage():
        if not llr:
            return 0
        ctx.batch_alt_llr(read_start, 1)
        ctx.region_stats_begin(0, 1000000 + 400)
        ctx.region_stats_add_batch_llr(llr_thresh[0], llr_thresh[1], 0)
        return 1

    def e2e_step(raw_in):
        if not llr:
            ctx.resquiggle_batch(raw_in, raw_off, seq, seq_off, rp, sp, pol, out=out)
            return None
        # staged calls, host buffers in and out: H2D, kernels, LLR + counters, D2H
        ctx.batch_upload(raw_in, raw_off, seq, seq_off, rp, pol)
        ctx.batch_compute(rp, sp, pol)
        stats_stage()
        ctx.batch_download(out=out)
        return ctx.region_stats_finalize(2, 0)

    for _ in range(max(0, warmup)):                    # warm-up: full end-to-end steps
        e2e_step(raw)
    # ---- timed region A: inputs resident in HBM (kernel path only) ----
    ctx.batch_upload(raw, raw_off, seq, seq_off, rp, pol)
    for _ in range(max(0, warmup)):
        ctx.batch_compute(rp, sp, pol)
        stats_stage()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local)
    barrier(dist)
    sampler.start()
    t0 = time.perf_counter()
    dev_ms = dp_ms = dp_reads = dp_launches = 0.0
    for _ in range(steps):
        ctx.timer_start()
        ctx.batch_compute(rp, sp, pol)
        tm = ctx.last_timing()
        stats_stage()
        dev_ms += ctx.timer_stop()
        dp_ms += tm[1]; dp_launches += tm[2]; dp_reads += tm[3]
    t_res = time.perf_counter() - t0
    barrier(dist)
    clocks = sampler.stop()
    launches_timed = ctx.launch_count() - launches0
    ctx.batch_download(out=out)
    if dump_dir is not None:
        dump_outputs(dump_dir, name, ctx, out, llr)
    n_ok = int((out['status'] == 0).sum())
    n_rescued = int(((out['flags'] & 2) != 0).sum())
    # ---- timed region B: end to end through the C ABI with host buffers ----
    barrier(dist)
    t0 = time.perf_counter()
    reg = None
    for _ in range(steps):
        reg = e2e_step(raw)
    t_e2e = time.perf_counter() - t0
    barrier(dist)
    t_dev = reduce_max(dist, dev_ms / 1e3)
    t_res_w = reduce_max(dist, t_res)
    t_e2e_w = reduce_max(dist, t_e2e)
    tot_reads = reduce_sum(dist, float(n_reads)) * steps
    tot_samples = reduce_sum(dist, float(n_samples)) * steps
    tot_ok = reduce_sum(dist, float(n_ok))
    a_dp, cells = dp_algorithmic_bytes(raw_off, seq_off, k, rp)
    parity = None
    if do_parity and rank == 0:
        parity = parity_sample(name, cfg, out, raw, raw_off, seq, seq_off, means, sds, k, rp, sp,
                               rank, n_reads)
    e2e16 = None
    if int16_e2e:
        # the DAC dtype: int16 raw (2 bytes / sample over PCIe), tie rule pinned (DESIGN.md)
        raw16 = pin(n_samples, np.int16)
        np.round(raw, out=raw)            # the float copy is no longer needed
        raw16[:] = raw
        for _ in range(2):
            e2e_step(raw16)
        barrier(dist)
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step(raw16)
        t16 = reduce_max(dist, time.perf_counter() - t0)
        barrier(dist)
        e2e16 = {'t': t16, 'h2d': raw16.nbytes + seq.nbytes + raw_off.nbytes + seq_off.nbytes,
                 'ok': int((out['status'] == 0).sum())}
    peak, peak_src = peaks()
    bytes_per_read = float(a_dp.mean())
    ach = bytes_per_read * dp_reads / (dp_ms / 1e3) / 1e9 if dp_ms > 0 else 0.0
    tpr, tsrc = traffic_per_read()
    traffic = tpr * dp_reads / max(1.0, dp_launches) if (tpr and name == 'c1') else None
    res = {
        'metric': METRIC, 'value': tot_reads / t_dev, 'unit': 'reads/s',
        'samples_per_sec': tot_samples / t_dev,
        'n_gpus': n_gpus, 'steps': steps, 'warmup': warmup,
        'ms_per_step': 1e3 * t_dev / steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': cfg['label'] % n_reads, 'reads_per_gpu': n_reads,
                   'parallelism': 'reads sharded over %d GPU(s), no collective' % n_gpus,
                   'l2': 'inputs %.2f GB per step >> 126 MB L2 (no flush needed)'
                         % (raw.nbytes / 1e9),
                   'value_wall_clock_reads_per_s': tot_reads / t_res_w,
                   'reads_ok_frac': tot_ok / (tot_reads / steps),
                   'reads_rescued': n_rescued},
        'roofline': {'bound': 'hbm', 'kernel': 'k_align (banded DP + traceback)',
                     'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                     'frac': ach / peak, 'traffic': traffic, 'traffic_source': tsrc,
                     'peak_source': peak_src,
                     'algorithmic_bytes_per_read': bytes_per_read,
                     'launches': dp_launches, 'avg_launch_ms': dp_ms / max(1.0, dp_launches),
                     'dp_share_of_step': dp_ms / max(1e-9, dev_ms),
                     'cell_updates_per_s': float(cells.mean()) * dp_reads / (dp_ms / 1e3)
                     if dp_ms > 0 else 0.0},
        'e2e': {'value': tot_reads / t_e2e_w, 'unit': 'reads/s',
                'samples_per_sec': tot_samples / t_e2e_w,
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'path': 'staged upload/compute/LLR/download' if llr else
                        'tb2_resquiggle_batch (pipelined chunks)'},
        'gpu_launches': int(launches_timed),
        'clocks': clocks,
    }
    if e2e16 is not None:
        res['e2e_int16'] = {'value': tot_reads / e2e16['t'], 'unit': 'reads/s',
                            'h2d_bytes_per_step': e2e16['h2d'], 'd2h_bytes_per_step': d2h,
                            'reads_ok_frac': e2e16['ok'] / float(n_reads),
                            'note': 'same reads rounded to the int16 DAC dtype'}
    if parity is not None:
        res['parity'] = parity
    if reg is not None:
        res['config']['region_positions'] = int(reg['pos'].shape[0])
        res['config']['llr_sites_per_step'] = int(reg['cov'].sum())
    return res


def parity_sample(name, cfg, out, raw, raw_off, seq, seq_off, means, sds, k, rp, sp, seed, n_reads):
    """bit-compare a random sample of the timed batch (results of the last end-to-end step)
    with the C oracle (oracle/ is the checker here, after the timed regions)"""
    sys.path.insert(0, os.path.join(REPO, 'oracle'))
    import oracle as orc
    rs = np.random.RandomState(12345)
    m = min(cfg['parity'], n_reads)
    idx = np.sort(rs.choice(n_reads, m, replace=False))
    nb = (seq_off[1:] - seq_off[:-1]) - (k - 1)
    res = dict(out)
    res['seg_off'] = np.concatenate([[0], np.cumsum(nb + 1)])
    t0 = time.perf_counter()
    o = orc.run_batch(raw, raw_off, seq, seq_off, means, sds, k, rp, sp,
                      orc.policy(cfg['kind'], subsample_seed=seed), indices=idx)
    bad = orc.compare_batch(res, o)
    return {'checked': int(m), 'mismatches': len(bad), 'fields': 'status, segs, '
            'read_start_rel_to_raw, shift, scale, limits, score, n_iters, rescued, changed',
            'oracle_failed_too': int(sum(1 for v in o.values() if v['status'] != 0)),
            'first': [str(b) for b in bad[:3]], 'oracle_s': round(time.perf_counter() - t0, 2)}


def run_queue_mode(args, rank, world, local, dist):
    """strong scaling: ONE read set (mixed lengths), cut into length buckets, pulled by the
    ranks from a shared NCCL-free queue (tombo_b200.multi_gpu.WorkQueue)."""
    from tombo_b200 import _lib, synthetic as syn, multi_gpu as mg
    cfg = CONFIGS[args.workload]
    numa = mg.bind_to_gpu_numa_node(local)
    # one context (stream + device pools) per worker thread: while one bucket drains its
    # last iterations or copies back, the other keeps the SMs and the copy engines busy
    ctxs = [_lib.Context(local) for _ in range(max(1, args.queue_threads))]
    ctx = ctxs[0]
    pinned = []

    def pin(n, dt):
        pa = _lib.PinnedArray((n,), dt)
        pinned.append(pa)
        return pa.array
    total = args.reads
    kmer_ref, cpos, raw, raw_off, seq, seq_off = make_workload(cfg, total, 1, None)
    k = len(kmer_ref[0][0])
    means, sds = syn.kmer_table(kmer_ref)
    for c in ctxs:
        c.set_model(means, sds, k, cpos)
    rp, sp = RP(cfg['aln'], cfg['seg']), RP(cfg['aln'], cfg['seg'], save=True)
    pol = _lib.make_policy(cfg['kind'], subsample_seed=0)
    lens = raw_off[1:] - raw_off[:-1]
    nb = (seq_off[1:] - seq_off[:-1]) - (k - 1)
    buckets = mg.length_buckets(lens, nb, target_samples=args.bucket_samples,
                                tail_fraction=args.bucket_tail, tail_divisor=args.bucket_tail_div)
    # every rank packs every bucket into pinned buffers (untimed; a loader would emit them)
    packed = []
    for b in buckets:
        r = pin(int(lens[b].sum()), np.float64)
        ro = np.concatenate([[0], np.cumsum(lens[b])]).astype(np.int64)
        so = np.concatenate([[0], np.cumsum(seq_off[b + 1] - seq_off[b])]).astype(np.int64)
        sq = pin(int(so[-1]), np.uint8)
        for j, i in enumerate(b):
            r[ro[j]:ro[j + 1]] = raw[raw_off[i]:raw_off[i + 1]]
            sq[so[j]:so[j + 1]] = seq[seq_off[i]:seq_off[i + 1]]
        packed.append((r, ro, sq, so))
    # result buffers: pinned, one set per worker, sized for the largest bucket (a bucket's
    # results are consumed -- here: counted -- before the worker takes the next one)
    max_n = max(len(b) for b in buckets)
    max_nb = max(int(nb[b].sum()) for b in buckets)
    outbufs = [{'segs': pin(max_nb + max_n, np.int64), 'rsrtr': pin(max_n, np.int64),
                'sv': pin(max_n * 5, np.float64), 'score': pin(max_n, np.float64),
                'norm_mean': pin(max_nb, np.float64), 'status': pin(max_n, np.int32),
                'n_iters': pin(max_n, np.int32), 'flags': pin(max_n, np.int32)} for _ in ctxs]
    qname = 'tb2_bench_queue_%s' % os.environ.get('MASTER_PORT', 'solo')
    results = {}

    def one_pass(tag):
        if rank == 0:
            q = mg.WorkQueue(qname + tag, len(buckets), create=True)
        barrier(dist)
        if rank != 0:
            q = mg.WorkQueue(qname + tag, len(buckets))
        barrier(dist)
        t0 = time.perf_counter()
        mine = []

        def worker(c, ob):
            while True:
                i = q.next()
                if i is None:
                    break
                r, ro, sq, so = packed[i]
                n_i, nb_i = len(buckets[i]), int(nb[buckets[i]].sum())
                out = {'segs': ob['segs'][:nb_i + n_i], 'read_start_rel_to_raw': ob['rsrtr'][:n_i],
                       'scale_values': ob['sv'][:n_i * 5].reshape(n_i, 5),
                       'sig_match_score': ob['score'][:n_i], 'norm_mean': ob['norm_mean'][:nb_i],
                       'status': ob['status'][:n_i], 'n_iters': ob['n_iters'][:n_i],
                       'flags': ob['flags'][:n_i]}
                c.resquiggle_batch(r, ro, sq, so, rp, sp, pol, out=out)
                results[i] = int((out['status'] == 0).sum())
                mine.append(i)
        if len(ctxs) == 1:
            worker(ctx, outbufs[0])
        else:
            import threading
            th = [threading.Thread(target=worker, args=(c, ob)) for c, ob in zip(ctxs, outbufs)]
            for x in th:
                x.start()
            for x in th:
                x.join()
        t = time.perf_counter() - t0
        barrier(dist)
        q.close(unlink=(rank == 0))
        return t, mine
    for w in range(max(1, args.warmup)):
        one_pass('w%d' % w)
    sampler = ClockSampler(local)
    sampler.start()
    ts, counts = [], []
    for s in range(args.steps):
        t, mine = one_pass('s%d' % s)
        ts.append(t); counts.append(len(mine))
    clocks = sampler.stop()
    t_max = reduce_max(dist, sum(ts))
    t_min = -reduce_max(dist, -sum(ts))
    my_reads = sum(len(buckets[i]) for i in mine)
    ok = sum(results[i] for i in mine)
    tot_ok = reduce_sum(dist, float(ok))
    if rank == 0:
        line = {'metric': METRIC, 'value': total * args.steps / t_max, 'unit': 'reads/s',
                'samples_per_sec': float(raw_off[-1]) * args.steps / t_max,
                'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': 1e3 * t_max / args.steps, 'higher_is_better': True,
                'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': {'workload': cfg['label'] % total + ' -- ONE read set for all GPUs',
                           'queue': 'shared NCCL-free counter in /dev/shm, %d length buckets of '
                                    '<= %d samples (last %.0f %% of the samples: %dx smaller), longest first, %d worker '
                                    'threads (contexts) per rank' % (len(buckets), args.bucket_samples,
                                                                     100 * args.bucket_tail,
                                                                     args.bucket_tail_div, len(ctxs)),
                           'rank_time_min_over_max': t_min / t_max, 'numa': numa,
                           'reads_ok_frac': tot_ok / total,
                           'timing': 'end to end per bucket through tb2_resquiggle_batch, host '
                                     'buffers, wall clock max over ranks'},
                'e2e': {'value': total * args.steps / t_max, 'unit': 'reads/s',
                        'h2d_bytes_per_step': int(raw.nbytes + seq.nbytes),
                        'd2h_bytes_per_step': int(8 * (nb.sum() * 2 + total * 10))},
                'gpu_launches': int(sum(c.launch_count() for c in ctxs)), 'clocks': clocks}
        print(json.dumps(line))
    for pa in pinned:
        pa.free()
    for c in ctxs:
        c.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--reads', type=int, default=0, help='reads per GPU per step (0 = config default)')
    ap.add_argument('--cpu-sample', type=int, default=0, help='(kept for compatibility)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--workload', default='c1', choices=sorted(CONFIGS),
                    help='headline workload (default c1 = BASELINE configs[1])')
    ap.add_argument('--extras', default='mixed,rna,c5',
                    help='extra configs reported under extra_configs (N = 1 only); "" = none')
    ap.add_argument('--extra-steps', type=int, default=None,
                    help='timed steps of each extra config (default: --steps)')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--no-int16', action='store_true')
    ap.add_argument('--queue', action='store_true', help='strong scaling over a shared work queue')
    ap.add_argument('--bucket-tail', type=float, default=0.15,
                    help='--queue: fraction of the samples (the shortest reads) cut into smaller buckets')
    ap.add_argument('--bucket-tail-div', type=int, default=2)
    ap.add_argument('--queue-threads', type=int, default=4,
                    help='worker threads (one library context each) per rank in --queue mode')
    ap.add_argument('--bucket-samples', type=int, default=60_000_000)
    ap.add_argument('--cpu-leg', default='', help=argparse.SUPPRESS)
    ap.add_argument('--cpu-scale', type=float, default=1.0, help=argparse.SUPPRESS)
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='write a seeded sample of the last timed step\'s results to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.extra_steps is None:
        args.extra_steps = args.steps
    if args.dump_outputs and (args.queue or args.impl == 'reference'):
        ap.error('--dump-outputs applies to the GPU path without --queue')

    if args.cpu_leg:                      # child: the CPU legs in a clean interpreter
        names = [n for n in args.cpu_leg.split(',') if n]
        print(json.dumps(cpu_leg(names, host_cores(), cpu_baseline_kind(), steps=max(1, args.steps),
                                 scale=args.cpu_scale)))
        return
    rank, world, local, dist = dist_setup(args.gpus)
    cfg = CONFIGS[args.workload]
    n_reads = args.reads or cfg['reads']

    if args.impl == 'reference':
        if rank != 0:
            return
        # the reference's own CPU implementation, all host threads, same workload
        leg = cpu_leg([args.workload], host_cores(), cpu_baseline_kind(), steps=max(1, args.steps),
                      scale=1.5)
        c = leg[args.workload]['pool']
        cb = cpu_baseline_obj(leg, args.workload)
        line = {
            'impl': 'reference', 'metric': METRIC, 'value': c['reads_per_s'], 'unit': 'reads/s',
            'samples_per_sec': c['samples_per_s'], 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * c['wall_s'] / max(1, args.steps),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic',
            'config': {'workload': cfg['label'] % n_reads, 'reads_per_gpu': n_reads,
                       'reads_per_step': c['n'] // max(1, args.steps), 'l2': 'n/a (CPU)'},
            'cpu_baseline': cb,
            'e2e': {'value': c['reads_per_s'], 'unit': 'reads/s', 'h2d_bytes_per_step': 0,
                    'd2h_bytes_per_step': 0},
            'gpu_launches': 0,
        }
        print(json.dumps(line))
        return

    if args.queue:
        run_queue_mode(args, rank, world, local, dist)
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- ours ----------------
    extras = [e for e in args.extras.split(',') if e and e != args.workload] \
        if (args.gpus == 1 and world == 1) else []
    leg = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        # BEFORE the first CUDA call, in a clean interpreter
        try:
            leg = cpu_leg_subprocess([args.workload] + extras)
        except Exception as e:
            leg = {'error': repr(e)[:300]}
    from tombo_b200 import _lib, multi_gpu as mg
    numa = mg.bind_to_gpu_numa_node(local)      # before any pinned allocation
    ctx = _lib.Context(local)
    pinned = []

    def pin(n, dt):
        pa = _lib.PinnedArray((n,), dt)
        pinned.append(pa)
        return pa.array

    def free_pinned():
        while pinned:
            pinned.pop().free()
    dump_dir = args.dump_outputs if (args.dump_outputs and rank == 0) else None
    line = run_config(args.workload, n_reads, args.steps, args.warmup, ctx, rank, local, dist,
                      args.gpus, pin, do_parity=not args.no_parity, int16_e2e=not args.no_int16,
                      dump_dir=dump_dir)
    free_pinned()
    if rank == 0:
        line['config']['numa'] = numa
    if rank == 0 and leg is not None:
        if 'error' in leg:
            line['cpu_baseline'] = {'value': None, 'unit': 'reads/s', 'error': leg['error']}
        else:
            line['cpu_baseline'] = cpu_baseline_obj(leg, args.workload)
    ex_out = []
    for e in extras:
        try:
            r = run_config(e, CONFIGS[e]['reads'], args.extra_steps, max(3, min(args.warmup, 3)),
                           ctx, rank, local, dist, args.gpus, pin, do_parity=not args.no_parity,
                           dump_dir=dump_dir)
            r['name'] = e
            if leg is not None and e in leg:
                r['cpu_baseline'] = cpu_baseline_obj(leg, e)
            ex_out.append(r)
        except Exception as ex:     # an extra never takes the headline down
            ex_out.append({'name': e, 'error': repr(ex)[:300]})
        free_pinned()
    if rank == 0:
        if extras:
            line['extra_configs'] = ex_out
        print(json.dumps(line))
    free_pinned()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
