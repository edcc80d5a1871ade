#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Bifrost hot path.

Metric (BASELINE.json): Msamples/s through FDMT + FFT->detect->reduce on a
4096-chan ci8/int8 stream, and % of the HBM roofline.

  N = 1  (BASELINE config 2)  one "step" = one gulp of 4096 chan x 131072(+794)
         int8 samples through bfFdmtExecute (max_dm = 100 -> max_delay = 794).
         `value`: input resident in HBM, CUDA events on the launching stream.
         `e2e`:   the same call from pinned HOST buffers, H2D of the gulp and D2H
                  of the dispersion bank inside the timed region.
         `roofline`: algorithmic bytes / time / measured HBM peak; `traffic` is
                  measured in this run (a short ncu child process of this file).
         `chain`: the second half of the metric (config 3, fused GUPPI
                  spectrometer) with its own roofline object.
         `gpu_reference`: the reference's own CUDA kernels (oracle/_ref) timed on
                  the same box -- the "kernel to beat".
         `parity`: the timed gulp's output value-checked against the C oracle.
  N > 1  (BASELINE config 5, under torchrun)  STRONG scaling of that one gulp:
         rank 0 holds the 4096-chan gulp, NCCL scatters 4096/N-chan sub-bands,
         every rank runs bfFdmtInit(4096/N, max_delay_g, f0_g, df) + execute,
         NCCL gathers the [max_delay_g, ntime] banks to rank 0.  time = max over
         ranks including both collectives.  `replicas` keeps the weak-scaling
         figure (every rank its own full 4096-chan gulp, no collective).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

`--impl reference` times the CPU restatement of the reference algorithm
(oracle/fdmt_c.c, all host threads) on a bounded sample of the same gulp.
`--dry-run` exercises the multi-rank host logic on gloo with no GPU work.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NCHAN = 4096
NTIME_OUT = 131072
# bounded CPU sample, all 4096 channels: the whole gulp where the host has the cores to finish it
# in well under a second (the B200 boxes: 128), else 1/4 of its time span (env override: tests only)
def _mem_available_gb():
    try:
        for line in open('/proc/meminfo'):
            if line.startswith('MemAvailable:'):
                return int(line.split()[1]) / 2 ** 20
    except Exception:
        pass
    return 0.


# (the step-by-step oracle keeps two buffers of 8192 rows: 8.7 GB for the whole gulp)
CPU_SAMPLE_NTIME = int(os.environ.get('BENCH_CPU_SAMPLE_NTIME',
                                      NTIME_OUT if ((os.cpu_count() or 1) >= 64 and _mem_available_gb() >= 48)
                                      else NTIME_OUT // 4))
F0_MHZ = 1000.0
BW_MHZ = 400.0
DT_S = 256e-6
MAX_DM = 100.0
KDM = 4.148741601e3
METRIC = 'Msamples/s through FDMT+FFT->detect->reduce on 4096-chan ci8; % HBM roofline'


def max_delay_for(f0, df, nchan, dt, max_dm):
    """blocks/fdmt.py:79-81 of the reference."""
    rel = (f0 ** -2 - (f0 + nchan * df) ** -2)
    return int(np.ceil(abs(KDM / dt * max_dm * rel)))


def workload(rank=0):
    """Replica workload: rank r's own 4096-channel band above the previous one."""
    df = BW_MHZ / NCHAN
    f0 = F0_MHZ + rank * NCHAN * df
    md = max_delay_for(F0_MHZ, df, NCHAN, DT_S, MAX_DM)      # same bank depth on every rank
    return dict(nchan=NCHAN, ntime=NTIME_OUT + md, max_delay=md, f0=f0, df=df)


def subband(g, n):
    """Config 5: sub-band g of n of the one 4096-chan gulp, with the header a
    reference pipeline reading that sub-band file would carry."""
    w = workload(0)
    nc = NCHAN // n
    f0 = w['f0'] + g * nc * w['df']
    md = max_delay_for(f0, w['df'], nc, DT_S, MAX_DM)
    return dict(nchan=nc, chan0=g * nc, ntime=w['ntime'], max_delay=md, f0=f0, df=w['df'])


def bench_config(world):
    """The `config` object of the JSON line -- the same for the GPU arm and for
    `--impl reference` (the driver compares them)."""
    full = workload(0)
    md = full['max_delay']
    if world == 1:
        return dict(workload='BASELINE config 2: bfFdmtExecute, max_dm=100 '
                             f'(max_delay={md}) on {NCHAN}-chan x {NTIME_OUT}(+{md})-sample '
                             'int8 filterbank; f0=1000 MHz, bw=400 MHz, dt=256 us',
                    sharding='single GPU',
                    l2='input 540 MB + output 419 MB per step exceed the 126 MB L2')
    subs = [subband(g, world) for g in range(world)]
    nc = subs[0]['nchan']
    return dict(workload=f'BASELINE config 5: the one {NCHAN}-chan x {NTIME_OUT}(+{md})-sample int8 '
                         f'gulp of config 2 split into {world} sub-bands of {nc} channels',
                sharding=f'NCCL grouped send/recv scatter of the sub-bands from rank 0 -> per-GPU '
                         f'bfFdmtInit({nc}, max_delay_g, f0_g, df) + bfFdmtExecute -> NCCL grouped '
                         'send/recv gather of the [max_delay_g, ntime] f32 banks to rank 0',
                subband_max_delay=[s['max_delay'] for s in subs],
                subband_f0_mhz=[s['f0'] for s in subs],
                l2='per-GPU inputs and banks exceed L2 for N <= 4; the collectives stream through HBM')


def make_input(w, seed, ntime=None):
    """round(N(0,20)) clipped to int8 plus three dispersed pulses (BASELINE.md cfg 2)."""
    ntime = ntime or w['ntime']
    rng = np.random.default_rng(seed)
    x = np.empty((w['nchan'], ntime), np.int8)
    step = 256
    blk = rng.normal(0, 20, size=(step, ntime)).astype(np.float32)
    np.rint(blk, out=blk)
    np.clip(blk, -127, 127, out=blk)
    blk = blk.astype(np.int8)
    for i, c0 in enumerate(range(0, w['nchan'], step)):
        # one noise block reused with a different cyclic time shift per block
        x[c0:c0 + step] = np.roll(blk, 7919 * i, axis=1)[:min(step, w['nchan'] - c0)]
    f = w['f0'] + w['df'] * np.arange(w['nchan'])
    fmax = f[-1]
    rel = (f ** -2 - fmax ** -2) / (f[0] ** -2 - fmax ** -2)
    for frac_dm, t0 in ((0.2, ntime // 5), (0.5, ntime // 2), (0.9, (3 * ntime) // 4)):
        tt = t0 + np.rint(rel * frac_dm * (w['max_delay'] - 1)).astype(np.int64)
        ok = tt < ntime
        x[np.arange(w['nchan'])[ok], tt[ok]] = 100
    return x


def dump_output(dirname, name, a, keep):
    """--dump-outputs: `a` as dirname/name.npy in float32, on `keep` of its
    columns (last axis), a fixed seeded choice, so the dump stays small and
    two runs with the same arguments write the same elements."""
    a = np.asarray(a)
    if keep < a.shape[-1]:
        idx = np.sort(np.random.default_rng(0).choice(a.shape[-1], keep, replace=False))
        a = a[..., idx]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + '.npy'), np.ascontiguousarray(a, dtype=np.float32))


# columns of the dispersion bank kept by --dump-outputs: [max_delay, 8192] f32 (26 MB at max_delay 794)
DUMP_BANK_COLUMNS = 8192
# of the spectrometer's [4, 4096 * 1024] f32 output: [4, 2**20] (16 MB)
DUMP_SPECTRA_COLUMNS = 2 ** 20


class ClockSampler(object):
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    QUERY = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.QUERY}',
                 '--format=csv,noheader,nounits', '-lms', '50'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, smmax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smmax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None,
                    sm_max_mhz=float(np.max(smmax)) if smmax else None,
                    samples=len(sm), reasons=sorted(reasons))


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        try:
            return json.load(open(path)), 'measured'
        except Exception:
            pass
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0), 'fallback'


def bind_to_gpu_numa_node(index):
    """Pins this process (and the pinned host pages it allocates afterwards,
    first touch) to the CPUs of the NUMA node the GPU hangs off."""
    try:
        bus = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=pci.bus_id', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith('0000'):
            bus = bus[4:]                                   # sysfs uses a 4-digit domain
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            _ORIGINAL_AFFINITY.append(os.sched_getaffinity(0))
            os.sched_setaffinity(0, cpus)
            return dict(numa_node=node, cpus=len(cpus))
    except Exception:
        pass
    return None


_ORIGINAL_AFFINITY = []      # what bind_to_gpu_numa_node narrowed (the CPU baseline leg widens it again)


# --------------------------------------------------------------------------- CPU arm
class CpuFdmt(object):
    """The oracle (CPU restatement of the reference algorithm) on a bounded
    sample: the full 4096 channels, `ntime_sample` time samples.  Input and
    plan are built once; run() times one transform."""

    def __init__(self, w, ntime_sample, threads=None):
        try:
            from oracle import fdmt_c
            self.have_c = fdmt_c.available()
        except Exception:
            self.have_c = False
        if not self.have_c:
            ntime_sample = min(ntime_sample, 8192)        # the numpy port is ~10x slower
        self.w, self.ntime_sample = w, ntime_sample
        self.x = make_input(w, 4321, ntime=ntime_sample + w['max_delay'])
        self.nsamp = w['nchan'] * ntime_sample
        self.kind = 'port'
        if self.have_c:
            self.cores = threads or len(os.sched_getaffinity(0))
            self.plan = fdmt_c.Plan(w['nchan'], w['max_delay'], w['f0'], w['df'])
            self.out = np.zeros((w['max_delay'], self.x.shape[1]), np.float32)
            self.plan.execute(self.x, self.out, threads=self.cores)       # warm (page-in, thread pool)
        else:
            from oracle import fdmt as ofdmt
            self.cores = 1
            self.plan = ofdmt.FdmtPlan(w['nchan'], w['max_delay'], w['f0'], w['df'])

    def run(self):
        """Seconds of one transform of the sample."""
        t0 = time.perf_counter()
        if self.have_c:
            self.plan.execute(self.x, self.out, threads=self.cores)
        else:
            from oracle import fdmt as ofdmt
            ofdmt.fdmt(self.x, self.w['max_delay'], self.w['f0'], self.w['df'], plan=self.plan)
        return time.perf_counter() - t0

    def msamples_per_s(self, dt):
        return self.nsamp / dt / 1e6


def cpu_fdmt_sample(w, ntime_sample, threads=None):
    """One timed transform: (Msamples/s, kind, cores, seconds)."""
    c = CpuFdmt(w, ntime_sample, threads)
    dt = c.run()
    return c.msamples_per_s(dt), c.kind, c.cores, dt


def run_reference_arm(args, rank, world):
    """The reference has no CPU implementation of this path; its algorithm
    restated in C (oracle/fdmt_c.c) runs on all host threads of this box.  The
    workload is the one gulp of config 2 / config 5 whatever N is (the GPU arm
    scales strongly), so rank 0 alone runs it."""
    if rank != 0:
        return
    w = workload(0)
    cpu = CpuFdmt(w, CPU_SAMPLE_NTIME)
    ntime_sample, cores = cpu.ntime_sample, cpu.cores
    vals, secs = [], []
    for i in range(args.warmup + args.steps):
        dt = cpu.run()
        if i >= args.warmup:
            vals.append(cpu.msamples_per_s(dt))
            secs.append(dt)
    value = float(np.mean(vals))
    sample = (f"oracle CPU FDMT (oracle/fdmt_c.c, pthreads) on {w['nchan']} chan x {ntime_sample} samples "
              f"(1/{NTIME_OUT // ntime_sample} of the gulp) per step, {cores} threads")
    line = dict(impl='reference', metric=METRIC, value=value, unit='Msamples/s', n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=float(np.mean(secs) * 1e3),
                higher_is_better=True, scaling='strong' if args.gpus > 1 else 'weak', vs_baseline=None,
                dtype='f32', data='synthetic',
                # the GPU arm's config; what the CPU ran of it per step is cpu_baseline.sample
                # (the same one gulp at every N: the GPU arm scales strongly, CPU threads do not grow with N)
                config=bench_config(max(1, args.gpus)),
                cpu_baseline=dict(value=value, unit='Msamples/s', cores=cores, kind='port',
                                  sample=sample),
                e2e=dict(value=value, unit='Msamples/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# --------------------------------------------------------------------------- dry run
def run_dry(args, rank, world):
    """Multi-rank host logic without a GPU: the config-5 split (sub-band
    headers, bank offsets), barrier, max over ranks, gather of the banks."""
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group('gloo')
    sb = subband(rank, world)
    ms = 1.0 + 0.5 * rank                      # pretend rank r needs 1 + r/2 ms per step
    subs = [subband(g, world) for g in range(world)]
    offs = np.concatenate([[0], np.cumsum([s['max_delay'] for s in subs])])
    gathered = None
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms])
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        # a token "bank" per rank: md_g rows of the value g, gathered into rank 0's bank
        mine = torch.full((sb['max_delay'], 4), float(rank))
        if rank == 0:
            bank = torch.full((int(offs[-1]), 4), -1.0)
            bank[:sb['max_delay']] = mine
            reqs = [dist.irecv(bank[int(offs[g]):int(offs[g + 1])], g) for g in range(1, world)]
            for r in reqs:
                r.wait()
            gathered = [float(bank[int(offs[g])][0]) for g in range(world)] + [float(bank.min())]
        else:
            dist.isend(mine, 0).wait()
    if rank == 0:
        print(json.dumps(dict(dry_run=True, n_gpus=world, ms_per_step=ms, scaling='strong' if world > 1 else 'weak',
                              config=bench_config(world),
                              value=NCHAN * NTIME_OUT / (ms * 1e-3) / 1e6,
                              subband_f0_mhz=[s['f0'] for s in subs], subband_nchan=[s['nchan'] for s in subs],
                              subband_max_delay=[s['max_delay'] for s in subs], bank_offsets=[int(o) for o in offs],
                              gathered=gathered)))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- GPU arm
def log(*a):
    if os.environ.get('BENCH_VERBOSE'):
        print('[bench]', *a, file=sys.stderr, flush=True)


def traffic_probe():
    """Child mode (run under ncu by measure_traffic): a few resident steps."""
    import bifrost_b200 as bf
    from bifrost_b200.fdmt import Fdmt
    w = workload(0)
    x = make_input(w, 1234)
    d_in = bf.asarray(x, space='cuda')
    d_out = bf.empty((w['max_delay'], w['ntime']), dtype='f32', space='cuda')
    plan = Fdmt()
    plan.init(w['nchan'], w['max_delay'], w['f0'], w['df'])
    for _ in range(3):
        plan.execute(d_in, d_out)
    bf.device.stream_synchronize()


def measure_traffic(launches_per_step):
    """DRAM bytes of one bfFdmtExecute, measured now: ncu replays this file's
    --traffic-probe mode with the two dram__bytes counters.  None when ncu (or
    the permission to read counters) is not there."""
    import shutil
    ncu = shutil.which('ncu') or '/usr/local/cuda/bin/ncu'
    if not os.path.exists(ncu):
        return None, 'ncu not found'
    cmd = [ncu, '--metrics', 'dram__bytes_read.sum,dram__bytes_write.sum', '--clock-control', 'none',
           '-k', 'regex:fdmt', '--csv', sys.executable, os.path.abspath(__file__), '--traffic-probe']
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=300).stdout
    except Exception as e:
        return None, f'ncu failed: {e}'
    import csv
    rows = [r for r in csv.reader(out.splitlines()) if len(r) > 8]
    if not rows or 'Metric Value' not in rows[0]:
        return None, 'ncu printed no metrics (no permission to read counters?)'
    h = rows[0]
    iv, iu, iid = h.index('Metric Value'), h.index('Metric Unit'), h.index('ID')
    scale = {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    per = {}
    for r in rows[1:]:
        try:
            per.setdefault(int(r[iid]), 0.0)
            per[int(r[iid])] += float(r[iv].replace(',', '')) * scale.get(r[iu], 1)
        except (ValueError, IndexError):
            continue
    ids = sorted(per)
    if len(ids) < launches_per_step:
        return None, 'too few launches captured'
    last = ids[-launches_per_step:]                     # the last (warm) step
    return float(sum(per[i] for i in last)), f'ncu dram__bytes_read+write.sum over the {launches_per_step} launch(es) of one warm step, this run'


def oracle_window_check(x, got_fn, w, windows):
    """Bit-for-bit check of output columns [a, a+n) against the C oracle run on
    the input slice those columns depend on."""
    from oracle import fdmt_c
    if not fdmt_c.available():
        return dict(ok=None, note='oracle/libfdmt_oracle.so not built')
    md, ntime = w['max_delay'], x.shape[1]
    plan = fdmt_c.Plan(w['nchan'], md, w['f0'], w['df'])
    bad = 0
    for a, n in windows:
        b = min(ntime, a + n + md)
        want = np.zeros((md, b - a), np.float32)
        plan.execute(np.ascontiguousarray(x[:, a:b]), want)
        m = min(n, b - a)
        got = got_fn(a, m)
        # cells past ntime - r are never written by either side; compare written ones
        r = np.arange(md)[:, None]
        c = np.arange(m)[None, :] + a
        valid = c < ntime - r
        bad += int(((got.view(np.uint32) != want[:, :m].view(np.uint32)) & valid).sum())
    return dict(ok=bad == 0, mismatches=bad, windows=len(windows),
                how='output columns of the timed gulp vs oracle/fdmt_c.c on the input slices they depend on, bit for bit')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20,
                    help='timed steps of each figure: the resident FDMT step, e2e and the spectrometer chain '
                         '(N > 1: the strong-scaling step and e2e; the per-phase, full-band and replica '
                         'breakdowns time a fixed 5 or 10)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-chain', action='store_true')
    ap.add_argument('--no-fullband', action='store_true', help='N > 1: skip the cross-GPU full-band transform')
    ap.add_argument('--fullband-peer', action='store_true',
                    help='N > 1: also time the full-band transform with phase 1 reading peer memory (CUDA IPC)')
    ap.add_argument('--no-traffic', action='store_true')
    ap.add_argument('--no-gpu-reference', action='store_true')
    ap.add_argument('--dry-run', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed to DIR/<name>.npy (float32): fdmt_bank = '
                         'the dispersion bank (N > 1: the gathered one), spectrometer = the fused chain\'s '
                         'output, each on a fixed seeded sample of its columns')
    ap.add_argument('--traffic-probe', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl == 'reference' or args.dry_run):
        ap.error('--dump-outputs writes what the GPU arm computes')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.traffic_probe:
        traffic_probe()
        return
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
        return
    if args.dry_run:
        run_dry(args, rank, world)
        return

    numa = bind_to_gpu_numa_node(local_rank)           # before any pinned allocation
    import torch
    import torch.distributed as dist
    import bifrost_b200 as bf
    from bifrost_b200.fdmt import Fdmt

    torch.cuda.set_device(local_rank)
    bf.device.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    stream = torch.cuda.current_stream()
    bf.device.set_stream(stream.cuda_stream)
    peaks, peak_kind = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device='cuda')
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(fn, nwarm, nstep, sampler=None, post=None):
        for _ in range(nwarm):
            fn()
        if sampler:
            # (before the barrier: only one rank samples, and a rank that entered
            # the timed region late would make its peers wait inside it)
            sampler.start()
            time.sleep(0.1)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = bf.launch_count()
        ev0.record(stream)
        for _ in range(nstep):
            fn()
        ev1.record(stream)
        barrier()
        launches = bf.launch_count() - launches0
        clocks = None
        if sampler:
            # the timed region can be shorter than nvidia-smi's sampling period:
            # keep the same load running (untimed) until a few samples exist.
            # Only the rank that samples runs this, so with several ranks the
            # post-roll must be collective-free (`post`): the other ranks are
            # already waiting in max_over_ranks.
            t_end = time.time() + 1.5
            while len(sampler.lines) < 8 and time.time() < t_end:
                for _ in range(5):
                    (post or fn)()
                torch.cuda.synchronize()
            clocks = sampler.stop()
            clocks['window'] = 'timed steps + untimed post-roll of the same steps (nvidia-smi -lms 50)'
        return max_over_ranks(ev0.elapsed_time(ev1)), launches, clocks

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if world > 1:
        run_multi(args, rank, local_rank, world, bf, Fdmt, torch, dist, stream, timed, barrier, max_over_ranks,
                  sampler, peaks, peak_kind, numa)
        dist.destroy_process_group()
        return

    # ------------------------------------------------------------------ N = 1
    w = workload(0)
    nchan, ntime, md = w['nchan'], w['ntime'], w['max_delay']
    x_host = make_input(w, 1234)
    pinned_in = bf.empty((nchan, ntime), dtype='i8', space='cuda_host')
    np.copyto(np.asarray(pinned_in), x_host)
    pinned_out = bf.empty((md, ntime), dtype='f32', space='cuda_host')
    d_in = bf.empty((nchan, ntime), dtype='i8', space='cuda')
    d_out = bf.empty((md, ntime), dtype='f32', space='cuda')
    bf.copy_array(d_in, pinned_in)
    bf.memset_array(d_out, 0)
    plan = Fdmt()
    plan.init(nchan, md, w['f0'], w['df'])
    ws_size = plan.get_workspace_size(d_in, d_out)
    ws = bf.empty((ws_size,), dtype='u8', space='cuda')
    log('workspace', ws_size)

    def step_resident():
        plan.execute_workspace(d_in, d_out, ws.ctypes.data, ws_size)

    def step_e2e():
        bf.copy_array(d_in, pinned_in)            # H2D of this gulp (pinned, async on the stream)
        plan.execute_workspace(d_in, d_out, ws.ctypes.data, ws_size)
        bf.copy_array(pinned_out, d_out)          # D2H of the dispersion bank (+ stream sync)

    ms_total, launches, clocks = timed(step_resident, args.warmup, args.steps, sampler)
    ms_step = ms_total / args.steps
    launches_per_step = max(1, launches // args.steps)
    log('resident ms/step', ms_step)
    if args.dump_outputs:                          # before anything below reuses d_out
        dump_output(args.dump_outputs, 'fdmt_bank', d_out.copy('system'), keep=DUMP_BANK_COLUMNS)

    # value check of exactly this gulp (untimed): five windows, both edges
    got_dev = d_out

    def got_fn(a, n):
        return np.asarray(got_dev[:, a:a + n].copy('system'))
    parity = oracle_window_check(x_host, got_fn, w, [(0, 4096), (40000, 4096), (65536 + 3, 4096), (100001, 4096),
                                                       (ntime - 4096 - md, 4096 + md)])

    ms_e2e_total, _, _ = timed(step_e2e, 2, args.steps)
    ms_e2e_serial = ms_e2e_total / args.steps

    # The same three calls as a host pipeline, the way bifrost runs blocks: one
    # thread (and thread-local stream) per stage -- copy(H2D) -> fdmt -> copy(D2H)
    # -- double-buffered, each stage synchronising its own stream per gulp
    # (pipeline.py:628 of the reference).  Every gulp's H2D and D2H is inside
    # the timed region; consecutive gulps overlap on the copy engines.
    import queue
    d_in2 = [d_in, bf.empty((nchan, ntime), dtype='i8', space='cuda')]
    d_out2 = [d_out, bf.empty((md, ntime), dtype='f32', space='cuda')]
    ws2 = [ws, bf.empty((ws_size,), dtype='u8', space='cuda')]

    def run_pipeline(nstep):
        q_in_free, q_in_full = queue.Queue(), queue.Queue()
        q_out_free, q_out_full = queue.Queue(), queue.Queue()
        for i in range(2):
            q_in_free.put(i)
            q_out_free.put(i)
        errors = []

        def stage(fn):
            def body():
                try:
                    bf.device.set_device(local_rank)
                    fn()
                except Exception as e:      # surfaces in the main thread
                    errors.append(e)
            return threading.Thread(target=body)

        def h2d():
            for _ in range(nstep):
                i = q_in_free.get()
                bf.copy_array(d_in2[i], pinned_in)
                bf.device.stream_synchronize()
                q_in_full.put(i)

        def compute():
            for _ in range(nstep):
                i = q_in_full.get()
                o = q_out_free.get()
                plan.execute_workspace(d_in2[i], d_out2[o], ws2[o].ctypes.data, ws_size)
                bf.device.stream_synchronize()
                q_in_free.put(i)
                q_out_full.put(o)

        def d2h():
            for _ in range(nstep):
                o = q_out_full.get()
                bf.copy_array(pinned_out, d_out2[o])
                bf.device.stream_synchronize()
                q_out_free.put(o)

        threads = [stage(h2d), stage(compute), stage(d2h)]
        barrier()
        t0 = time.perf_counter()
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if errors:
            raise errors[0]
        return dt * 1e3

    try:
        run_pipeline(2)                                # warm-up
        ms_pipe = run_pipeline(args.steps) / args.steps
    except Exception as e:                             # keep the serial figure
        log('pipelined e2e failed:', e)
        ms_pipe = float('inf')
    ms_e2e = min(ms_pipe, ms_e2e_serial)
    del d_in2, d_out2, ws2
    log('e2e ms/step', ms_e2e)

    samples_per_step = nchan * NTIME_OUT                    # pol not counted (SURVEY 8d)
    value = samples_per_step / (ms_step * 1e-3) / 1e6
    e2e_value = samples_per_step / (ms_e2e * 1e-3) / 1e6

    # Roofline of the op (all kernels of one bfFdmtExecute): compulsory bytes
    # ntime*(nchan*1 + max_delay*4) per gulp (SURVEY 8d).
    alg_bytes = ntime * (nchan * 1 + md * 4)
    achieved = alg_bytes / (ms_step * 1e-3) / 1e9
    traffic, traffic_how = (None, 'skipped')
    if not args.no_traffic:
        traffic, traffic_how = measure_traffic(launches_per_step)
    roofline = dict(bound='hbm',
                    kernel=f'bfFdmtExecute = {launches_per_step} launch(es) per gulp (fdmt_packed*: packed-integer '
                           'schedule, see DESIGN.md 4.1); bytes and time are those of the whole call',
                    achieved=achieved, peak=peaks['hbm_gbs'], peak_source=peak_kind, unit='GB/s',
                    frac=achieved / peaks['hbm_gbs'], algorithmic_bytes=alg_bytes,
                    traffic=traffic, traffic_source=traffic_how,
                    traffic_over_algorithmic=(traffic / alg_bytes) if traffic else None)

    # ---- the reference's own CUDA kernels on this box (the "kernel to beat")
    gpu_reference = None
    if not args.no_gpu_reference:
        gpu_reference = time_gpu_reference(bf, torch, stream, d_in, d_out, w)

    # ---- second half of the metric: the fused GUPPI chain (config 3)
    chain = None
    if not args.no_chain:
        del ws
        chain = time_chain(bf, torch, timed, peaks, args.steps, args.dump_outputs)

    cpu = None
    if not args.no_cpu_baseline:
        if _ORIGINAL_AFFINITY:                       # the CPU leg gets every host core back
            os.sched_setaffinity(0, _ORIGINAL_AFFINITY[0])
        v, kind, cores, dt = cpu_fdmt_sample(w, CPU_SAMPLE_NTIME)
        cpu = dict(value=v, unit='Msamples/s', cores=cores, kind=kind,
                   sample=f"oracle CPU FDMT: {nchan} chan x {CPU_SAMPLE_NTIME} samples "
                          f"(1/{NTIME_OUT // CPU_SAMPLE_NTIME} of the gulp), {dt:.2f} s, "
                          f"{cores} thread(s) of {os.cpu_count()} host cores")

    line = dict(metric=METRIC, value=value, unit='Msamples/s', n_gpus=1, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True,
                scaling='weak', vs_baseline=None, dtype='u16/f32 (exact integers; bit-identical to the reference\'s f32)',
                data='synthetic',
                config=bench_config(1), host_numa=numa,
                roofline=roofline, cpu_baseline=cpu, gpu_reference=gpu_reference, parity=parity,
                e2e=dict(value=e2e_value, unit='Msamples/s', ms_per_step=ms_e2e,
                         ms_per_step_serial=ms_e2e_serial, ms_per_step_pipelined=ms_pipe,
                         how='host buffers -> bf.copy_array(H2D) -> Fdmt.execute -> bf.copy_array(D2H) per gulp; '
                             'pipelined = one host thread + stream per stage, double-buffered (wall clock, '
                             'device synchronised both sides); serial = one stream',
                         h2d_bytes_per_step=int(nchan * ntime), d2h_bytes_per_step=int(md * ntime * 4)),
                gpu_launches=int(launches), clocks=clocks, chain=chain)
    print(json.dumps(line))


def time_gpu_reference(bf, torch, stream, d_in, d_out, w):
    """oracle/_ref/libbifrost_ref.so = the reference's own fdmt.cu compiled for
    sm_100 (oracle/ref_build.sh): same device buffers, same stream."""
    import ctypes
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    try:
        import reflib
        ref = reflib.load()
    except Exception:
        ref = None
    if ref is None:
        return dict(available=False, note='oracle/_ref/libbifrost_ref.so did not travel')
    try:
        from bifrost_b200.libbifrost import _check
        h = ctypes.c_void_p(stream.cuda_stream)
        ref.bfStreamSet(ctypes.byref(h))
        plan = ctypes.c_void_p()
        _check(ref.bfFdmtCreate(ctypes.byref(plan)))
        _check(ref.bfFdmtInit(plan, w['nchan'], w['max_delay'], w['f0'], w['df'], -2.0, 2, None, None))
        a_in, a_out = d_in.as_BFarray(), d_out.as_BFarray()
        for _ in range(2):
            _check(ref.bfFdmtExecute(plan, a_in, a_out, 0, None, None))
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            _check(ref.bfFdmtExecute(plan, a_in, a_out, 0, None, None))
            e1.record(stream)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        _check(ref.bfFdmtDestroy(plan))
        ms = float(np.median(times))
        return dict(available=True, fdmt_ms_per_gulp=ms,
                    fdmt_Msamples_s=w['nchan'] * NTIME_OUT / (ms * 1e-3) / 1e6,
                    what="the reference's src/fdmt.cu kernels (13 launches) on the same gulp, same box")
    except Exception as e:
        return dict(available=False, note=f'reference library failed: {e}')


def time_chain(bf, torch, timed, peaks, nstep, dump_dir=None):
    nframe, cchan, nfft, f_avg = 32, 4096, 4096, 4
    nbyte = nframe * cchan * nfft * 4
    gen = torch.Generator(device='cuda').manual_seed(1234)
    raw = torch.randint(-127, 128, (nbyte,), dtype=torch.int8, device='cuda', generator=gen)
    xg = bf.empty((nframe, cchan, nfft, 2), 'ci8', 'cuda')
    from bifrost_b200.libbifrost import _bf, _check
    _check(_bf.bfMemcpy(xg.ctypes.data, xg.as_BFarray().space, raw.data_ptr(),
                        xg.as_BFarray().space, nbyte))
    torch.cuda.synchronize()
    del raw
    og = bf.zeros((4, cchan * nfft // f_avg), 'f32', 'cuda')
    ms_c, _, _ = timed(lambda: bf.spectrometer(xg, og, nfft, f_avg, 0.0), 3, nstep)
    ms_c /= nstep
    if dump_dir:
        dump_output(dump_dir, 'spectrometer', og.copy('system'), keep=DUMP_SPECTRA_COLUMNS)
    gbs = nbyte / (ms_c * 1e-3) / 1e9
    # useful fp32 work: 2 pols x 5 N log2 N per 4096-point FFT + detect/reduce (~16 flop/sample)
    flops = nframe * cchan * (2 * 5 * nfft * 12 + 16 * nfft)
    tflops = flops / (ms_c * 1e-3) / 1e12
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12                 # SMs x lanes x FMA x GHz
    return dict(workload='BASELINE config 3: GUPPI ci8 [32 frames, 4096 chan, 4096 fine_time, 2 pol] -> '
                         'fft(fine_time, fftshift) -> stokes -> reduce(f_avg=4) -> accumulate(32 frames); '
                         'bfSpectrometerFused, one kernel per gulp',
                ms_per_gulp=ms_c, value=nframe * cchan * nfft / (ms_c * 1e-3) / 1e6, unit='Msamples/s',
                roofline=dict(bound='fp32 issue (2 x 4096-pt FFT per 16 KB read; SURVEY 8d)',
                              hbm_GBps=gbs, hbm_frac=gbs / peaks['hbm_gbs'], algorithmic_bytes=nbyte,
                              fp32_tflops=tflops, fp32_peak_tflops=fp32_peak, fp32_frac=tflops / fp32_peak))


def run_multi(args, rank, local_rank, world, bf, Fdmt, torch, dist, stream, timed, barrier, max_over_ranks,
              sampler, peaks, peak_kind, numa):
    """Config 5: one gulp, N sub-bands, NCCL scatter + gather (strong scaling),
    plus the replica (weak) figure."""
    full = workload(0)
    ntime = full['ntime']
    subs = [subband(g, world) for g in range(world)]
    sb = subs[rank]
    nc, md = sb['nchan'], sb['max_delay']
    offs = np.concatenate([[0], np.cumsum([s['max_delay'] for s in subs])]).astype(np.int64)
    x_full = make_input(full, 1234)
    x_sub = np.ascontiguousarray(x_full[sb['chan0']:sb['chan0'] + nc])
    # device buffers as torch tensors (NCCL) viewed as bf arrays (C ABI)
    t_in = torch.empty((nc, ntime), dtype=torch.int8, device='cuda')
    t_full = torch.from_numpy(x_full).cuda() if rank == 0 else None
    t_bank = torch.zeros((int(offs[-1]), ntime), dtype=torch.float32, device='cuda') if rank == 0 else None
    t_out = t_bank[:md] if rank == 0 else torch.zeros((md, ntime), dtype=torch.float32, device='cuda')
    a_in = bf.ndarray(base=(t_full[:nc] if rank == 0 else t_in))
    a_out = bf.ndarray(base=t_out)
    plan = Fdmt()
    plan.init(nc, md, sb['f0'], sb['df'])
    ws_size = plan.get_workspace_size(a_in, a_out)
    ws = bf.empty((ws_size,), dtype='u8', space='cuda')
    P2P = dist.P2POp

    def scatter():
        if rank == 0:
            ops = [P2P(dist.isend, t_full[g * nc:(g + 1) * nc], g) for g in range(1, world)]
        else:
            ops = [P2P(dist.irecv, t_in, 0)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()

    def gather():
        if rank == 0:
            ops = [P2P(dist.irecv, t_bank[int(offs[g]):int(offs[g + 1])], g) for g in range(1, world)]
        else:
            ops = [P2P(dist.isend, t_out, 0)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()

    def compute():
        plan.execute_workspace(a_in, a_out, ws.ctypes.data, ws_size)

    def step_strong():
        scatter()
        compute()
        gather()

    ms_total, launches, clocks = timed(step_strong, args.warmup, args.steps, sampler, post=compute)
    ms_step = ms_total / args.steps
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, 'fdmt_bank', t_bank.cpu().numpy(), keep=DUMP_BANK_COLUMNS)
    ms_scatter = timed(scatter, 2, 5)[0] / 5
    ms_compute = timed(compute, 2, 5)[0] / 5
    ms_gather = timed(gather, 2, 5)[0] / 5

    # per-sub-band parity (untimed): this rank's bank against the oracle run with
    # (nchan/N, f0_g, max_delay_g); rank 0 additionally checks a gathered bank
    step_strong()
    torch.cuda.synchronize()

    def got_fn(a, n):
        return t_out[:, a:a + n].cpu().numpy()
    par = oracle_window_check(x_sub, got_fn, sb, [(0, 4096), (65536 + 3, 4096), (ntime - 4096 - md, 4096 + md)])
    bad = torch.tensor([0 if par.get('ok') else 1], device='cuda')
    dist.all_reduce(bad)
    gathered_ok = None
    if rank == 0:
        g = world - 1
        sg = subs[g]
        xg = np.ascontiguousarray(x_full[sg['chan0']:sg['chan0'] + nc])
        gathered_ok = oracle_window_check(xg, lambda a, n: t_bank[int(offs[g]):int(offs[g + 1]), a:a + n].cpu().numpy(),
                                          sg, [(30000, 4096)]).get('ok')

    # e2e: every rank H2D's its own sub-band from its own pinned buffer (NUMA-local),
    # FDMT, gather to rank 0, rank 0 D2H of the whole bank
    pinned_in = bf.empty((nc, ntime), dtype='i8', space='cuda_host')
    np.copyto(np.asarray(pinned_in), x_sub)
    a_in_e2e = bf.ndarray(base=t_in) if rank != 0 else a_in
    pinned_bank = bf.empty((int(offs[-1]), ntime), dtype='f32', space='cuda_host') if rank == 0 else None
    a_bank = bf.ndarray(base=t_bank) if rank == 0 else None

    def step_e2e():
        bf.copy_array(a_in_e2e, pinned_in)
        plan.execute_workspace(a_in_e2e, a_out, ws.ctypes.data, ws_size)
        gather()
        if rank == 0:
            bf.copy_array(pinned_bank, a_bank)

    ms_e2e = timed(step_e2e, 2, args.steps)[0] / args.steps
    del pinned_in, pinned_bank

    # cross-GPU FULL-BAND transform of the same gulp (SURVEY 8f.1): every rank
    # keeps its sub-band's channels, the merge tree is cut where it has `world`
    # sub-bands, the cut-step rows are exchanged with NCCL, rank 0 gathers the
    # bank.  The sub-bands of the scatter above are exactly the shards.
    fullband = None
    if not args.no_fullband:
        from bifrost_b200.fdmt_sharded import ShardedFdmt
        try:
            sf = ShardedFdmt().init(full['nchan'], full['max_delay'], full['f0'], full['df'])
            shard_ok = 1
        except Exception as e:                         # e.g. a world size the tree does not split into
            sf, shard_ok, shard_err = None, 0, str(e)
        agree = torch.tensor([shard_ok], device='cuda')
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        if int(agree.item()) == 1:
            x_loc = t_full[:nc] if rank == 0 else t_in
            t_fb = torch.zeros((full['max_delay'], ntime), dtype=torch.float32, device='cuda')
            ms_fb = timed(lambda: sf.execute(x_loc, t_fb, gather_to=0), 2, 5)[0] / 5
            ms_fb_nogather = timed(lambda: sf.execute(x_loc, t_fb), 2, 5)[0] / 5
            lay = sf.layout(ntime)
            wins = [(0, 2048), (70000 + 1, 2048), (ntime - 2048 - full['max_delay'], 2048 + full['max_delay'])]
            sf.execute(x_loc, t_fb, gather_to=0)
            torch.cuda.synchronize()
            fb_par = None
            if rank == 0:
                fb_par = oracle_window_check(x_full, lambda a, n: t_fb[:, a:a + n].cpu().numpy(), full, wins)
            # the same with phase 1 reading the peers' rows in place over NVLink (no exchange)
            peer = None
            if not args.fullband_peer:
                peer_ok = -1
            else:
              try:
                t_fb.zero_()
                sf.execute(x_loc, t_fb, gather_to=0, peer=True)
                torch.cuda.synchronize()
                peer_ok = 1
              except Exception as e:
                peer_ok, peer_err = 0, str(e)
            agree = torch.tensor([peer_ok], device='cuda')
            dist.all_reduce(agree, op=dist.ReduceOp.MIN)
            if int(agree.item()) == -1:
                peer = dict(available=None, note='not requested (--fullband-peer); see profiles/r02_sharded_2gpu.txt')
            elif int(agree.item()) == 1:
                peer_par = oracle_window_check(x_full, lambda a, n: t_fb[:, a:a + n].cpu().numpy(), full, wins) if rank == 0 else None
                ms_peer = timed(lambda: sf.execute(x_loc, t_fb, peer=True), 2, 5)[0] / 5
                peer = dict(what='phase 1 fetches every cut-step row straight from the HBM of the rank that produced it '
                                 '(CUDA IPC mappings, NVLink peer access; ' + ('cp.async.bulk' if os.environ.get('BFB_FDMT_PEER_TMA') == '1' else '16-byte loads') +
                                 '); NCCL carries two barriers per gulp, no data',
                            ms_per_step_without_gather=ms_peer, parity=peer_par)
            else:
                peer = dict(available=False, note=peer_err if not peer_ok else 'another rank failed')
            blk = lay['row_start']
            fullband = dict(what='ONE full-band dispersion bank [max_delay, ntime] of the gulp, channels partitioned over the '
                                 'ranks: local steps -> NCCL broadcast of every rank\'s block of cut-step rows -> each rank\'s '
                                 'delay blocks of the remaining steps -> NCCL gather on rank 0 (bifrost_b200/fdmt_sharded.py)',
                            split_step=lay['split_step'], ms_per_step=ms_fb, ms_per_step_without_gather=ms_fb_nogather,
                            value=NCHAN * NTIME_OUT / (ms_fb * 1e-3) / 1e6, unit='Msamples/s',
                            exchange_bytes_per_rank=int((blk[-1] - (blk[rank + 1] - blk[rank])) * lay['pitch']),
                            gather_bytes=int(sum(nd for _, nd, o in lay['blocks'] if o != 0) * ntime * 4),
                            parity=fb_par, peer_access=peer)
            del t_fb, sf
        else:
            fullband = dict(available=False, note=shard_err if not shard_ok else 'another rank could not build the sharded plan')

    # replicas (weak scaling, no collective): every rank its own full gulp
    del ws
    wr = workload(rank)
    t_rin = torch.from_numpy(make_input(wr, 1234 + rank)).cuda() if rank != 0 else t_full
    a_rin = bf.ndarray(base=t_rin)
    a_rout = bf.empty((wr['max_delay'], wr['ntime']), dtype='f32', space='cuda')
    rplan = Fdmt()
    rplan.init(wr['nchan'], wr['max_delay'], wr['f0'], wr['df'])
    ms_rep = timed(lambda: rplan.execute(a_rin, a_rout), 3, 10)[0] / 10

    if rank != 0:
        return
    samples = NCHAN * NTIME_OUT
    nvlink_scatter = (world - 1) * nc * ntime
    nvlink_gather = int(offs[-1] - offs[1]) * ntime * 4
    alg_bytes = ntime * (NCHAN + 4 * int(offs[-1]))
    line = dict(metric=METRIC, value=samples / (ms_step * 1e-3) / 1e6, unit='Msamples/s', n_gpus=world,
                steps=args.steps, warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True,
                scaling='strong', vs_baseline=None,
                dtype='u16/f32 (exact integers; bit-identical to the reference\'s f32)', data='synthetic',
                config=bench_config(world), host_numa=numa,
                comm=dict(collective='ncclSend/ncclRecv groups (torch.distributed.batch_isend_irecv)',
                          nvlink_bytes_per_step=int(nvlink_scatter + nvlink_gather),
                          scatter_bytes=int(nvlink_scatter), gather_bytes=int(nvlink_gather),
                          ms_scatter=ms_scatter, ms_compute_max_rank=ms_compute, ms_gather=ms_gather,
                          limit='the gather: rank 0 receives (N-1)/N of the 420 MB bank over its NVLink ingress, '
                                'which takes longer than one GPU needs to compute the whole bank'),
                parity=dict(per_subband_ok=bool(int(bad.item()) == 0), gathered_bank_ok=gathered_ok,
                            how='each rank: its bank vs oracle/fdmt_c.c with (nchan/N, f0_g, max_delay_g) on 3 windows, '
                                'bit for bit; rank 0: one gathered bank after the collective'),
                roofline=dict(bound='nvlink+hbm', achieved=alg_bytes / (ms_step * 1e-3) / 1e9, unit='GB/s',
                              peak=peaks['hbm_gbs'], peak_source=peak_kind,
                              frac=alg_bytes / (ms_step * 1e-3) / 1e9 / peaks['hbm_gbs'],
                              algorithmic_bytes=alg_bytes, traffic=None,
                              note='single-GPU HBM peak as denominator; the step is NVLink-bound (comm.limit)'),
                e2e=dict(value=samples / (ms_e2e * 1e-3) / 1e6, unit='Msamples/s', ms_per_step=ms_e2e,
                         how='every rank: pinned host sub-band -> H2D -> Fdmt.execute -> NCCL gather; rank 0: D2H of '
                             'the whole bank to pinned host memory; one stream per rank, max over ranks',
                         h2d_bytes_per_step=int(NCHAN * ntime), d2h_bytes_per_step=int(offs[-1]) * ntime * 4),
                fullband=fullband,
                replicas=dict(scaling='weak', what='every rank its own full 4096-chan gulp (sub-band above the '
                                                   'previous rank\'s), no collective; max over ranks',
                              ms_per_step=ms_rep, value=samples * world / (ms_rep * 1e-3) / 1e6, unit='Msamples/s'),
                gpu_launches=int(launches), clocks=clocks)
    print(json.dumps(line))


if __name__ == '__main__':
    main()
