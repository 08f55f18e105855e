#!/usr/bin/env python
"""bench.py -- protein pairs/sec of the IEGMN hot path (IEGMN layers + keypoints + Kabsch).

    python bench.py --gpus N --steps K --warmup W            # B200 engine (this repo)
    python bench.py --impl reference --gpus N ...            # CPU reference arm (oracle port, rank 0)
    python bench.py --workload {db5-shaped,db5-testset,large,train} ...
    python bench.py ... --dump-outputs DIR                  # also write the last timed step's outputs as DIR/<name>.npy

Workloads (BASELINE.json configs):
  db5-shaped   (headline, north_star / configs[1] shape) synthetic DB5.5-shaped residue graphs, 200+200 residues, k=10,
               8-layer IEGMN with the shipped DIPS checkpoint's weights, batched inference, 370 pairs/step/GPU (the batch is
               sized to the machine: 370 pairs = 1480 attention tiles, 1157 node tiles and 12 334 edge tiles, i.e. 5.00 / 3.91 /
               41.7 rounds of the 296 resident tile groups of a B200, where 256 pairs left the last attention / node round
               54 % / 30 % empty: +5.5 % pairs/s).
  db5-testset  (configs[1] literally) 25 pairs with the (N_l, N_r) sizes of the DB5.5 test set as ONE ragged batch.
  large        (configs[4]) synthetic 2000+2000-residue complexes, 8 pairs/step/GPU.
  train        (configs[2]/[3]) DIPS-shaped ragged batch of 32 pairs/GPU, 5-layer shared IEGMN, forward + losses
               (MSE, exact EMD, body intersection) + backward + flat NCCL gradient all-reduce + clip + Adam.
Pairs shard across ranks by estimated cost (equidock_public_b200.sharding) with no data-path collective (weak scaling).
One step = one pass of the hot path over the rank's batch.  Prints ONE JSON line on rank 0.

Timing protocol: W warm-up steps, then R repetitions (default 5) of EXACTLY K steps, each repetition bracketed by a
barrier + torch.cuda.synchronize() on both sides and timed with CUDA events on the launching stream; a repetition's
time is the MAX over ranks; `value` is the MEDIAN repetition (all repetitions are in `rep_ms`).  Clocks are sampled
in-process through NVML from one second before the first repetition to the end of the last.
"""
from __future__ import annotations

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
sys.path.insert(0, os.path.join(ROOT, 'tests'))

KNN = 10
# (N_l, N_r) of the 25 DB5.5 test pairs (SURVEY 8d: min 55+574 ... max 548+2000, sum N_l 4121, sum N_r 8709); the five
# fixture pairs carry their true sizes, the others are drawn once (seed 55) to match the published totals
DB5_TEST_SIZES = None


def db5_test_sizes():
    global DB5_TEST_SIZES
    if DB5_TEST_SIZES is None:
        known = [(172, 223), (327, 368), (548, 2000), (95, 102), (125, 195), (55, 574)]
        rng = np.random.default_rng(55)
        rest_l, rest_r = 4121 - sum(a for a, _ in known), 8709 - sum(b for _, b in known)
        n = 25 - len(known)
        wl, wr = rng.dirichlet(np.full(n, 4.0)), rng.dirichlet(np.full(n, 4.0))
        ls = np.maximum(40, np.round(wl * rest_l)).astype(int)
        rs = np.maximum(60, np.round(wr * rest_r)).astype(int)
        ls[-1] += rest_l - ls.sum()
        rs[-1] += rest_r - rs.sum()
        DB5_TEST_SIZES = known + [(int(a), int(b)) for a, b in zip(ls, rs)]
    return DB5_TEST_SIZES


WORKLOADS = {
    'db5-shaped': dict(n_layers=8, ckpt='dips', pairs_per_gpu=370, flop_per_pair=1.781e9, bytes_per_pair=6.20e6,
                       text='synthetic DB5.5-shaped 200+200 residues k=10, 8-layer IEGMN (DIPS checkpoint weights), '
                            'batched inference'),
    'db5-testset': dict(n_layers=8, ckpt='dips', pairs_per_gpu=25, flop_per_pair=None, bytes_per_pair=None,
                        text='25 synthetic pairs with the DB5.5 test set sizes (55+574 ... 548+2000) as ONE ragged '
                             'batch, k=10, 8-layer IEGMN (DIPS checkpoint weights), batched inference'),
    'large': dict(n_layers=8, ckpt='dips', pairs_per_gpu=8, flop_per_pair=32.7e9, bytes_per_pair=62.0e6,
                  text='synthetic 2000+2000-residue complexes k=10, 8-layer IEGMN (DIPS checkpoint weights), '
                       'batched inference'),
    'train': dict(n_layers=5, ckpt='db5', pairs_per_gpu=32, flop_per_pair=None, bytes_per_pair=None,
                  text='synthetic DIPS-shaped ragged pairs (60..1112 residues, median 225+214), k=10, 5-layer shared '
                       'IEGMN (DB5 checkpoint weights), training step: forward + MSE/EMD/intersection losses + backward '
                       '+ flat gradient all-reduce + clip + Adam'),
}


def pair_sizes(workload: str, n_pairs: int, seed: int = 0):
    """Global (N_l, N_r) list of the job's pairs -- identical on every rank."""
    if workload == 'db5-shaped':
        return [(200, 200)] * n_pairs
    if workload == 'large':
        return [(2000, 2000)] * n_pairs
    if workload == 'db5-testset':
        base = db5_test_sizes()
        return [base[i % 25] for i in range(n_pairs)]
    rng = np.random.default_rng(1000 + seed)      # DIPS test distribution (SURVEY 8d config 3): log-normal, clipped
    l = np.clip(np.exp(rng.normal(np.log(225), 0.55, n_pairs)), 60, 1112).astype(int)
    r = np.clip(np.exp(rng.normal(np.log(214), 0.55, n_pairs)), 61, 1112).astype(int)
    return [(int(a), int(b)) for a, b in zip(l, r)]


def workload_config(args, world: int):
    """The SAME dict in both arms (driver: vs_reference.same_config)."""
    w = WORKLOADS[args.workload]
    return {'workload': f"{w['text']}, {args.pairs_per_gpu} pairs/step/GPU", 'pairs_per_gpu': args.pairs_per_gpu,
            'parallelism': f'dp{world} (pairs sharded by cost, no data-path collective)'}


def make_pairs(args, rank: int, world: int):
    """This rank's cost-balanced contiguous shard of the job's global pair list (sharding.shard_bounds); every pair is
    generated from its own seed (job seed, global pair index), so the data do not depend on the world size."""
    from equidock_public_b200 import sharding, synthetic
    sizes = pair_sizes(args.workload, args.pairs_per_gpu * world)
    L = WORKLOADS[args.workload]['n_layers']
    costs = [sharding.pair_cost(a, b, KNN * a, KNN * b, L) for a, b in sizes]
    lo, hi = sharding.my_shard(costs, world, rank)
    pairs = [synthetic.synthetic_pair(np.random.default_rng([args.seed, i]), sizes[i][0], sizes[i][1], KNN)
             for i in range(lo, hi)]
    return pairs, (lo, hi), sizes


def edge_stage_algorithmic_bytes(n_nodes: int, n_edges: int) -> float:
    """Compulsory HBM bytes of ONE edge-stage launch (one layer): he (27 fp32 / edge), CSR ids (4(E+N+2)), coordinates
    in + out (12 B / node each), and the Psrc / Pdst rows the design makes compulsory by projecting per node instead of
    per edge (2 x 256 B per node, each read at least once)."""
    return 4.0 * 27 * n_edges + 4.0 * (n_edges + n_nodes + 2) + 12.0 * 2 * n_nodes + 512.0 * n_nodes


def edge_stage_algorithmic_flops(n_edges: int, dh: int = 64) -> float:
    """fp32 FLOPs of ONE edge-stage launch in the reference formulation (SURVEY 8(d) per-layer edge terms, MAC = 2):
    edge_mlp.0 on cat[h_src, h_dst, he, rbf] (2E(2 dh + 42) 64), edge_mlp.4 and coors_mlp.0 (2E 64 64 each),
    coors_mlp.4 (2E 64)."""
    return n_edges * (2.0 * (2 * dh + 42) * 64 + 2 * 2.0 * 64 * 64 + 2.0 * 64)


# bf16 FLOPs the tensor-core edge stage really issues per edge: (K 48 x N 64 + K 64 x N 128) MACs x 6 split products
EDGE_TC_BF16_FLOP_PER_EDGE = 2.0 * (48 * 64 + 64 * 128) * 6
# dram__bytes_read.sum + dram__bytes_write.sum of one edge_stage_tc_kernel launch of the headline workload
# (ncu --set full, profiles/): filled from the committed summary of the current round
EDGE_TC_NCU_TRAFFIC_BYTES = {370: 286.8e6,   # profiles/r02_final_edge_stage_tc_370pairs_ncu_summary.txt: 255.1 MB read + 31.7 MB written
                             256: 195.3e6}   # profiles/r02_final_edge_stage_tc_ncu_summary.txt: 176.5 MB read + 18.7 MB written


def bind_to_gpu_numa(local_rank: int):
    """Pins this process to the cores of the NUMA node its GPU hangs off (before any allocation, so that first-touch
    places the pinned staging buffers there too).  Eight unpinned ranks otherwise stream 20+ GB/s each of pinned H2D
    traffic across the socket interconnect.  Silent no-op where sysfs does not say."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(':')[0]) == 8:
            bus = bus[4:]
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {'numa_node': node, 'cpus': len(cpus)}
    except Exception:
        return None
    return None


class ClockSampler:
    """SM clock / throttle reasons of one GPU sampled in-process through NVML every 100 ms (falls back to one
    `nvidia-smi` child started well before the timed region).  Started >= 1 s before the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int):
        self.gpu, self.sm, self.smax, self.reasons, self.power = gpu_index, [], [], set(), []
        self.stop_flag, self.thread, self.proc, self.rows = threading.Event(), None, None, []
        self.mode = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nv = pynvml
            self.smax.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)))
            self.mode = 'nvml'
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.mode = 'nvidia-smi'
            try:
                self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                              '-lms', '200', '-i', str(self.gpu)], stdout=subprocess.PIPE,
                                             stderr=subprocess.DEVNULL, text=True)
                threading.Thread(target=self._pump, daemon=True).start()
            except OSError:
                self.proc = None

    def _loop(self):
        nv = self.nv
        bits = {'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown,
                'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """Samples before this call (the >= 1 s lead-in) are dropped from the medians."""
        self.lead = len(self.sm) if self.mode == 'nvml' else len(self.rows)

    def stop(self):
        lead = getattr(self, 'lead', 0)
        if self.mode == 'nvml':
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            sm = self.sm[lead:] or self.sm
            return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(self.smax) if self.smax else None,
                    'reasons': sorted(self.reasons), 'samples': len(sm), 'source': 'nvml in-process, 100 ms',
                    'power_w_max': max(self.power) if self.power else None}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows[lead:]:
            f = [c.strip() for c in r.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi child, 200 ms'}


def measured_peaks():
    """(HBM GB/s, dense bf16 TFLOP/s sustained, source).  The edge stage is timed inside a long step, so the sustained
    tensor figure is the denominator."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        with open(p) as fh:
            d = json.load(fh)
        return (float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1380.0))),
                'measured (MEASURED_PEAKS.json)')
    return 6650.0, 1380.0, 'fallback (B200_PROFILING.md)'


def effective_cores() -> int:
    """Host cores this process may really use: min(affinity, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


# ---- CPU reference arm ------------------------------------------------------------------------------------------------
_REF = {}


def _ref_init(threads, ckpt, n_layers, train):
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import golden_io as gio
    import iegmn_oracle_torch as ot
    torch.set_num_threads(threads)
    sd, margs = gio.load_checkpoint(ckpt), gio.load_args(ckpt)
    _REF['model'] = ot.TorchOracle(sd, n_layers, margs['skip_weight_h'], margs['x_connection_init'],
                                   margs['leakyrelu_neg_slope'], margs['num_att_heads'])
    _REF['train'] = train
    if train:
        _REF['model'].parameters_for_grad()


def _ref_run(pairs):
    if _REF['train']:
        import train_oracle
        for p in pairs:
            train_oracle.reference_train_pair(_REF['model'], p)
        return len(pairs)
    for p in pairs:
        _REF['model'].forward_pair(*p)
    return len(pairs)


class ReferencePool:
    """The CPU reference arm on ALL usable host cores: `workers` processes x `threads` torch threads, each
    running the oracle's torch port one pair per call (pairs are independent, like the GPU shards)."""

    def __init__(self, cores: int, workload: str, threads: int = 4):
        import multiprocessing as mp
        w = WORKLOADS[workload]
        self.threads = min(threads, cores)
        self.workers = max(1, cores // self.threads)
        self.pool = mp.get_context('spawn').Pool(self.workers, initializer=_ref_init,
                                                 initargs=(self.threads, w['ckpt'], w['n_layers'], workload == 'train'))

    def run(self, pairs):
        chunks = [pairs[i::self.workers] for i in range(self.workers)]
        return sum(self.pool.map(_ref_run, [c for c in chunks if c]))

    def close(self):
        self.pool.close()
        self.pool.join()


METRIC = {'db5-shaped': 'protein_pairs_per_sec_iegmn_fwd_kabsch', 'db5-testset': 'protein_pairs_per_sec_iegmn_fwd_kabsch',
          'large': 'protein_pairs_per_sec_iegmn_fwd_kabsch', 'train': 'protein_pairs_per_sec_iegmn_train_step'}


def run_reference(args, rank, world):
    """CPU reference arm: the oracle's PyTorch port (the reference's own op sequence, fp32, all host threads), one pair
    per call like src/inference_rigid.py.  Each step = the rank-0 shard of the SAME workload the engine arm times
    (bounded with --ref-sample for the large workloads); rank 0 only."""
    if rank != 0:
        return
    cores = effective_cores()
    if args.workload == 'train':
        import bench_train
        pairs, _, _ = bench_train.make_train_pairs(args, 0, world, sys.modules[__name__])
    else:
        pairs, _, _ = make_pairs(args, 0, world)
    pool = ReferencePool(cores, args.workload)
    for _ in range(max(1, min(args.warmup, 2))):
        pool.run(pairs[:pool.workers])
    if args.ref_sample > 0:
        sample = min(args.ref_sample, len(pairs))
    else:   # the whole step batch, unless K steps of it would not end within a few minutes on this box: then a bounded prefix
        ncal = min(len(pairs), 2 * pool.workers)
        tc = time.perf_counter()
        pool.run(pairs[:ncal])
        rate = ncal / max(time.perf_counter() - tc, 1e-6)
        sample = min(len(pairs), max(pool.workers, int(rate * args.ref_budget_s / max(args.steps, 1))))
    pairs = pairs[:sample]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pool.run(pairs)
    dt = time.perf_counter() - t0
    pool.close()
    val = args.steps * sample / dt
    line = {'impl': 'reference', 'metric': METRIC[args.workload], 'value': val, 'unit': 'pairs/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, world),
            'cpu_baseline': {'value': val, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                             'sample': f'each step = {sample} pairs of the {args.pairs_per_gpu}-pair step batch, one pair '
                                       f'per call like src/inference_rigid.py; torch fp32 port of the reference op '
                                       f'sequence, {pool.workers} processes x {pool.threads} threads = {cores} usable host cores'},
            'e2e': {'value': val, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ---- engine arm -------------------------------------------------------------------------------------------------------

class Dist:
    def __init__(self, world, dev, torch):
        self.world, self.dev, self.torch = world, dev, torch
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group('nccl', device_id=dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather(self, v):
        if self.world == 1:
            return [v]
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def timed_reps(torch, D: Dist, reps: int, body):
    """R repetitions of `body()` (= exactly K steps incl. the wait for the last one), each bracketed by barrier + sync and
    timed with CUDA events on the current stream.  Returns (per-rep max-over-ranks ms, per-rank ms of the median rep)."""
    rep_ms, per_rank = [], []
    for _ in range(reps):
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        body()
        e1.record()
        D.barrier()
        mine = e0.elapsed_time(e1)
        per_rank.append(D.gather(mine))
        rep_ms.append(max(per_rank[-1]))
    med = int(np.argsort(rep_ms)[len(rep_ms) // 2])
    return rep_ms, med, per_rank[med]


OUTPUT_NAMES = ('ligand_coors', 'keypts_ligand', 'keypts_receptor', 'rotation', 'translation')
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, result, limit: int = DUMP_LIMIT_BYTES):
    """Writes one step's result -- the model's 5-tuple of per-pair lists -- as out_dir/<name>.npy: the ligand coordinates
    of all pairs concatenated in pair order, the other outputs stacked.  float64 outputs stay float64, the others are
    written as float32.  Where the whole result exceeds `limit` bytes, a fixed random subset of the pairs (seed 0, kept
    in pair order) that fits is written instead, so that two runs with the same arguments write the same pairs."""
    import torch
    n_lig = np.array([c.shape[0] for c in result[0]])
    host = {'ligand_coors': torch.cat(result[0]).cpu().numpy()}
    host.update({k: torch.stack(v).cpu().numpy() for k, v in zip(OUTPUT_NAMES[1:], result[1:])})
    host = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32, copy=False) for k, v in host.items()}
    lig = host['ligand_coors']
    pair_bytes = n_lig * lig.itemsize * lig.shape[1] + sum(host[k][0].nbytes for k in OUTPUT_NAMES[1:])
    keep = np.arange(len(n_lig))
    if pair_bytes.sum() > limit:
        order = np.random.default_rng(0).permutation(len(n_lig))
        keep = np.sort(order[np.cumsum(pair_bytes[order]) <= limit])
        start = np.concatenate([[0], np.cumsum(n_lig)[:-1]])
        rows = np.concatenate([np.arange(start[i], start[i] + n_lig[i]) for i in keep]) if len(keep) else []
        host = {k: (v[rows] if k == 'ligand_coors' else v[keep]) for k, v in host.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), v)
    print(f'bench: wrote the last timed step\'s outputs of {len(keep)} of {len(n_lig)} pairs to {out_dir}',
          file=sys.stderr, flush=True)
    return keep


def run_engine(args, rank, local_rank, world):
    numa = bind_to_gpu_numa(local_rank) if not args.no_numa_bind else None
    import torch
    import golden_io as gio
    from equidock_public_b200 import hetero_graph as hg
    from equidock_public_b200 import synthetic
    from equidock_public_b200 import engine as engine_mod
    from equidock_public_b200.engine import IEGMNEngine

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    D = Dist(world, dev, torch)
    wl = WORKLOADS[args.workload]
    pairs, (lo, hi), sizes = make_pairs(args, rank, world)
    B = len(pairs)
    total_pairs = len(sizes)
    sd, margs = gio.load_checkpoint(wl['ckpt']), gio.load_args(wl['ckpt'])
    margs = dict(margs)
    margs['iegmn_n_lays'] = wl['n_layers']
    if wl['n_layers'] != int(gio.load_args(wl['ckpt'])['iegmn_n_lays']):
        raise SystemExit('workload depth must match the checkpoint')
    model = gio.build_model(wl['ckpt'], dev, sd=sd, args=margs)
    host_batch = hg.batch_pairs(synthetic.to_torch_pairs(pairs)).pin_memory()
    dev_batches = [host_batch.to(dev) for _ in range(2)]
    n_nodes, n_edges = host_batch.num_nodes(), host_batch.num_edges()
    K, W, R = args.steps, max(args.warmup, 3), args.reps
    n_layers = wl['n_layers']

    # ---- device-resident throughput ("value"): CUDA-graph replay, two graphs (two steps) in flight ------------------
    use_graph = not args.no_cuda_graph and not engine_mod._PY_FORWARD
    if use_graph:
        graphs = [model.graphed(b) for b in dev_batches]
        launch = lambda i: graphs[i & 1].launch()
    else:
        launch = lambda i: model.forward_async(dev_batches[i & 1], 0)

    last = None

    def value_body():
        nonlocal last
        pending = None
        for i in range(K):          # step i is launched before step i-1's status words are read
            nxt = launch(i)
            if pending is not None:
                pending.result()
            pending = nxt
        pending.result()
        last = pending

    for _ in range(W):
        launch(0).result()
    sampler = ClockSampler(local_rank)
    sampler.start()
    D.barrier()
    t_lead = time.perf_counter()
    while time.perf_counter() - t_lead < 1.0:      # >= 1 s of sampler lead-in, GPU kept busy so clocks are ramped
        launch(0).result()
    sampler.mark()
    rep_ms, med, per_rank_ms = timed_reps(torch, D, R, value_body)
    ms_total = rep_ms[med]
    value = total_pairs * K / (ms_total * 1e-3)
    # The loop keeps only the last step's handle: holding its result (~2000 tensor views) across repetitions moved one
    # of the interpreter's full garbage collections (~33 ms) into the timed window of the default run.  result()
    # re-reads that step's output buffers, so it must run before anything is launched again.
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f'rank{rank}'), last.result())

    # ---- instrumented pass: the same K steps on the eager path with CUDA events around every edge / node stage ------
    timer = engine_mod.NativeStageTimer()
    timer.reserve(K, n_layers)                      # all events are created here, outside the timed loop
    orig_forward = IEGMNEngine.forward
    IEGMNEngine.forward = lambda self, *a, **k: orig_forward(self, *a, stage_timer=timer, **k)
    D.barrier()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    pending = None
    for i in range(K):
        nxt = model.forward_async(dev_batches[i & 1], 0)
        if pending is not None:
            pending.result()
        pending = nxt
    pending.result()
    i1.record()
    D.barrier()
    IEGMNEngine.forward = orig_forward
    instr_ms = D.max(i0.elapsed_time(i1))

    # ---- end to end through the public API with HOST buffers ("e2e") -------------------------------------------------
    # every step: H2D of that step's pinned inputs, the forward, D2H of coordinates / R / t into pinned memory;
    # serving.PipelinedInference overlaps the copy of batch k+1 with the kernels of batch k (3 slots, CUDA graphs).
    from equidock_public_b200.serving import PipelinedInference
    pipe = PipelinedInference(model, dev, use_cuda_graph=use_graph)
    d2h_bytes = 0

    def drain(n_steps):
        nonlocal d2h_bytes
        last = None
        for res in pipe.run(host_batch for _ in range(n_steps)):
            last = res
        last['_event'].synchronize()
        d2h_bytes = sum(int(v.numel() * v.element_size()) for k, v in last.items() if k != '_event')

    drain(max(W, 4))
    e2e_rep = []
    for _ in range(R):
        D.barrier()
        t0 = time.perf_counter()
        drain(K)
        D.barrier()
        e2e_rep.append(D.max(time.perf_counter() - t0))
    # ---- e2e from RESIDUES: compact all-atom inputs over PCIe, graph construction + forward as one CUDA graph -----------
    e2e_res = None
    if args.workload == 'db5-shaped' and use_graph and not args.no_residue_e2e:
        from equidock_public_b200.graph_build import ResidueBatch, ResidueGraphedForward
        rpairs = [synthetic.synthetic_residue_pair(np.random.default_rng([args.seed, 11, i]), sizes[i][0], sizes[i][1])
                  for i in range(lo, hi)]
        rb = ResidueBatch(rpairs, pin=True)
        slots = [ResidueGraphedForward(model, rb, dev) for _ in range(2)]
        pinned = [{k: torch.empty(sh, dtype=torch.float32, pin_memory=True) for k, sh in
                   (('ligand_coors', (sum(rb.n_lig), 3)), ('rotation', (B, 3, 3)), ('translation', (B, 1, 3)))} for _ in range(2)]

        def res_body(n_steps):
            pend = None
            for i in range(n_steps):
                sl = slots[i & 1]
                sl.upload(rb)                        # H2D of this step's inputs (compute stream: 13 MB, no overlap needed)
                nxt = (sl.launch(), i & 1)
                if pend is not None:
                    raw = pend[0].raw_result()
                    for k, hb in pinned[pend[1]].items():
                        hb.copy_(raw[k], non_blocking=True)
                pend = nxt
            raw = pend[0].raw_result()
            for k, hb in pinned[pend[1]].items():
                hb.copy_(raw[k], non_blocking=True)
            torch.cuda.synchronize()

        res_body(W)
        rr_rep = []
        for _ in range(R):
            D.barrier()
            t0 = time.perf_counter()
            res_body(K)
            D.barrier()
            rr_rep.append(D.max(time.perf_counter() - t0))
        e2e_res = {'value': total_pairs * K / float(np.median(rr_rep)), 'unit': 'pairs/s', 'h2d_bytes_per_step': rb.nbytes(),
                   'd2h_bytes_per_step': sum(int(v.numel() * 4) for v in pinned[0].values()), 'rep_s': rr_rep,
                   'note': 'inputs = all-atom coordinates per residue (synthetic.synthetic_residue_pair); the k-NN graph and its '
                           '27 edge features are built on the device (graph_build.cu) inside the same CUDA graph as the forward'}
    clocks = sampler.stop()
    e2e_s = float(np.median(e2e_rep))
    e2e_val = total_pairs * K / e2e_s
    h2d_bytes = host_batch.nbytes()
    rank_clocks = D.gather(clocks.get('sm_mhz') or 0.0)

    if rank != 0:
        return D
    hbm_peak, tc_peak, peak_src = measured_peaks()
    edge_ms = timer.mean_ms('edge_stage')
    node_ms = timer.mean_ms('node_stage')
    alg = edge_stage_algorithmic_bytes(n_nodes, n_edges)
    ach = alg / (edge_ms * 1e-3) / 1e9
    alg_flops = edge_stage_algorithmic_flops(n_edges)
    step_ms = ms_total / K
    sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    line = {
        'metric': METRIC[args.workload], 'value': value, 'unit': 'pairs/s', 'n_gpus': world,
        'steps': K, 'warmup': W, 'ms_per_step': step_ms, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, world),
        'notes': {'l2': f'per-step working set {(n_edges * 108 + n_nodes * 3880) / 1e6:.0f} MB vs 126 MB L2; two device '
                        f'batches alternate',
                  'coords_and_head_dtype': 'f64',
                  'value_protocol': f'median of {R} repetitions of the {K}-step loop, each bracketed by barrier+sync, CUDA '
                                    f'events, max over ranks; forward replayed from a CUDA graph' if use_graph else
                                    f'median of {R} repetitions of the {K}-step loop (eager launches)',
                  'topology_cached': 'value reuses each device batch\'s GraphPlan (CSR / tile lists built once); only '
                                     'e2e rebuilds the topology arrays every step (GraphPlan.refresh)',
                  'numa': numa, 'shard': [lo, hi], 'pairs_total': total_pairs},
        'rep_ms': rep_ms, 'per_rank_ms_per_step': [m / K for m in per_rank_ms],
        'e2e': {'value': e2e_val, 'unit': 'pairs/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': d2h_bytes,
                'rep_s': e2e_rep},
        'e2e_from_residues': e2e_res,
        'gpu_launches': IEGMNEngine.launches_per_forward(n_layers) * K * R,
        'clocks': {**clocks, 'per_rank_sm_mhz': rank_clocks},
        'roofline': {'kernel': 'edge_stage_tc_kernel', 'bound': 'tensor', 'achieved': alg_flops / (edge_ms * 1e-3) / 1e12,
                     'peak': tc_peak, 'unit': 'TFLOP/s', 'frac': alg_flops / (edge_ms * 1e-3) / 1e12 / tc_peak,
                     'traffic': EDGE_TC_NCU_TRAFFIC_BYTES.get(B) if args.workload == 'db5-shaped' else None,
                     'peak_source': peak_src + ', sustained bf16',
                     'algorithmic_flops_per_launch': alg_flops, 'launch_ms': edge_ms,
                     'launch_ms_source': f'CUDA events recorded by eqd_iegmn_forward around every edge-stage launch over an '
                                         f'instrumented (eager) pass of the same {K} steps, {instr_ms / K:.3f} ms/step',
                     'issued_bf16_tflops': n_edges * EDGE_TC_BF16_FLOP_PER_EDGE / (edge_ms * 1e-3) / 1e12,
                     'issued_bf16_frac': n_edges * EDGE_TC_BF16_FLOP_PER_EDGE / (edge_ms * 1e-3) / 1e12 / tc_peak,
                     'hbm': {'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                             'algorithmic_bytes_per_launch': alg},
                     'share_of_step': timer.total_ms('edge_stage') / K / step_ms,
                     'share_of_instrumented_step': timer.total_ms('edge_stage') / instr_ms,
                     'note': 'fp32-accurate GEMMs as 6 bf16 split products on tcgen05 (bf16x6): the tensor ceiling in '
                             'algorithmic fp32 FLOPs is peak x 38272 / 135168 = 0.283 x peak; AI ~290 FLOP/B, so the HBM '
                             'fraction (north star) is small by construction'},
        'kernels_ms': {'edge_stage': edge_ms, 'node_stage': node_ms,
                       'edge_share': timer.total_ms('edge_stage') / K / step_ms,
                       'node_share': timer.total_ms('node_stage') / K / step_ms},
    }
    if wl['flop_per_pair']:
        line['step_roofline'] = {'hbm_frac': value / world * wl['bytes_per_pair'] / 1e9 / hbm_peak,
                                 'fp32_tflops': value / world * wl['flop_per_pair'] / 1e12, 'fp32_peak_tflops': fp32_peak,
                                 'fp32_frac': value / world * wl['flop_per_pair'] / 1e12 / fp32_peak,
                                 'algorithmic': f"SURVEY 8(d): {wl['flop_per_pair'] / 1e9:.3f} GFLOP, "
                                                f"{wl['bytes_per_pair'] / 1e6:.2f} MB per pair (reference formulation)"}
    timer.close()
    if world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline(pairs, args.cpu_seconds, args.workload)
    print(json.dumps(line), flush=True)
    return D


def cpu_baseline(pairs, budget_s, workload):
    """Oracle port timed on this box's usable host cores on a bounded sample of the same workload."""
    cores = effective_cores()
    pool = ReferencePool(cores, workload)
    pool.run(pairs[:pool.workers])                       # warm-up: imports, weights, first-call allocations
    t0 = time.perf_counter()
    pool.run(pairs[:2 * pool.workers])
    rate = min(len(pairs), 2 * pool.workers) / (time.perf_counter() - t0)
    n = int(min(len(pairs), max(2 * pool.workers, rate * budget_s)))
    t0 = time.perf_counter()
    done = pool.run(pairs[:n])
    dt = time.perf_counter() - t0
    pool.close()
    return {'value': done / dt, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
            'sample': f'first {done} pairs of the step batch, one pair per call, torch fp32 port of the reference op '
                      f'sequence, {pool.workers} processes x {pool.threads} threads'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--reps', type=int, default=5, help='repetitions of the K-step timed loop (value = median)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='db5-shaped', choices=sorted(WORKLOADS))
    ap.add_argument('--pairs-per-gpu', type=int, default=0, help='0 = the workload\'s default')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--ref-sample', type=int, default=0,
                    help='pairs per step of the CPU reference arm (0 = the whole rank-0 step batch, like the engine arm)')
    ap.add_argument('--ref-budget-s', type=float, default=240.0,
                    help='CPU reference arm: shrink the per-step sample so that the K timed steps fit in about this many seconds')
    ap.add_argument('--cpu-seconds', type=float, default=15.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-cuda-graph', action='store_true')
    ap.add_argument('--no-numa-bind', action='store_true')
    ap.add_argument('--no-residue-e2e', action='store_true')
    ap.add_argument('--watchdog-seconds', type=int, default=1500,
                    help='abort (with a stack dump) instead of stalling forever if the run has not finished by then')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32 / float64, '
                         'at most 64 MB: a fixed sample of the pairs beyond that); with several ranks, DIR/rank<r>/')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl == 'reference' or args.workload == 'train'):
        ap.error('--dump-outputs needs an inference workload of the engine arm: the train workload updates the weights '
                 'during a clock-timed lead-in, so its last step is not reproducible, and the reference arm keeps no outputs')
    if args.pairs_per_gpu <= 0:
        args.pairs_per_gpu = WORKLOADS[args.workload]['pairs_per_gpu']
    if args.watchdog_seconds > 0:
        import faulthandler
        faulthandler.dump_traceback_later(args.watchdog_seconds, exit=True)
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if args.workload == 'train':
        import bench_train
        D = bench_train.run(args, rank, local_rank, world, sys.modules[__name__])
    else:
        D = run_engine(args, rank, local_rank, world)
    if D is not None:
        D.close()


if __name__ == '__main__':
    main()
