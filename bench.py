#!/usr/bin/env python
"""bench.py -- queries/sec of the PQ-HNSW search path (BASELINE.json configs[1]: 1M x 128d fp32,
M=8 PQ, HNSW M=16 ef_construction=200, ef=64, k=10) on N B200s of one node.

A "step" is one pass of the hot path (ADC tables -> HNSW walk -> top-k; since round 2 ONE kernel, hnsw_walk4,
which builds each query's table in shared memory) over one batch of synthetic queries.  Prints ONE JSON line (rank 0):
  value     : whole-job QPS with the query batch already resident in HBM (device in, device out)
  e2e       : same metric through the host-buffer C-ABI call (H2D of queries + K1 + K3 + D2H of results)
  roofline  : dominant kernel (K3 walk): algorithmic bytes / CUDA-event time vs measured HBM peak
  cpu_baseline : the C oracle port timed on the host cores on a bounded sample of the same batch
`--impl reference` times the reference's own CPU path (oracle/_ref: compiled from /root/reference)
on the same config: batched get_dist_mat + knn_query with all host threads.

Multi-GPU (`torchrun ... bench.py --gpus N`): the index is replicated (1M x 384 B records = 384 MB
fits every GPU) and every rank serves its own query batch -> no data-path collective, weak
scaling.  `--mode shard` range-shards the base vectors instead (one graph per rank, labels =
global ids), replicates the queries and merges per-shard top-k with one NCCL all-gather + the
merge kernel.  With N > 1 the default run ALSO times that sharded step and reports it under the key
"shard" of the same JSON line (its QPS is what one GPU reaches on an N/G-node graph: sharding buys capacity,
not speed, at a size that fits one GPU -- configs[2] / configs[4] are the sizes it exists for).
"""
import argparse
import atexit
import hashlib
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
# codebooks and built indexes are cached outside the tree, which may be read-only
CACHE = os.path.join(tempfile.gettempdir(), f'annlite_b200_bench_{os.getuid()}')
DUMP_LIMIT = 64 << 20   # bytes --dump-outputs may write


def filtered_leg(timeout_s=240):
    """configs[3] (1M cosine, random 50 % filter, ef=64, k=10, 10 000-query batches) as an UNTIMED side measurement
    after the headline legs: `scripts/bench_configs.py c4` in a child process, so that nothing there can take the
    headline line with it.  Reports the filtered walk's kernel time, the streamed (annb_search_submit_filtered, pinned
    buffers, two batches in flight) and blocking end-to-end rates, and parity against the oracle's filtered search on
    a 2 000-query sample of the same graph."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', 'bench_configs.py'), 'c4'], cwd=ROOT,
                           env=dict(os.environ, C4_SKIP_REF='1'), capture_output=True, text=True, timeout=timeout_s)
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])
        keep = ('config', 'filtered_kernel', 'gpu_filtered_kernel_ms', 'gpu_filtered_qps_streamed_host_buffers',
                'streamed_ms_per_batch', 'streamed_rows_equal_blocking_call', 'gpu_filtered_qps_host_buffers',
                'flagged_walk_fallback_queries', 'round1_flagged_walk', 'unfiltered_kernel_ms', 'hops_per_query',
                'unfiltered_hops_per_query', 'all_results_pass_filter', 'parity_sample', 'rows_exact', 'rows_tie', 'rows_diff',
                'recall_vs_oracle_ids', 'max_rel_dist_err_equal_ids')
        out = {k_: d.get(k_) for k_ in keep}
        out['note'] = ('untimed side measurement in a child process; cosine => the device l2_normalize makes distance BITS '
                       'differ on part of the rows (rows_diff) at <= 1e-6 relative, ids are the oracle\'s (recall_vs_oracle_ids)')
        return out
    except Exception as ex:   # never at the expense of the headline line
        return {'unavailable': repr(ex)[:300]}


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--n', '--base-n', dest='n', type=int, default=1_000_000)   # use --base-n under torchrun (its parser treats --n as ambiguous)
    ap.add_argument('--dim', type=int, default=128)
    ap.add_argument('--m', type=int, default=8)
    ap.add_argument('--ks', type=int, default=256)
    ap.add_argument('--batch', type=int, default=10_000)
    ap.add_argument('--ef', type=int, default=64)
    ap.add_argument('--k', type=int, default=10)
    ap.add_argument('--M', type=int, default=16, help='HNSW max_connection')
    ap.add_argument('--efc', type=int, default=200)
    ap.add_argument('--dist', default='gaussian', choices=['gaussian', 'blobs'])
    ap.add_argument('--metric', default='euclidean')
    ap.add_argument('--mode', default='replicate', choices=['replicate', 'shard'])
    ap.add_argument('--build-threads', type=int, default=0)
    ap.add_argument('--no-cache', action='store_true')
    ap.add_argument('--cpu-sample', type=int, default=20000)
    ap.add_argument('--ref-sample', type=int, default=10000)
    ap.add_argument('--chunks', type=int, default=0, help='host-buffer pipeline depth inside annb_search (0 = auto)')
    ap.add_argument('--pool', type=int, default=4, help='distinct query batches cycled through the steps')
    ap.add_argument('--no-filtered-leg', action='store_true',
                    help='skip the configs[3] side measurement (filtered search, child process, ~20 s, untimed)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last headline step returned (rank 0) to DIR as .npy: '
                         'labels.npy (float64, -1 = no result), distances.npy (float32) and rows.npy (the query rows '
                         'written: all of them, or a fixed seeded sample when the batch exceeds 64 MB).  Queries, base '
                         'vectors and codebook are the same on every run, and the index is built sequentially '
                         '(--build-threads 1, several minutes at 1M rows) unless --build-threads says otherwise')
    a = ap.parse_args(argv)
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.build_threads == 0:
        # the concurrent builders make a different graph on every build, and two graphs share few result rows
        a.build_threads = 1
    return a


# ---------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md section 8d, C2: seed 2)
# ---------------------------------------------------------------------------------------------------
def make_base(a, lo=0, hi=None):
    hi = a.n if hi is None else hi
    if a.dist == 'gaussian':
        # chunked so any [lo, hi) slice is reproducible without generating the whole matrix
        out = np.empty((hi - lo, a.dim), dtype=np.float32)
        CH = 100_000
        for c in range(lo // CH, (hi + CH - 1) // CH):
            rng = np.random.default_rng([2, c])
            blk = rng.standard_normal((CH, a.dim), dtype=np.float32)
            s, e = max(lo, c * CH), min(hi, (c + 1) * CH)
            out[s - lo:e - lo] = blk[s - c * CH:e - c * CH]
        return out
    rng = np.random.default_rng(123)   # examples/pq_benchmark.py:25-28 shape: 3 gaussian blobs
    centers = rng.uniform(-10, 10, (3, a.dim)).astype(np.float32)
    rng = np.random.default_rng([2, 77])
    lab = rng.integers(0, 3, a.n)
    x = centers[lab] + rng.standard_normal((a.n, a.dim), dtype=np.float32)
    return np.ascontiguousarray(x[lo:hi])


def make_queries(a, nb, rank=0):
    rng = np.random.default_rng([2, 1000 + rank])
    if a.dist == 'gaussian':
        return rng.standard_normal((nb, a.batch, a.dim), dtype=np.float32)
    crng = np.random.default_rng(123)
    centers = crng.uniform(-10, 10, (3, a.dim)).astype(np.float32)
    lab = rng.integers(0, 3, (nb, a.batch))
    return (centers[lab] + rng.standard_normal((nb, a.batch, a.dim), dtype=np.float32)).astype(np.float32)


def cfg_key(a, extra=''):
    s = f'{a.n}-{a.dim}-{a.m}-{a.ks}-{a.M}-{a.efc}-{a.dist}-{a.metric}-{extra}'
    return hashlib.md5(s.encode()).hexdigest()[:12]


def train_codebook(a, X10k):
    """PQ training is out of scope (an input to the path): sklearn KMeans like PQCodec.fit
    (pq.py:89-115) with the SURVEY 8d settings (random_state=0, n_init=1, max_iter=20)."""
    os.makedirs(CACHE, exist_ok=True)
    p = os.path.join(CACHE, f'codebook_{cfg_key(a)}.npy')
    if os.path.exists(p) and not a.no_cache:
        return np.load(p)
    from sklearn.cluster import KMeans
    from threadpoolctl import threadpool_limits
    ds = a.dim // a.m
    if a.metric == 'cosine':
        X10k = X10k / np.maximum(np.linalg.norm(X10k, axis=1, keepdims=True), 1e-12)
    cb = np.empty((a.m, a.ks, ds), dtype=np.float32)
    with threadpool_limits(1):   # KMeans sums in thread order: one thread gives the same codebook on every machine
        for m in range(a.m):
            km = KMeans(n_clusters=a.ks, max_iter=20, n_init=1, random_state=0).fit(X10k[:, m * ds:(m + 1) * ds])
            cb[m] = km.cluster_centers_
    np.save(p, cb)
    return cb


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu=0):
        self.gpu, self.rows, self.p = gpu, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}',
                                       '--format=csv,noheader,nounits', '-lms', '20'],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.p.kill)   # nvidia-smi -lms never exits on its own
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.p:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        time.sleep(0.15)
        self.p.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 8 and r[4 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


def ncu_traffic_bytes():
    """DRAM bytes per K3 launch from the committed ncu capture of this same command (profiles/)."""
    p = os.path.join(ROOT, 'profiles', 'r02_k3_walk4_fused_ncu.txt')
    try:
        tot = 0.0
        for line in open(p):
            f = line.split()
            if f and f[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                tot += float(f[1]) * {'Mbyte': 1e6, 'Gbyte': 1e9, 'Kbyte': 1e3, 'byte': 1}[f[2]]
        return tot or None
    except Exception:
        return None


def dump_outputs(out_dir, labels, dists):
    """labels (B,k) int64, dists (B,k) float32 -> out_dir/{labels,distances,rows}.npy, at most DUMP_LIMIT bytes."""
    os.makedirs(out_dir, exist_ok=True)
    B, k = labels.shape
    row_bytes = k * (8 + 4) + 8
    rows = np.arange(B)
    if B * row_bytes > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(B, (DUMP_LIMIT - 4096) // row_bytes, replace=False))   # 4 KB: .npy headers
    np.save(os.path.join(out_dir, 'labels.npy'), labels[rows].astype(np.float64))
    np.save(os.path.join(out_dir, 'distances.npy'), dists[rows].astype(np.float32))
    np.save(os.path.join(out_dir, 'rows.npy'), rows.astype(np.float64))


def recall_at_k(pred, truth):
    return float(np.mean([len(set(p.tolist()) & set(t.tolist())) / len(t) for p, t in zip(pred, truth)]))


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def _timed(torch, dist, e, world, fn, steps, warmup, drain=None):
    """W warm-up steps, then exactly `steps` steps between barrier + synchronize on both sides; CUDA events on
    the Engine's stream, max over ranks.  Streamed legs finish on two internal streams: their step time is the
    larger of the event span on lane 0 and the host span that encloses the final synchronisation of both."""
    stream = torch.cuda.ExternalStream(e.stream)
    for i in range(warmup):
        fn(i)
    if drain:
        drain()
    e.sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = e.launch_count
    t0 = time.perf_counter()
    ev0.record(stream)
    for i in range(steps):
        fn(warmup + i)
    if drain:
        drain()
    e.sync()
    ev1.record(stream)
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(ev0.elapsed_time(ev1), 0.0)
    ms = max(ms, wall_ms) if drain else ms
    launches = e.launch_count - l0
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, launches


def _build_or_load(a, e, lo, hi, path, threads):
    """Index over base rows [lo, hi) (labels = global ids): from the cache file, else built and saved."""
    if os.path.exists(path) and not a.no_cache:
        e.load_index(path)
        return 0.0
    X = make_base(a, lo, hi)
    e.init_graph(hi - lo, M=a.M, ef_construction=a.efc)
    t0 = time.time()
    e.add_items(X, np.arange(lo, hi, dtype=np.uint64), num_threads=threads)
    t_build = time.time() - t0
    e.save_index(path + f'.tmp{os.getpid()}')
    os.replace(path + f'.tmp{os.getpid()}', path)
    return t_build


def shard_leg(a, cb, rank, world, local, ncores, torch, dist):
    """The range-sharded step: every rank walks ITS graph over base rows [r*N/G, (r+1)*N/G) for ALL queries, one
    all-gather of the packed (B,k) {fp32, u64} results over NCCL, merge kernel -- enqueued on one stream of the
    Engine with no host synchronisation, two batches in flight (annlite_b200.sharded.ShardedEngine)."""
    from annlite_b200.engine import Engine
    from annlite_b200.sharded import ShardedEngine
    es = Engine(a.dim, a.m, a.ks, a.metric, device=local)
    es.set_codebook(cb)
    lo, hi = rank * a.n // world, (rank + 1) * a.n // world
    path = os.path.join(CACHE, f'ours_{cfg_key(a, f"shard{rank}of{world}")}.hnsw')
    t_build = _build_or_load(a, es, lo, hi, path, a.build_threads or min(32, max(1, ncores // world)))
    B, k = a.batch, a.k
    nb = max(1, min(a.pool, a.steps + a.warmup))
    Qh = make_queries(a, nb, rank=0)                                 # the same queries on every rank
    Qd = torch.from_numpy(Qh).cuda()
    Qp = torch.from_numpy(Qh).pin_memory().numpy()
    hl = [torch.empty((B, k), dtype=torch.int64).pin_memory() for _ in range(2)]
    hd = [torch.empty((B, k), dtype=torch.float32).pin_memory() for _ in range(2)]
    norm = 2 if a.metric == 'cosine' else 0
    se = ShardedEngine(es, B, k)
    pend = []

    def drain():
        while pend:
            se.wait(pend.pop(0))

    def step_dev(i):
        if len(pend) == 2:
            se.wait(pend.pop(0))
        pend.append(se.submit(Qd[i % nb], a.ef, normalize=norm))

    def step_e2e(i):
        if len(pend) == 2:
            se.wait(pend.pop(0))
        pend.append(se.submit(Qp[i % nb], a.ef, normalize=norm, host_labels=hl[i & 1], host_dists=hd[i & 1]))

    ms, launches = _timed(torch, dist, es, world, step_dev, a.steps, a.warmup, drain)
    ms_e2e, _ = _timed(torch, dist, es, world, step_e2e, a.steps, max(3, a.warmup // 2), drain)
    # the walk alone (blocking call, CUDA events around the kernel): what the gather + merge add on top
    ol = torch.empty((B, k), dtype=torch.int64, device='cuda')
    od = torch.empty((B, k), dtype=torch.float32, device='cuda')
    walk_ms = 0.0
    for i in range(5):
        es.search(queries=Qd[i % nb], k=k, ef=a.ef, normalize=norm, out_labels=ol, out_dists=od)
        walk_ms += es.last_kernel_ms()['search_ms'] / 5
    t = torch.tensor([walk_ms], device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    walk_ms = float(t.item())
    total_q = B * a.steps
    res = {'value': round(total_q / (ms / 1e3), 1), 'unit': 'queries/s', 'ms_per_step': round(ms / a.steps, 4),
           'scaling': 'strong', 'parallelism': f'shard{world}', 'nodes_per_shard': hi - lo,
           'e2e': {'value': round(total_q / (ms_e2e / 1e3), 1), 'unit': 'queries/s', 'ms_per_step': round(ms_e2e / a.steps, 4),
                   'h2d_bytes_per_step': B * a.dim * 4, 'd2h_bytes_per_step': B * k * 12},
           'walk_ms_per_step_max_over_ranks': round(walk_ms, 4),
           'gather_merge_overhead_ms': round(ms / a.steps - walk_ms, 4),
           'collective': f'1 all_gather_into_tensor of {se.stride} bytes/rank/step on the Engine stream, then merge_sorted_kernel',
           'gpu_launches': int(launches), 'shard_build_s': round(t_build, 1),
           'note': 'every shard walks every query: QPS ~ one GPU on an N/G-node graph; sharding is for capacity (configs[2], [4])'}
    return res, es, Qh


def run_ours(a):
    import torch
    import torch.distributed as dist
    from annlite_b200.engine import Engine

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    ncores = os.cpu_count() or 1
    shard_main = a.mode == 'shard' and world > 1
    if shard_main and a.dump_outputs:
        raise SystemExit('--dump-outputs writes the replicated step; run it without --mode shard')

    # ---- index: replicated on every rank (rank 0 builds, the others load the file) -----------------
    cb = train_codebook(a, make_base(a, 0, 10_000)) if rank == 0 else None
    if world > 1:
        obj = [cb]
        dist.broadcast_object_list(obj, src=0)
        cb = obj[0]
    os.makedirs(CACHE, exist_ok=True)
    e = Engine(a.dim, a.m, a.ks, a.metric, device=local)
    e.set_codebook(cb)
    if a.chunks:
        e.set_option('chunks', a.chunks)
    t_build = 0.0
    path = os.path.join(CACHE, f'ours_{cfg_key(a, "sequential" if a.build_threads == 1 else "")}.hnsw')
    if rank == 0:
        t_build = _build_or_load(a, e, 0, a.n, path, a.build_threads)   # 0 threads = library default (<= 32, quota-aware)
    if world > 1:
        dist.barrier()
    if e.element_count == 0:
        e.load_index(path)

    # ---- queries --------------------------------------------------------------------------------
    nb = max(1, min(a.pool, a.steps + a.warmup))
    Qh = make_queries(a, nb, rank=rank)
    Qd = torch.from_numpy(Qh).cuda()
    B, k = a.batch, a.k
    out_l = torch.empty((B, k), dtype=torch.int64, device='cuda')
    out_d = torch.empty((B, k), dtype=torch.float32, device='cuda')
    norm = 2 if a.metric == 'cosine' else 0
    Qp = torch.from_numpy(Qh).pin_memory()
    hl = torch.empty((B, k), dtype=torch.int64).pin_memory()
    hd = torch.empty((B, k), dtype=torch.float32).pin_memory()
    Qp_np, hl_np, hd_np = Qp.numpy(), hl.numpy().view(np.uint64), hd.numpy()

    def step_dev(i):
        e.search(queries=Qd[i % nb], k=k, ef=a.ef, normalize=norm, out_labels=out_l, out_dists=out_d)

    def step_e2e(i):
        e.search(queries=Qp_np[i % nb], k=k, ef=a.ef, normalize=norm, out_labels=hl_np, out_dists=hd_np)

    # streamed (submit / wait, two batches in flight): the serving-loop shape
    out_l2 = [torch.empty((B, k), dtype=torch.int64, device='cuda') for _ in range(2)]
    out_d2 = [torch.empty((B, k), dtype=torch.float32, device='cuda') for _ in range(2)]
    hl2 = [torch.empty((B, k), dtype=torch.int64).pin_memory() for _ in range(2)]
    hd2 = [torch.empty((B, k), dtype=torch.float32).pin_memory() for _ in range(2)]
    hl2_np = [t.numpy().view(np.uint64) for t in hl2]
    hd2_np = [t.numpy() for t in hd2]
    pending = []

    def drain():
        while pending:
            e.search_wait(pending.pop(0))

    def step_dev_stream(i):
        if len(pending) == 2:
            e.search_wait(pending.pop(0))
        pending.append(e.search_submit(Qd[i % nb], out_l2[i & 1], out_d2[i & 1], k=k, ef=a.ef, normalize=norm))

    def step_e2e_stream(i):
        if len(pending) == 2:
            e.search_wait(pending.pop(0))
        pending.append(e.search_submit(Qp_np[i % nb], hl2_np[i & 1], hd2_np[i & 1], k=k, ef=a.ef, normalize=norm))

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.05)
    ms, launches = _timed(torch, dist, e, world, step_dev_stream, a.steps, a.warmup, drain)
    last = (a.warmup + a.steps - 1) & 1                                      # step i wrote out_l2[i & 1]
    last_step = (out_l2[last].cpu().numpy(), out_d2[last].cpu().numpy()) if a.dump_outputs else None
    ms_e2e, _ = _timed(torch, dist, e, world, step_e2e_stream, a.steps, max(3, a.warmup // 2), drain)
    ms_sync, _ = _timed(torch, dist, e, world, step_dev, a.steps, 3)            # one blocking call per step, for reference
    ms_e2e_sync, _ = _timed(torch, dist, e, world, step_e2e, a.steps, 3)
    # the same blocking call with ordinary (pageable) numpy buffers: what a caller pays without pinning anything
    pg_l = np.empty((B, k), dtype=np.uint64)
    pg_d = np.empty((B, k), dtype=np.float32)

    def step_e2e_pageable(i):
        e.search(queries=Qh[i % nb], k=k, ef=a.ef, normalize=norm, out_labels=pg_l, out_dists=pg_d)

    n_pg = max(1, min(a.steps, 50))
    ms_e2e_pg, _ = _timed(torch, dist, e, world, step_e2e_pageable, n_pg, 3)
    shard_res = None
    if world > 1:
        shard_res, es, Qh_sh = shard_leg(a, cb, rank, world, local, ncores, torch, dist)
    ck = clocks.stop() if rank == 0 else None   # sampled across all timed regions
    # walk kernel duration per launch: CUDA events around the kernel on its own stream, blocking calls, untimed here
    kern_ms = 0.0
    for i in range(5):
        step_dev(i)
        kern_ms += e.last_kernel_ms()['search_ms'] / 5

    total_q = B * a.steps * world
    value = total_q / (ms / 1e3)
    e2e = total_q / (ms_e2e / 1e3)

    # ---- untimed: work counters (roofline), recall, CPU baseline + parity --------------------------
    result = None
    if rank == 0:
        labels, dists, stats = e.search(queries=Qh[0], k=k, ef=a.ef, normalize=norm, with_stats=True)
        hops, nbrs = stats[:, 0].astype(np.float64), stats[:, 1].astype(np.float64)
        code_row = a.m * (1 if a.ks <= 256 else 2)
        M0 = 2 * a.M
        # SURVEY.md 8d, K3: hops*(4+4*M0) + evals*(M*code_bytes) + evals/8 + k*12 per query ("evals" = neighbours
        # listed, metric_distance_computations); K1 is fused (table in shared memory: 0 bytes) and adds only the
        # query read D*4.  hops and neighbours are counted by the kernel.
        alg_bytes_q = hops * (4 + 4 * M0) + nbrs * code_row + nbrs / 8 + k * 12 + a.dim * 4
        alg_bytes_launch = float(alg_bytes_q.sum())
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        achieved = alg_bytes_launch / (kern_ms / 1e3) / 1e9
        traffic = ncu_traffic_bytes() if (a.n == 1_000_000 and a.batch == 10_000) else None
        roof = {'bound': 'hbm', 'kernel': 'hnsw_walk4 (ADC table build fused into the walk)', 'achieved': round(achieved, 2),
                'peak': peak, 'peak_source': 'MEASURED_PEAKS.json' if 'hbm_gbs' in peaks else 'fallback 6.65 TB/s',
                'unit': 'GB/s', 'frac': round(achieved / peak, 5), 'traffic': traffic,
                'traffic_source': 'committed profile profiles/r02_k3_walk4_fused_ncu.txt (ncu --set full of this workload): '
                                  'dram__bytes_read.sum + dram__bytes_write.sum per launch; not re-measured in this run',
                'alg_bytes_per_launch': round(alg_bytes_launch),
                'ms_per_launch': round(kern_ms, 4), 'alg_bytes_per_query': round(float(alg_bytes_q.mean()), 1),
                'hops_per_query': round(float(hops.mean()), 2), 'nbrs_per_query': round(float(nbrs.mean()), 1),
                'note': 'dependent pointer chase: latency-bound, not bandwidth-bound; moved bytes/query = hops*record(384B)'}
        # recall vs exhaustive ADC on the same codes (GPU K2) and vs true L2 on a sample
        sample = min(1000, B)
        g = e.get_graph()
        n = g['cur_element_count']
        codes = g['data_level0'].reshape(n, -1)[:, g['offset_data']:g['label_offset']].copy()
        lab = np.ascontiguousarray(g['data_level0'].reshape(n, -1)[:, g['label_offset']:g['label_offset'] + 8]).view(np.uint64).ravel()
        e.set_codes(codes.view(np.uint8 if a.ks <= 256 else np.uint16).reshape(n, a.m))
        rec_adc = None
        k2 = None
        if a.metric == 'euclidean':
            tbl = e.adc_table(Qh[0][:sample])
            gt_i, _ = e.scan_topk(tables=tbl, k=k)
            rec_adc = recall_at_k(labels[:sample], lab[gt_i])
            # K2 (exhaustive ADC + top-k, the recall ground truth above) against ITS roofline: one shared-memory
            # lookup per (query, row, subquantiser); an SM serves 32 four-byte lookups per clock
            e.scan_topk(tables=tbl, k=k)
            k2_ms = e.last_kernel_ms()['scan_ms']
            e.set_option('scan_kernel', 1)       # round 1's kernel (lanes = rows, one table per warp) for the before/after
            gt_old, _ = e.scan_topk(tables=tbl, k=k)
            e.scan_topk(tables=tbl, k=k)
            k2_ms_old = e.last_kernel_ms()['scan_ms']
            e.set_option('scan_kernel', 0)
            if k2_ms and k2_ms > 0:
                peak_lk = 148 * 32 * (ck['sm_mhz'] or 1965.0) * 1e6 if isinstance(ck, dict) else 148 * 32 * 1.965e9
                lk = float(sample) * n * a.m
                k2 = {'kernel': 'scan_topk_tiled2_kernel (16-query interleaved table tile, lanes = queries) + merge_topk_kernel',
                      'round1_kernel_ms': round(k2_ms_old, 3), 'ids_equal_round1_kernel': bool(np.array_equal(gt_i, gt_old)),
                      'queries': int(sample), 'rows': int(n),
                      'ms': round(k2_ms, 3), 'qps': round(sample / (k2_ms / 1e3), 1), 'bound': 'shared-memory gather',
                      'lookups_per_s': round(lk / (k2_ms / 1e3), 1), 'peak_lookups_per_s': peak_lk,
                      'frac': round(lk / (k2_ms / 1e3) / peak_lk, 4), 'hbm_bytes_algorithmic': int(n * a.m * ((sample + 7) // 8)),
                      'note': 'untimed side measurement (not part of value / e2e)'}
        Xd = torch.from_numpy(make_base(a)).cuda()
        qd = Qd[0][:sample]
        d2 = (qd * qd).sum(1, keepdim=True) - 2 * qd @ Xd.T + (Xd * Xd).sum(1)[None]
        gt = d2.topk(k, dim=1, largest=False).indices.cpu().numpy()
        rec_l2 = recall_at_k(labels[:sample].astype(np.int64), gt)
        del Xd, d2
        # CPU baseline: C oracle port over the same graph, all host threads, bounded sample; its answers double as
        # the parity check of this very run (same graph, same queries)
        cpu, parity = (None, None)
        if world == 1:   # reported at N=1 only
            cpu, parity = cpu_port_baseline(a, e, Qh, cb, ncores, labels, dists, lab, gt_i if rec_adc is not None else None)
        result = {
            'metric': 'queries/sec (PQ-HNSW search, 1M x 128d, M=8, ef=64, k=10)', 'value': round(value, 1),
            'unit': 'queries/s', 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': round(ms / a.steps, 4), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'configs[1]: {a.n}x{a.dim} fp32 {a.dist}, PQ M={a.m} Ks={a.ks}, HNSW M={a.M} '
                                   f'efc={a.efc}, ef={a.ef}, k={a.k}, batch={a.batch} queries/step/GPU',
                       'parallelism': 'replicate' + str(world),
                       'l2_policy': 'index (384 MB walk records) exceeds the 126 MB L2; query batches rotate '
                                    f'through a pool of {nb}',
                       'metric_space': a.metric, 'index_build_s': round(t_build, 1), 'host_cores': ncores,
                       'api': 'streamed: annb_search_submit/wait with two batches in flight (value and e2e); '
                              'blocking_call_value = one annb_search call at a time'},
            'e2e': {'value': round(e2e, 1), 'unit': 'queries/s', 'h2d_bytes_per_step': B * a.dim * 4,
                    'd2h_bytes_per_step': B * k * 12 + B * 4, 'ms_per_step': round(ms_e2e / a.steps, 4),
                    'api': 'annb_search_submit/wait, 2 batches in flight, pinned host buffers',
                    'blocking_call_value': round(total_q / (ms_e2e_sync / 1e3), 1),
                    'blocking_call_pageable_buffers_value': round(B * n_pg * world / (ms_e2e_pg / 1e3), 1)},
            'blocking_call_value': round(total_q / (ms_sync / 1e3), 1),
            'gpu_launches': int(launches), 'clocks': ck, 'roofline': roof, 'cpu_baseline': cpu,
            'recall_at_k': {'vs_exhaustive_adc': rec_adc, 'vs_true_l2': rec_l2, 'sample': sample},
            'parity': parity, 'k2_exhaustive_scan': k2,
        }
        if shard_res is not None:
            result['shard'] = shard_res
            if shard_main:   # --mode shard: the sharded step is the headline of this line
                for key in ('value', 'ms_per_step', 'scaling', 'gpu_launches'):
                    result['replicate_' + key] = result[key]
                    result[key] = shard_res[key]
                result['e2e'] = dict(result['e2e'], **shard_res['e2e'], api='ShardedEngine: submit + all-gather + merge, 2 batches in flight')
                result['config']['parallelism'] = f'shard{world}'
        if world == 1 and a.steps >= 20 and not a.no_filtered_leg and a.n == 1_000_000 and a.metric == 'euclidean':
            result['filtered_configs3'] = filtered_leg()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if last_step is not None:
            dump_outputs(a.dump_outputs, *last_step)
        print(json.dumps(result))


def cpu_port_baseline(a, e, Qh, cb, ncores, gpu_labels, gpu_dists, lab_by_id, gt_adc):
    """oracle port (C restatement, oracle/pq_oracle.c) on the host cores: tables + walk, threads over
    query slices (ctypes releases the GIL).  Bounded sample of the same query batches.  Its answers for batch 0
    are compared row by row with what the GPU returned for the same queries on the same graph: `parity`."""
    import oracle as O
    g = O.Graph.from_state(e.get_graph(), a.m, a.ks)
    S = min(a.cpu_sample, Qh.shape[0] * Qh.shape[1])
    q = Qh.reshape(-1, a.dim)[:S]
    T = min(ncores, 64)
    parts = [p for p in np.array_split(np.arange(S), T) if len(p)]
    out = [None] * len(parts)

    def work(j, idx):
        t = O.adc_table(q[idx], cb, a.metric)
        out[j] = O.hnsw_search(g, t, a.k, a.ef)

    O.hnsw_search(g, O.adc_table(q[:64], cb, a.metric), a.k, a.ef)  # warm
    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(j, p)) for j, p in enumerate(parts)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    cpu = {'value': round(S / dt, 1), 'unit': 'queries/s', 'cores': T, 'kind': 'port',
           'sample': f'{S} queries of the same batches (tables + walk), {T} threads, {dt:.2f}s'}
    ol = np.concatenate([o[0] for o in out])
    od = np.concatenate([o[1] for o in out])
    R = min(S, gpu_labels.shape[0])
    parity = None
    if a.metric != 'cosine':   # cosine: device l2_normalize is tolerance-level, rows are compared in the tests
        gl, gd = gpu_labels[:R], gpu_dists[:R]
        same_d = (gd.view(np.uint32) == od[:R].view(np.uint32)).all(axis=1)
        same_l = (gl == ol[:R]).all(axis=1)
        exact = int((same_d & same_l).sum())
        tie = int((same_d & ~same_l).sum())   # equal distance bits, labels permuted/chosen among exact fp32 ties
        parity = {'rows': int(R), 'exact': exact, 'tie': tie, 'diff': int(R - exact - tie),
                  'checker': 'C oracle (searchKnn restatement) on the same graph and queries',
                  'recall_gpu_vs_oracle_ids': recall_at_k(gl, ol[:R])}
        if gt_adc is not None:
            sm = min(R, gt_adc.shape[0])
            parity['recall_at_k_gpu'] = recall_at_k(gl[:sm], lab_by_id[gt_adc[:sm]])
            parity['recall_at_k_oracle'] = recall_at_k(ol[:sm], lab_by_id[gt_adc[:sm]])
    return cpu, parity


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU path (oracle/_ref), all host threads
# ---------------------------------------------------------------------------------------------------
def run_reference(a):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    from oracle import ref_driver as R
    if not R.available():
        print(json.dumps({'impl': 'reference', 'unavailable': 'oracle/_ref not built (needs /root/reference at build time)'}))
        return
    ncores = os.cpu_count() or 1
    world = int(os.environ.get('WORLD_SIZE', 1))
    cb = train_codebook(a, make_base(a, 0, 10_000))
    codec = R.RefCodec(cb, a.metric)
    X = make_base(a)
    idx = R.RefHnswIndex(codec, a.metric, capacity=a.n, ef_construction=a.efc, ef_search=a.ef, max_connection=a.M)
    t0 = time.time()
    idx.add_with_ids(X, np.arange(a.n), num_threads=ncores, batch=5000)
    t_build = time.time() - t0
    nb = max(1, min(a.pool, a.steps + a.warmup))
    Qh = make_queries(a, nb, rank=0)
    # bounded sample per step so that the whole --steps/--warmup run stays within a couple of minutes
    S = min(a.ref_sample, a.batch, max(256, 1_500_000 // max(1, a.steps + a.warmup)))

    def step(i):
        q = Qh[i % nb][:S]
        tables = codec.get_dist_mat(idx._pre(q))           # pq_bind (single-threaded Cython)
        return idx.knn_query(q, a.k, num_threads=ncores, tables=tables)   # hnsw_bind, all threads

    for i in range(a.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(a.steps):
        labels, dists = step(a.warmup + i)
    dt = time.perf_counter() - t0
    qps = S * a.steps / dt
    # walk-only rate (tables prebuilt) for context
    q = Qh[0][:S]
    tables = codec.get_dist_mat(idx._pre(q))
    t1 = time.perf_counter()
    idx.knn_query(q, a.k, num_threads=ncores, tables=tables)
    walk_qps = S / (time.perf_counter() - t1)
    # as-shipped semantics: one query per call (AnnLite.search loop), bounded
    t2 = time.perf_counter()
    for j in range(300):
        idx.search(Qh[0][j], limit=a.k)
    loop_qps = 300 / (time.perf_counter() - t2)
    # recall@k of what the reference returned: against the exhaustive ADC scan over its own codes (oracle scan, sample)
    import oracle as O
    stt = idx.state()
    n_el = int(stt['cur_element_count'])
    rec = np.asarray(stt['data_level0']).view(np.uint8).reshape(-1, int(stt['size_data_per_element']))[:n_el]
    codes = np.ascontiguousarray(rec[:, int(stt['offset_data']):int(stt['label_offset'])]).view(np.uint8 if a.ks <= 256 else np.uint16)
    lab = np.ascontiguousarray(rec[:, int(stt['label_offset']):int(stt['label_offset']) + 8]).view(np.uint64).ravel()
    rs = min(200, S)
    gt_i, _ = O.scan_topk(tables[:rs], codes.reshape(n_el, a.m), a.k)
    ref_l, _ = idx.knn_query(q[:rs], a.k, num_threads=ncores, tables=tables[:rs])
    rec_adc = recall_at_k(np.asarray(ref_l), lab[gt_i])
    res = {
        'impl': 'reference', 'metric': 'queries/sec (PQ-HNSW search, 1M x 128d, M=8, ef=64, k=10)',
        'value': round(qps, 1), 'unit': 'queries/s', 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
        'ms_per_step': round(dt / a.steps * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'configs[1]: {a.n}x{a.dim} fp32 {a.dist}, PQ M={a.m} Ks={a.ks}, HNSW M={a.M} '
                               f'efc={a.efc}, ef={a.ef}, k={a.k}; each step = {S} queries (bounded sample of the '
                               f'{a.batch}-query batch)', 'index_build_s': round(t_build, 1), 'host_cores': ncores,
                   'walk_only_qps': round(walk_qps, 1), 'one_query_per_call_qps': round(loop_qps, 1)},
        'cpu_baseline': {'value': round(qps, 1), 'unit': 'queries/s', 'cores': ncores, 'kind': 'reference',
                         'sample': f'{S} queries/step: pq_bind.batch_precompute_adc_table (1 thread) + '
                                   f'hnsw_bind.Index.knn_query ({ncores} threads)'},
        'e2e': {'value': round(qps, 1), 'unit': 'queries/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'recall_at_k': {'vs_exhaustive_adc': rec_adc, 'sample': rs},
    }
    print(json.dumps(res))


if __name__ == '__main__':
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
