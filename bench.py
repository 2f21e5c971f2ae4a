#!/usr/bin/env python
"""bench.py -- the reference's headline metric on its headline config, measured on B200.

metric   : SPD pair dist+grad evals/sec (BASELINE.json), unit "pairs/s"
workload : BASELINE config 5 -- synthetic 2M-node scale-free graph, SPD 4x4 affine-invariant embedding (fp32),
           2^24 sampled pairs per step built as 1024 BFS sources x 16384 random targets, hop-count targets from the
           multi-source BFS kernel, distortion loss (QuotientLoss, both terms), RiemannianAdam(lr .01, clip 100,
           exact) -- graphembed/experiments/run_grid.py:24-36,108-138 hyper-parameters.
step     : zero grad -> ONE fused pair kernel (gather + distance + loss + gradient + scatter-add) over the batch
           -> ONE fused optimizer kernel over all 2M points.  N>1: pairs sharded over ranks, and the optimizer
           kernel is the peer-memory owner update (pull+sum the owned gradient rows of every rank over NVLink, update,
           push the new rows to every rank) -- NCCL reduce-scatter / all-gather only if CUDA IPC is unavailable.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--pairs-log2 24] [--nodes 2000000]
                  [--dump-outputs DIR]

`value`  : whole-job pairs/s with the pair batches resident in HBM (CUDA events, max over ranks).
`e2e`    : same metric through the public API from PINNED HOST buffers.  Sampled path: the step's input is its 1024
           BFS source ids (4 KB upload); the 16384 targets per source are DRAWN INSIDE the
           pair kernel (counter hash of (seed, pair number), GM_PAIRS_SAMPLED) and their hop counts read from the BFS
           level matrix of those sources, which stays resident in HBM (the landmark set is fixed, BFS once); the loss is
           read back every step (PairTrainer.step_sampled_host).  The other path, PairTrainer.step_host_grouped, uploads
           the step's explicit source-grouped (sources, offsets, j | hops << 24) pair list, 4 bytes per pair, overlapped
           with the previous step.  Measured on B200: lists 1.31 ms/step at 1 GPU but host-memory bound beyond 2 GPUs of
           one host (3.05 ms at 8); sampled +0.33 ms per step at any GPU count (one random byte per pair costs a DRAM
           line).  --e2e auto (default) takes lists up to 2 GPUs and sampled beyond; --e2e lists|sampled forces one.
`secondary`: (N=1) epoch time of BASELINE configs 1-4 through TrainingEngine on the shipped graphs, each with its
           roofline and the CPU reference beside it, and the multi-source BFS kernel with a fresh BFS every step.
`roofline`: fused pair kernel, algorithmic bytes (268 B/pair, SURVEY 8d) / its CUDA-event duration vs the
           measured HBM copy bandwidth in MEASURED_PEAKS.json.
`cpu_baseline`: the oracle port (same torch/LAPACK calls as the reference) on the host cores, bounded sample.
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
sys.path.insert(0, os.path.join(ROOT, 'matrix-manifolds_b200'))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'spd4_pair_dist_grad_evals_per_sec'
UNIT = 'pairs/s'
BYTES_PER_PAIR = 4 * 16 * 4 + 4 + 8  # SURVEY 8(d): 2 endpoint reads + 2 gradient accumulations + target + 2 indices
N_SOURCES = 1024
DUMP_ROWS = 1 << 18  # --dump-outputs: 16 MB of the 128 MB point table


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--pairs-log2', type=int, default=24)
    ap.add_argument('--nodes', type=int, default=2_000_000)
    ap.add_argument('--batches', type=int, default=3, help='distinct pre-generated pair batches cycled through')
    ap.add_argument('--cpu-pairs-log2', type=int, default=17)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-peer', action='store_true', help='N>1: NCCL reduce-scatter / all-gather owner update instead '
                    'of the fused peer-memory kernel (A/B)')
    ap.add_argument('--unpacked', action='store_true', help='separate uint8 hop-count vector instead of the packed '
                    '(j | hops << 24) pair format')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'], help='weak: 2^pairs_log2 pairs per GPU per '
                    'step; strong: 2^pairs_log2 pairs per step in total, split over the GPUs (BASELINE config 5 as '
                    'written)')
    ap.add_argument('--e2e', default='auto', choices=['auto', 'lists', 'sampled'], help='end-to-end leg: `lists` uploads '
                    'explicit pair lists (4 B/pair, PCIe / host-memory bound beyond 2 GPUs of one host), `sampled` uploads '
                    'the source ids and draws the pairs inside the pair kernel (one extra random byte read per pair); '
                    'auto = lists up to 2 GPUs, sampled beyond')
    ap.add_argument('--lists3', action='store_true', help='--e2e lists: upload 3-byte pair words (pack_hops3) instead of '
                    '4-byte ones; measured on one B200 it is NOT faster (1.339 vs 1.31 ms per step: the step is not PCIe '
                    'bound at 4 B/pair and the extra expansion kernel costs 0.03 ms)')
    ap.add_argument('--lists-format', default='auto', choices=['auto', '2', '4'], help='--e2e lists: bytes per pair on '
                    'the host->device link.  4: int32 j | hops << 24.  2 (= auto whenever the batch fits): the gap format '
                    '(pack_hops2: every group\'s targets sorted by row, 13-bit gap + 3 bits of hop count, expanded on the '
                    'device by gm_unpack_pairs2 together with the first-endpoint vector, 53 us per 2^24 pairs).  Measured '
                    'end to end on one GPU: 1.197 ms per step with 2-byte words (device bound), 1.285 ms with 4-byte '
                    'words (PCIe bound: 67 MB per step at 52 GB/s)')
    ap.add_argument('--layout', default='replicated', choices=['replicated', 'sharded'], help='N>1: `replicated` = every '
                    'rank holds the whole point table, partial gradients exchanged by the peer-memory owner update after '
                    'the pair kernel; `sharded` = ROW-SHARDED embeddings (engine.ShardedPairTrainer): every rank holds '
                    '1/N of the rows, the pair kernel gathers / reduces remote rows over NVLink, the optimizer is local')
    ap.add_argument('--windows', type=int, default=8, help='order every batch by (window of the target row, source) '
                    'and let the pair kernel walk the windows one after another (gm_pairs_t.segments): the rows it '
                    'gathers and reduces into stay L2 resident and the launch takes the specialised instantiation of '
                    'the kernel (0.957 vs 1.008 ms).  0: plain source-grouped batches')
    ap.add_argument('--no-secondary', action='store_true', help='skip the secondary lines (configs 1-4, BFS)')
    ap.add_argument('--workload', default='5', help="'5' (default, the bench line) or one of 1, 2a, 2b, 3a, 3b, 4 (or a "
                    "comma list / 'all'): epoch time of that BASELINE config -- on the GPU through TrainingEngine, or "
                    "with --impl reference on the host CPU")
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last device-resident timed step returned as '
                    'DIR/<name>.npy: loss.npy (float64, the step loss) and points.npy (float32, the updated SPD 4x4 '
                    f'points of a fixed, seeded sample of min(N, {DUMP_ROWS}) rows in ascending row order), so that '
                    'two builds run with the same arguments can be compared output for output.  The inputs are the '
                    'same on every run; the gradient is summed with atomics, so two runs agree to summation order, '
                    'not bit for bit')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


# ---------------------------------------------------------------------------------------------------------------------
# synthetic workload
# ---------------------------------------------------------------------------------------------------------------------
def scale_free_edges(n, m, seed):
    """Preferential-attachment graph (Barabasi-Albert style, m edges per new node), vectorised: every edge of node t
    either copies the target of a uniformly chosen earlier edge (degree-proportional choice) or picks a uniform earlier
    node; copy chains are resolved by pointer jumping.  Connected by construction (edge 0 of node t goes to t-1's
    component)."""
    rng = np.random.RandomState(seed)
    t = np.repeat(np.arange(1, n, dtype=np.int64), m)  # source node of every edge
    e = np.arange(t.size, dtype=np.int64)
    first_edge_of_t = (t - 1) * m
    uniform_target = (rng.random_sample(t.size) * t).astype(np.int64)
    copy = (rng.random_sample(t.size) < 0.5) & (first_edge_of_t > 0)
    parent = np.where(copy, (rng.random_sample(t.size) * np.maximum(first_edge_of_t, 1)).astype(np.int64), e)
    for _ in range(64):  # pointer jumping until every chain ends in a non-copy edge
        nxt = parent[parent]
        if np.array_equal(nxt, parent):
            break
        parent = nxt
    target = uniform_target[parent]
    return np.stack([t, target], axis=1)


def make_pair_batches(n_nodes, log2_pairs, n_batches, device, seed, n_src=None, keep_levels=False, graph=None,
                      windows=0):
    """[(I int32, J int32, hops uint8, sources int32, offsets int64, J|hops<<24 int32)] pinned host tensors + max
    hop^2; hop targets come from the multi-source BFS kernel.  (sources, offsets) is the source-grouped form of I, the
    last entry the packed 4-byte-per-pair form of (J, hops).  windows > 1: every batch is put into (window of the target
    row, source) order (graphembed.engine.window_order) -- the groups are then the (window, source) runs -- for a launch
    with gm_pairs_t.segments = windows."""
    from graphembed.data import bfs_levels, edges_to_csr
    from graphembed.engine import pack_hops, pack_hops2, pack_hops3, window_groups
    from graphembed import _lib as L
    P = 1 << log2_pairs
    per_src = max(1, P // N_SOURCES)
    if n_src is None:
        n_src = P // per_src
    if graph is None:
        edges = scale_free_edges(n_nodes, 4, 1234)  # ONE graph for every rank; the ranks differ in what they sample
        rowptr, colidx = edges_to_csr(n_nodes, edges)
        graph = (torch.as_tensor(rowptr, device=device), torch.as_tensor(colidx, device=device))
    rp, ci = graph
    gen = torch.Generator(device='cpu').manual_seed(seed)
    batches, max_h, kept = [], 0, []
    for b in range(n_batches):
        src = torch.randperm(n_nodes, generator=gen)[:n_src].int()
        levels = bfs_levels(rp, ci, sources=src.to(device), device=device, level_bytes=1)  # (n_src, N) uint8
        slot = torch.arange(n_src, dtype=torch.int32).repeat_interleave(per_src)
        I = src[slot.long()].contiguous()
        J = torch.randint(n_nodes - 1, (n_src * per_src,), generator=gen, dtype=torch.int32)
        J = torch.where(J >= I, J + 1, J).contiguous()  # uniform over nodes != i
        hops = torch.empty(n_src * per_src, dtype=torch.uint8, device=device)
        sd, jd = slot.to(device), J.to(device)
        rc = L.lib().gm_gather_levels(1, L.ptr(levels), n_nodes, L.ptr(sd), L.ptr(jd), hops.numel(), L.ptr(hops),
                                      L.stream_ptr(device))
        L.check(rc, 'gm_gather_levels')
        max_h = max(max_h, int(levels.max().item()))
        assert int(hops.min().item()) >= 1 and int(hops.max().item()) < 255
        offsets = (torch.arange(n_src + 1, dtype=torch.int64) * per_src)
        hops_h = hops.cpu()
        if windows > 1:
            order, src_groups, offsets = window_groups(src, offsets, J, n_nodes, windows)
            I, J, hops_h = I[order].contiguous(), J[order].contiguous(), hops_h[order].contiguous()
        else:
            src_groups = src
        three = n_nodes <= (1 << 21) and int(hops_h.max()) <= 8  # (j, hops - 1) fit 21 + 3 bits: 3 bytes per pair
        two = pack_hops2(offsets, J, hops_h)  # every group's targets sorted by row, 2-byte gap words (None: no fit)
        batches.append((I.pin_memory(), J.pin_memory(), hops_h.pin_memory(), src_groups.contiguous().pin_memory(),
                        offsets.pin_memory(), pack_hops(J, hops_h).pin_memory(),
                        pack_hops3(J, hops_h).pin_memory() if three else None,
                        None if two is None else (two[0].pin_memory(), two[1].pin_memory())))
        if keep_levels:
            kept.append(levels)  # (n_src, N) uint8, resident: the hop counts of this batch's landmark sources
        del levels
    if keep_levels:
        return batches, float(max_h * max_h), kept, per_src, graph
    return batches, float(max_h * max_h)


# ---------------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '20'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[k] for r in self.rows if len(r) >= 6 for k in range(4) if r[2 + k].startswith('Active')})
        return {'sm_mhz': int(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


class NvlinkCounter:
    """NVLink payload bytes of one GPU over a timed region, from the driver's own counters (NVML field
    NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX / _RX summed over the links, KiB): the measured traffic of the fused
    peer-memory owner update (ncu cannot replay a kernel that handshakes with other ranks)."""

    def __init__(self, index):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.fields = [pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX]
        except Exception:  # noqa: BLE001 -- counters are optional evidence
            self.h = None

    def _read(self):
        """[tx KiB, rx KiB] summed over the links (scope id = link number; a few drivers also take UINT_MAX = all)."""
        tot = [0, 0]
        got = False
        for link in range(18):
            try:
                vals = self.nv.nvmlDeviceGetFieldValues(self.h, [(f, link) for f in self.fields])
            except Exception:  # noqa: BLE001
                break
            for k, v in enumerate(vals):
                if getattr(v, 'nvmlReturn', 0) == 0:
                    tot[k] += int(v.value.ullVal)
                    got = True
        return tot if got else None

    def start(self):
        self.t0 = self._read() if self.h is not None else None

    def stop(self, steps):
        t1 = self._read() if self.h is not None else None
        if not self.t0 or not t1:
            return {'available': False}
        tx, rx = (t1[0] - self.t0[0]) * 1024, (t1[1] - self.t0[1]) * 1024
        return {'available': True, 'tx_bytes_per_step': tx / steps, 'rx_bytes_per_step': rx / steps,
                'source': 'NVML NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX/RX, summed over the links, across 5 extra steps'}


# ---------------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port): same step on a bounded sample of the workload
# ---------------------------------------------------------------------------------------------------------------------
def cpu_step_rate(log2_pairs, steps, warmup, seed=0, device='cpu'):
    """The reference's implementation of the step (oracle port: the same torch / LAPACK calls) on a bounded sample.
    device='cpu': the host cores (the reference arm).  device='cuda': the same torch-op path on the same B200 -- the
    "second comparator" of SURVEY 8(d): what the reference's own PyTorch code does when its tensors live on the GPU
    (run.py:33-35): every op on the device except the symmetric eigendecomposition, which the reference's wrapper
    round-trips through the host (linalg/torch_batch.py:94-135, cpu_offload=True by default) -- reproduced here as is.
    (Keeping eigh on the device is not an option on this stack anyway: torch 2.11's batched cuSOLVER syevBatched path
    rejects a 2^17 x 4 x 4 fp32 batch with CUSOLVER_STATUS_INVALID_VALUE.)"""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import manifolds_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = 1 << log2_pairs
    n = max(64, P // 8)  # same pairs-per-node ratio as the full workload (2^24 pairs / 2M nodes)
    gen = torch.Generator().manual_seed(seed)
    orc = O.SpdOracle(4)
    eigh_saved = O._eigh
    if device != 'cpu':  # tb.symeig's cpu_offload=True: eigh on the host, results back on the device (differentiable)
        O._eigh = lambda m: tuple(r.to(m.device) for r in torch.linalg.eigh(m.cpu(), UPLO='U'))
    x = orc.rand(n, ir=0.1, dtype=torch.float32, generator=gen).to(device)
    I = torch.randint(n, (P,), generator=gen).to(device)
    J = ((I.cpu() + 1 + torch.randint(n - 1, (P,), generator=gen)) % n).to(device)
    t = (torch.randint(1, 9, (P,), generator=gen).float().pow(2) / 64.0).to(device)
    sp = torch.nn.functional.softplus(torch.tensor(0.5)).to(device)
    state = {}
    times = []
    import contextlib
    # tensors the port creates itself (identities for the triangular solves ...) must land on the same device
    factory_device = torch.device(device) if device != 'cpu' else contextlib.nullcontext()
    for k in range(warmup + steps):
        if device != 'cpu':
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        with factory_device:
            xr = x.clone().requires_grad_()
            loss = O.quotient_loss(t, sp * orc.dist2(xr[I], xr[J]), 1.0, 1)
            loss.backward()
            x = O.radam_step(orc, x, xr.grad, state, lr=0.01, max_grad_norm=100, exact=True).detach()
        if device != 'cpu':
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
    O._eigh = eigh_saved
    med = float(np.median(times))
    return P / med, med, cores, f'2^{log2_pairs} pairs over {n} points per step (pairs:points = 8:1 as the full workload), ' \
                                f'fwd+bwd+RAdam step, median of {steps}'


# BASELINE configs 1-4 on the host cores: (factors, dtype, optimizer, nodes, node batch or None, CPU node sample)
CPU_CONFIGS = {
    '1': ([('spd', 3)], torch.float64, 'rsgd', 1000, None, 1000),
    '2a': ([('lorentz', 11)], torch.float32, 'radam', 4941, 512, 512),
    '2b': ([('stein', 4)], torch.float32, 'radam', 4941, 512, 512),
    '3a': ([('grassmann', (6, 2))], torch.float64, 'radam', 4039, 512, 512),
    '3b': ([('spd', 3), ('lorentz', 5)], torch.float32, 'radam', 4039, 512, 512),
    '4': ([('spd', 6)], torch.float32, 'radam', 21363, None, 1024),
}


def cpu_config_epoch(tag, steps, warmup, seed=0):
    """Epoch time of BASELINE config `tag` with the reference's CPU implementation (oracle port): times the
    forward + backward + optimizer step of ONE node batch (configs 1-3: the real batch; config 4: a 1024-node sample of
    its single 21363-node batch) and scales by pairs per epoch."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import manifolds_oracle as O
    factors, dtype, opt_name, n, batch, sample = CPU_CONFIGS[tag]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen = torch.Generator().manual_seed(seed)
    oracles, xs = [], []
    for fam, arg in factors:
        if fam in ('spd', 'stein'):
            o = O.SpdOracle(arg, stein=(fam == 'stein'))
            x = o.rand(sample, ir=0.1, dtype=dtype, generator=gen)
        elif fam == 'lorentz':
            o = O.LorentzOracle(arg)
            x = o.rand(sample, ir=1e-2, dtype=dtype, generator=gen)
        else:
            o = O.GrassmannOracle(*arg)
            x = o.rand_uniform(sample, dtype=dtype, generator=gen)
        oracles.append(o)
        xs.append(x)
    P = sample * (sample - 1) // 2
    t = (torch.randint(1, 9, (P,), generator=gen).to(dtype).pow(2) / 64.0)
    scales = [torch.tensor(0.5, dtype=dtype) for _ in factors]
    states = [{} for _ in factors]
    times = []
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        xr = [x.clone().requires_grad_() for x in xs]
        m = O.product_dist2(oracles, xr, scales, lambda o, x: o.pdist2(x))
        loss = O.quotient_loss(t, m, 1.0, 1)
        loss.backward()
        for f, (o, x, g, st) in enumerate(zip(oracles, xs, xr, states)):
            if opt_name == 'rsgd':
                xs[f] = O.rsgd_step(o, x, g.grad, st, lr=1e-3, max_grad_norm=20, exact=True).detach()
            else:
                xs[f] = O.radam_step(o, x, g.grad, st, lr=1e-3, max_grad_norm=100, exact=True).detach()
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
    med = float(np.median(times))
    bs = n if batch is None else batch
    pairs_epoch = sum(b * (b - 1) // 2 for b in (min(bs, n - i) for i in range(0, n, bs)) if b >= 50)
    rate = P / med
    return dict(config=tag, nodes=n, dtype='f32' if dtype == torch.float32 else 'f64', cores=cores,
                sample=f'one batch of {sample} nodes = {P} pairs, fwd+bwd+{opt_name} step, median of {steps}',
                pairs_per_s=rate, pairs_per_epoch=pairs_epoch, epoch_ms=pairs_epoch / rate * 1e3, kind='port')


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port: identical torch/LAPACK calls;
    the Python reference itself cannot travel to the GPU box) on all host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warmup = max(1, min(args.steps, 8)), max(1, min(args.warmup, 2))
    if args.workload != '5':  # secondary: CPU epoch time of BASELINE configs 1-4, one JSON line each
        for tag in ([t for t in CPU_CONFIGS] if args.workload == 'all' else args.workload.split(',')):
            print(json.dumps(dict(impl='reference', **cpu_config_epoch(tag, min(steps, 3), 1))), flush=True)
        return
    rate, med, cores, sample = cpu_step_rate(args.cpu_pairs_log2, steps, warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warmup, 'ms_per_step': med * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'BASELINE config 5 (SPD 4x4 affine-invariant, sampled pairs, QuotientLoss, RAdam exact '
                               'clip 100), bounded CPU sample', 'pairs_per_step': 1 << args.cpu_pairs_log2},
        'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE configs 1-4 on the GPU: epoch time through the public training API on the shipped graphs
# ---------------------------------------------------------------------------------------------------------------------
GPU_CONFIGS = {
    # tag: (graph, factors, dtype, optimizer, node batch or None, E per factor, flops per pair (SURVEY 8d estimate))
    '1': ('tree1000', [('spd', dict(n=3))], torch.float64, 'rsgd', None, [9], 900),
    '2a': ('power', [('lorentz', dict(n=11))], torch.float32, 'radam', 512, [11], None),
    '2b': ('power', [('spd', dict(n=4, use_stein_div=True))], torch.float32, 'radam', 512, [16], None),
    '3a': ('facebook', [('grassmann', dict(n=6, p=2))], torch.float64, 'radam', 512, [12], None),
    '3b': ('facebook', [('spd', dict(n=3)), ('lorentz', dict(n=5))], torch.float32, 'radam', 512, [9, 5], None),
    '4': ('condmat', [('spd', dict(n=6))], torch.float32, 'radam', None, [36], 7500),
}
GRAPH_SIZES = {'tree1000': 1000, 'power': 4941, 'facebook': 4039, 'condmat': 21363}
# non-tensor vector-pipe peaks of one B200 (148 SMs x 128 FP32 lanes (64 FP64) x 2 flop x 1.965 GHz): the bound of the
# all-pairs configs, whose traffic per pair is one target value (SURVEY 8d)
FP32_PEAK_TFLOPS, FP64_PEAK_TFLOPS = 74.4, 37.2


def load_graph(name):
    """(n, edges, source): the shipped edge list as the reference's loader numbers it (tests/golden/graphs/*.npz, made
    from /root/reference/data/<name>.edges.gz by tests/golden/make_golden_r2.py), else a synthetic scale-free graph
    of the same size -- and says which."""
    path = os.path.join(ROOT, 'tests', 'golden', 'graphs', f'{name}.npz')
    if os.path.isfile(path):
        with np.load(path) as z:
            return int(z['n']), z['edges'].astype(np.int64), f'data/{name}.edges.gz'
    n = GRAPH_SIZES[name]
    return n, scale_free_edges(n, 3, 0), f'synthetic scale-free graph of {n} nodes (shipped edge list not found)'


def gpu_config_epoch(tag, epochs, dev, with_cpu=True):
    """One BASELINE config through TrainingEngine on one GPU: median epoch ms (CUDA-synchronised wall clock around
    TrainingEngine._train, validation off), pairs/s, the pair kernels' share (CUDA events) and a roofline."""
    from graphembed import _lib as L, _ops
    from graphembed import manifolds as M
    from graphembed.data import bfs_levels, edges_to_csr
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam, RiemannianSGD
    from graphembed.train import TrainingEngine
    gname, factors, dtype, opt_name, batch_nodes, E_list, flops_pair = GPU_CONFIGS[tag]
    n, edges, gsrc = load_graph(gname)
    prev_dev = torch.empty(0).device
    torch.set_default_device(dev)  # as run.py does: the per-epoch randperm and its slices stay on the GPU
    try:
        torch.manual_seed(42)
        rowptr, colidx = edges_to_csr(n, edges)
        levels = bfs_levels(rowptr, colidx, device=dev, level_bytes=1)
        max_sq = float(levels.max().item()) ** 2
        dense = torch.empty(n, n, dtype=dtype, device=dev)
        L.check(L.lib().gm_levels_to_dense_targets(1, L.ptr(levels), n, max_sq, L.dtype_code(dtype), L.ptr(dense),
                                                   L.stream_ptr(dev)), 'gm_levels_to_dense_targets')
        del levels

        class DenseDataset:  # GraphDataset (data/dataset.py:9-27) over the already normalised dense target matrix
            pdists = dense
            device = dense.device

            def __len__(self):
                return n

        def mk(fam, kw):
            return (M.SymmetricPositiveDefinite(**kw) if fam == 'spd' else M.Lorentz(kw['n']) if fam == 'lorentz'
                    else M.Grassmann(kw['n'], kw['p']))

        emb = ManifoldEmbedding(n, [mk(f, kw) for f, kw in factors], device=dev, dtype=dtype)
        if opt_name == 'rsgd':
            opt = RiemannianSGD(emb.xs, lr=0.01, max_grad_norm=20, exact=True)   # run_grid.py:30-33
        else:
            opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)  # run_grid.py:25-28
        save_dir = tempfile.TemporaryDirectory(prefix='bench_configs_')
        eng = TrainingEngine(embedding=emb, optimizer=opt, objective_fn=QuotientLoss(), n_epochs=epochs, alpha=1.0,
                             batch_size=batch_nodes, tensorboard=False, save_dir=save_dir.name)
        kernel_events, epoch_ms = [], []

        def timed(fn):
            def wrapper(*a, **kw):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*a, **kw)
                e1.record()
                kernel_events.append((e0, e1))
                return r
            return wrapper

        saved = (_ops.pairs_loss_fused, _ops.pairs_dist2, _ops.pairs_grad)
        _ops.pairs_loss_fused, _ops.pairs_dist2, _ops.pairs_grad = (timed(f) for f in saved)
        orig_train = eng._train

        def timed_train(*a, **kw):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            r = orig_train(*a, **kw)
            torch.cuda.synchronize(dev)
            epoch_ms.append((time.perf_counter() - t0) * 1e3)
            return r

        eng._train = timed_train
        launches0 = L.launch_count()
        try:
            eng(DenseDataset())
        finally:
            _ops.pairs_loss_fused, _ops.pairs_dist2, _ops.pairs_grad = saved
        launches = L.launch_count() - launches0
        final_loss = float(eng.writer.history['quotient_loss'][-1][1])
        save_dir.cleanup()
    finally:
        torch.set_default_device(prev_dev)
    bs = n if batch_nodes is None else min(n, batch_nodes)
    sizes = [b for b in (min(bs, n - i) for i in range(0, n, bs)) if b >= 50]
    pairs = sum(b * (b - 1) // 2 for b in sizes)
    med = float(np.median(epoch_ms[1:] if len(epoch_ms) > 1 else epoch_ms))
    kernel_ms = sum(a.elapsed_time(b) for a, b in kernel_events) / max(len(epoch_ms), 1)
    kernel_basis = 'pair kernel time (CUDA events)'
    if not kernel_events:  # the whole epoch ran inside ONE native call (gm_train_epoch): kernels back to back
        kernel_ms, kernel_basis = med, 'epoch time (pair + optimizer kernels enqueued back to back by gm_train_epoch)'
    s_ = 4 if dtype == torch.float32 else 8
    bpp = sum(4 * E * s_ for E in E_list) + s_ + 8
    peak, _ = hbm_peak()
    hbm = pairs * bpp / (med * 1e-3) / 1e9
    line = {
        'workload': f'BASELINE config {tag}', 'graph': gsrc, 'nodes': n, 'dtype': 'f32' if s_ == 4 else 'f64',
        'factors': [f'{f}{tuple(kw.values())}' for f, kw in factors], 'optimizer': opt_name, 'batch_nodes': batch_nodes,
        'steps_per_epoch': len(sizes), 'pairs_per_epoch': pairs, 'epoch_ms': med, 'pairs_per_s': pairs / (med * 1e-3),
        'pair_kernels_ms_per_epoch': kernel_ms, 'gpu_launches_per_epoch': launches / max(len(epoch_ms), 1),
        'final_loss': final_loss,
        'roofline': {'bound': 'hbm', 'achieved': hbm, 'peak': peak, 'unit': 'GB/s', 'frac': hbm / peak,
                     'bytes_per_pair': bpp, 'basis': 'whole epoch (pair + optimizer kernels + launch gaps)'},
    }
    if flops_pair:  # all-pairs configs: the vector pipe is the bound (SURVEY 8d), flops per pair are SURVEY's estimate
        vpeak = FP32_PEAK_TFLOPS if s_ == 4 else FP64_PEAK_TFLOPS
        ach = pairs * flops_pair / (kernel_ms * 1e-3) / 1e12
        line['roofline_vector_pipe'] = {'bound': 'fp32_pipe' if s_ == 4 else 'fp64_pipe', 'achieved': ach, 'peak': vpeak,
                                        'unit': 'TFLOP/s', 'frac': ach / vpeak, 'flops_per_pair_estimate': flops_pair,
                                        'basis': kernel_basis}
    if with_cpu:
        c = cpu_config_epoch(tag, 1, 1 if tag in ('1', '2a', '3a', '3b') else 0)
        line['cpu_baseline'] = {'value': c['epoch_ms'], 'unit': 'ms/epoch', 'cores': c['cores'], 'kind': 'port',
                                'sample': c['sample']}
        line['speedup_vs_cpu'] = c['epoch_ms'] / med
    del eng, emb, dense
    torch.cuda.empty_cache()
    return line


def hbm_peak():
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(peaks_path):
        return json.load(open(peaks_path))['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def bfs_secondary(graph, n_nodes, dev, reps=5):
    """The multi-source BFS kernel with a FRESH BFS every step: 1024 new random sources of the 2 M-node bench graph
    per call, CUDA events around each call."""
    from graphembed.data import bfs_levels
    rp, ci = graph
    gen = torch.Generator().manual_seed(99)
    times, depth = [], 0
    for k in range(reps + 1):
        src = torch.randperm(n_nodes, generator=gen)[:N_SOURCES].int().to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lv = bfs_levels(rp, ci, sources=src, device=dev, level_bytes=1)
        e1.record()
        torch.cuda.synchronize(dev)
        if k:
            times.append(e0.elapsed_time(e1))
        depth = max(depth, int(lv.max().item()))
        del lv
    ms = float(np.median(times))
    m_edges = int(ci.numel())
    # algorithmic bytes of one BFS of S sources: the (S, N) uint8 level matrix written once, plus per level one pass
    # over the CSR arrays and the W = S/64 frontier words of every node read + the visited/next words read-modify-written
    W = N_SOURCES // 64
    per_level = m_edges * 4 + (n_nodes + 1) * 4 + n_nodes * W * 8 * 3
    alg = N_SOURCES * n_nodes + (depth + 1) * per_level
    peak, src_ = hbm_peak()
    return {'workload': f'multi-source BFS, {N_SOURCES} fresh sources per call on the {n_nodes}-node bench graph '
                        f'({m_edges} directed edges, depth {depth})', 'ms_per_call': ms,
            'source_node_levels_per_s': N_SOURCES * n_nodes / (ms * 1e-3),
            'roofline': {'bound': 'hbm', 'achieved': alg / (ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                         'frac': alg / (ms * 1e-3) / 1e9 / peak, 'algorithmic_bytes_per_call': alg,
                         'basis': 'level matrix written once + per level: CSR read, frontier words read, visited and '
                                  'next words updated'}}


def output_snapshot(trainer, loss, n_points, sharded):
    """--dump-outputs: host copies of what the step handed back -- its loss and the updated point table, of which a
    fixed sample of rows (the same rows on every run) keeps the dump small.  Row-sharded: every rank must call it."""
    x = trainer.gather() if sharded else trainer.emb.xs[0].detach()
    rows = torch.randperm(n_points, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    return {'loss': loss.detach().double().reshape(1).cpu().numpy(),
            'points': x.index_select(0, rows.to(x.device)).float().cpu().numpy()}


# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if args.workload != '5':  # one JSON line per requested BASELINE config (GPU arm), rank 0 only
        if rank == 0:
            tags = list(GPU_CONFIGS) if args.workload == 'all' else args.workload.split(',')
            for tag in tags:
                print(json.dumps({'metric': 'epoch_time', 'unit': 'ms', 'higher_is_better': False, 'n_gpus': 1,
                                  **gpu_config_epoch(tag, max(3, min(args.steps, 6)), dev,
                                                     with_cpu=not args.no_cpu_baseline)}), flush=True)
        return
    pg = None
    if args.no_peer:
        os.environ['GM_PEER_UPDATE'] = '0'
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
        pg = dist.group.WORLD

    from graphembed import _lib
    from graphembed.engine import PairTrainer
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam

    torch.manual_seed(42)  # identical replicas on every rank
    N, P_full = args.nodes, 1 << args.pairs_log2
    strong = args.scaling == 'strong' and world > 1
    n_src = N_SOURCES // world if strong else N_SOURCES  # strong: the step's 1024 sources are split over the ranks
    man = SymmetricPositiveDefinite(4)
    emb = ManifoldEmbedding(N, [man], device=dev, dtype=torch.float32)
    opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
    # every rank draws its own batches (different seed) on the same graph; embeddings replicated
    batches, max_sq, levels, per_src, graph = make_pair_batches(N, args.pairs_log2, args.batches, dev, seed=1234 + rank,
                                                                n_src=n_src, keep_levels=True, windows=args.windows)
    P = n_src * per_src  # pairs per step on this rank
    seg = args.windows if args.windows > 1 else 0
    if pg is not None:
        m = torch.tensor([max_sq], device=dev)
        torch.distributed.all_reduce(m, op=torch.distributed.ReduceOp.MAX)
        max_sq = float(m.item())
    sharded = args.layout == 'sharded' and world > 1
    if sharded:
        from graphembed.engine import ShardedPairTrainer
        trainer = ShardedPairTrainer(emb, opt, QuotientLoss(), max_hops_sq=max_sq, process_group=pg, alpha=1.0)
    else:
        trainer = PairTrainer(emb, opt, QuotientLoss(), max_hops_sq=max_sq, alpha=1.0, process_group=pg)
    if args.unpacked:
        dev_batches = [tuple(t.to(dev) for t in b[:3]) for b in batches]
    else:  # (i, j | hops << 24): the hop count rides in the top byte of the second index
        dev_batches = [(b[0].to(dev), b[5].to(dev), None) for b in batches]

    def barrier():
        if pg is not None:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing (value, roofline) ----------------------------------------------------------------
    for k in range(args.warmup):
        trainer.step(*dev_batches[k % len(dev_batches)], epoch=1, segments=seg)
    # per-kernel events for the dominant (pair) kernel: bracket it inside the step by patching the trainer's call
    from graphembed import _ops
    pair_events = []
    pair_fn = 'pairs_loss_fused_sharded' if sharded else 'pairs_loss_fused'
    orig = getattr(_ops, pair_fn)

    def timed_pairs(*a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig(*a, **kw)
        e1.record()
        pair_events.append((e0, e1))
        return r

    setattr(_ops, pair_fn, timed_pairs)
    # N>1: also bracket the optimizer call (the fused peer-memory owner update, or the owner update between the NCCL
    # reduce-scatter and all-gather); it includes the wait for the slowest rank's pair kernel
    upd_events = []
    opt_step = trainer.opt.step

    def timed_update(*a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = opt_step(*a, **kw)
        e1.record()
        upd_events.append((e0, e1))
        return r

    if world > 1:
        trainer.opt.step = timed_update
    clocks = ClockSampler(local)
    nvl = NvlinkCounter(local) if world > 1 else None
    barrier()
    if rank == 0:
        clocks.start()
    launches0 = _lib.launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    loss = None
    for k in range(args.steps):
        loss = trainer.step(*dev_batches[k % len(dev_batches)], epoch=1, segments=seg)
    t1.record()
    barrier()
    # taken before the steps below move the points on
    outputs = output_snapshot(trainer, loss, N, sharded) if args.dump_outputs and (rank == 0 or sharded) else None
    nvlink = None
    if nvl:  # NVLink payload bytes per step, from the driver's counters, over a few extra (untimed) steps
        nvl.start()
        for k in range(5):
            trainer.step(*dev_batches[k % len(dev_batches)], epoch=1, segments=seg)
        barrier()
        nvlink = nvl.stop(5)
    launches = _lib.launch_count() - launches0
    setattr(_ops, pair_fn, orig)
    trainer.opt.step = opt_step
    upd_ms = float(np.mean([a.elapsed_time(b) for a, b in upd_events])) if upd_events else None
    ms = t0.elapsed_time(t1)
    pair_ms = float(np.mean([a.elapsed_time(b) for a, b in pair_events]))
    final_loss = float(loss.item())

    # ---- end-to-end timing from pinned host buffers ----------------------------------------------------------------
    nb = len(batches)
    # auto: explicit lists at every GPU count, as 2-byte gap words (measured end to end, ms per step lists2 / sampled: 4 GPUs
    # 1.556 / 1.722, 8 GPUs 1.740 / 1.778 before the expansion kernel was vectorised; 4-byte lists at 4 GPUs: 1.909)
    e2e_mode = args.e2e if args.e2e != 'auto' else 'lists'
    if e2e_mode == 'lists':
        # source-grouped upload (sources, offsets, j, hops): 4-5 B/pair over PCIe; the next batch is uploaded on a
        # second stream while this one computes; every step ends with a device->host read of the loss
        use3 = args.lists3 and not args.unpacked and all(b[6] is not None for b in batches)
        use2 = (args.lists_format in ('2', 'auto') and not args.lists3
                and not args.unpacked and all(b[7] is not None for b in batches))

        def grouped(b):
            if use2:
                return (b[3], b[4], b[7][0], None, b[7][1])
            if use3:
                return (b[3], b[4], b[6], None, None)
            return (b[3], b[4], b[1], b[2], None) if args.unpacked else (b[3], b[4], b[5], None, None)

        def e2e_step(k):
            cur = grouped(batches[k % nb])
            return trainer.step_host_grouped(*cur[:4], epoch=1, next_batch=grouped(batches[(k + 1) % nb]),
                                             defer_loss=True, segments=seg, bases=cur[4])
        h2d_bytes = sum(t.numel() * t.element_size() for t in grouped(batches[0]) if t is not None)
        e2e_api = ('graphembed.engine.PairTrainer.step_host_grouped (pinned host int32 sources, int64 offsets, '
                   + ('int32 j, uint8 hops' if args.unpacked else
                      '2-byte words (every source\'s targets sorted by row: 13-bit gap | (hops - 1) << 13, + one int32 '
                      'base per source), expanded on the device by gm_unpack_pairs2' if use2 else
                      '3-byte words j | (hops - 1) << 21, expanded on the device' if use3 else 'int32 j | hops << 24')
                   + '; per rank); next batch '
                   'uploaded on a second stream, loss read back through pinned memory one step late')
    else:
        # the step's input is its list of BFS sources: 4 KB from pinned host memory per step; targets are drawn inside
        # the pair kernel, hop counts come from the resident level matrix of the batch's landmark sources
        def e2e_step(k):
            return trainer.step_sampled_host(batches[k % nb][3], levels[k % nb], per_src, seed=(0xB200 << 32) + k,
                                             epoch=1, defer_loss=True)
        h2d_bytes = batches[0][3].numel() * 4
        e2e_api = ('graphembed.engine.PairTrainer.step_sampled_host (pinned host int32 source ids of the step; '
                   f'{per_src} targets per source drawn inside the pair kernel from the counter hash of (seed, pair '
                   'number), hop counts from the HBM-resident BFS level matrix of the landmark sources); loss read back '
                   'through pinned memory one step late')
    for k in range(2):
        e2e_step(k)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    host_losses = [e2e_step(k) for k in range(args.steps)]
    host_losses.append(trainer.flush_loss())  # every step's loss reaches the host, one step late
    e1.record()
    barrier()
    assert all(v is not None and np.isfinite(v) for v in host_losses[1:]), host_losses
    ms_e2e = e0.elapsed_time(e1)
    clock_info = clocks.stop() if rank == 0 else None  # sampled over both timed regions

    if pg is not None:
        t = torch.tensor([ms, ms_e2e, pair_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms, ms_e2e, pair_ms = (float(v) for v in t.tolist())
    if rank != 0:
        if pg is not None:
            torch.distributed.destroy_process_group()
        return
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f'{name}.npy'), a)

    peak, peak_src = hbm_peak()
    achieved = P * BYTES_PER_PAIR / (pair_ms * 1e-3) / 1e9
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full capture
    tpath = os.path.join(ROOT, 'profiles', 'pair_kernel_traffic.json')
    if os.path.isfile(tpath) and P == (1 << 24) and N == 2_000_000:
        traffic = json.load(open(tpath)).get('dram_bytes_per_launch' if seg == 8 else 'dram_bytes_per_launch_windows0' if seg == 0 else 'none')
    total_pairs = P * world * args.steps
    line = {
        'metric': METRIC, 'value': total_pairs / (ms * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {
            'workload': 'BASELINE config 5: synthetic scale-free graph, SPD 4x4 affine-invariant, sampled pairs '
                        f'({N_SOURCES} BFS sources x targets per step' + (' in total, sources split over the GPUs'
                                                                         if strong else ' per GPU')
                        + '), QuotientLoss, RiemannianAdam(lr .01, clip 100, exact)',
            'nodes': N, 'pairs_per_step_per_gpu': P, 'layout': 'sharded' if sharded else 'replicated',
            'parallelism': f'pair-sharded x{world}'
            + (' + ROW-SHARDED embeddings (row v on rank v % G): the pair kernel gathers remote rows and reduces remote '
               'gradient rows over NVLink peer memory, two flag barriers, LOCAL optimizer update of the owned N/G rows '
               '(gm_pairs_loss_fused_sharded + gm_peer_barrier + gm_optim_step, no NCCL on the step path)'
               if sharded else
               ' + ONE fused kernel over NVLink peer memory: pull+sum the owned (N/G,4,4) gradient rows from every '
               'rank, optimizer update, push the new rows to every rank (gm_optim_step_peer, no NCCL on the step path)'
               if trainer.peer is not None else
               ' + NCCL reduce-scatter of the (N,4,4) gradient, owner-rank optimizer update, all-gather of the points'
               if trainer.shards is not None else (' + NCCL all-reduce of the (N,4,4) gradient' if world > 1 else '')),
            'l2_policy': f'inputs larger than L2: {len(batches)} distinct batches of '
                         f'{P * (9 if args.unpacked else 8) / 1e6:.0f} MB cycled, '
                         f'{N * 64 / 1e6:.0f} MB embedding + {N * 64 / 1e6:.0f} MB gradient touched at random'
                         + (f'; every batch is in (window of the target row, source) order, {seg} windows: inside a '
                            f'step the kernel works through one {N * 64 / seg / 1e6:.0f} MB slice of the embedding and '
                            'of the gradient at a time, which is meant to stay in L2 (gm_pairs_t.segments); nothing '
                            'is reused across steps' if seg else ''),
            'windows': seg,
            'final_loss': final_loss,
            **({'optimizer_call_ms_rank0': upd_ms} if upd_ms is not None else {}),
            **({'nvlink_rank0': nvlink} if nvlink is not None else {}),
        },
        'e2e': {'value': total_pairs / (ms_e2e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d_bytes,
                'd2h_bytes_per_step': 16, 'ms_per_step': ms_e2e / args.steps, 'api': e2e_api},
        'gpu_launches': int(launches),
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'kernel': 'spd_pair_stream_kernel<SpdAI<float,4>,K_FUSED>',
                     'kernel_ms': pair_ms, 'bytes_per_pair': BYTES_PER_PAIR, 'peak_source': peak_src,
                     'note': ('achieved = algorithmic bytes (268 B per pair: two 64-B rows read, two 64-B gradient rows '
                              'read-modify-written, index + hop word) / kernel time, as SURVEY 8(d) defines it.  With '
                              'window-ordered batches most of those bytes are served by L2 (traffic = measured DRAM '
                              'bytes per launch, far below the algorithmic figure) and the kernel is bound by '
                              'instruction issue (ncu: issue-active 74 %, profiles/r02_pairs_final_full.txt), not by HBM')
                     if seg else None},
        'clocks': clock_info,
    }
    if not args.no_cpu_baseline:
        rate, med, cores, sample = cpu_step_rate(args.cpu_pairs_log2, 3, 1)
        line['cpu_baseline'] = {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample}
        if world == 1:
            try:  # SURVEY 8(d) second comparator: the same torch-op path with its tensors on this B200
                rate_g, med_g, _, sample_g = cpu_step_rate(args.cpu_pairs_log2, 3, 1, device='cuda')
                line['cpu_baseline']['torch_ops_on_this_gpu'] = {
                    'value': rate_g, 'unit': UNIT, 'sample': sample_g,
                    'what': "the reference's PyTorch-op implementation (oracle port: batched torch.linalg.cholesky, "
                            'autograd, index_put_ scatter) with every tensor on the B200 and, as the reference does '
                            '(linalg/torch_batch.py:94-135 cpu_offload=True), the batched eigh round-tripped through '
                            'the host'}
            except Exception as e:  # noqa: BLE001 -- a comparator must not take the bench line down
                line['cpu_baseline']['torch_ops_on_this_gpu'] = {'unavailable': repr(e)[:200]}
    if world == 1 and not args.no_secondary:
        del trainer, emb, dev_batches, levels
        torch.cuda.empty_cache()
        sec = {'bfs': bfs_secondary(graph, N, dev)}
        sec['configs'] = [gpu_config_epoch(tag, 4, dev, with_cpu=not args.no_cpu_baseline) for tag in GPU_CONFIGS]
        line['secondary'] = sec
    print(json.dumps(line))
    if pg is not None:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
