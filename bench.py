#!/usr/bin/env python
"""Headline benchmark: forward point-clouds / second of the SE(3)-Transformer attention hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl ours|reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[1] ("cfg2": batch 4, N=1024, dim 512, heads 8, dim_head 64, depth 6, num_degrees 4,
k-NN 16) per GPU; with N GPUs every rank runs its own batch of 4 clouds (weak scaling, no data-path collective) and the
returned type-0 features are all-gathered so that every rank holds the whole batch.  A "step" is one forward pass.

  value  : clouds/s with the inputs already resident in HBM (CUDA events, max over ranks)
  e2e    : clouds/s through the public API with HOST inputs: pinned H2D of feats/coors/mask + forward + D2H of the result
  roofline: the dominant kernel (fused tcgen05 pairwise kernel): algorithmic FLOPs / CUDA-event time vs measured bf16 peak
  cpu_baseline / --impl reference: the numpy oracle (port of the reference algorithm) timed on the host cores on a
           bounded, width-preserving sample, extrapolated by algorithmic FLOPs (the full workload needs ~79 h on CPU).

--dump-outputs DIR writes what the last timed step returned (the headline arm: the forward's output, all-gathered over the
ranks; --impl reference: the sampled ConvSE3's output) as DIR/<name>.npy, so that two builds can be compared output for
output: inputs and weights come from fixed seeds, identical from run to run for the same arguments.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'cfg1': dict(ctor=dict(dim=64, depth=2, num_degrees=2, num_neighbors=8), b=1, n=32),
    'cfg2': dict(ctor=dict(dim=512, heads=8, dim_head=64, depth=6, num_degrees=4, num_neighbors=16), b=4, n=1024),
    'cfg3': dict(ctor=dict(dim=64, depth=2, input_degrees=1, num_degrees=2, output_degrees=2, reduce_dim_out=True, num_neighbors=16),
                 b=2, n=256, fwd=dict(return_type=1)),
    'cfg4': dict(ctor=dict(dim=128, depth=2, num_degrees=3, num_edge_tokens=4, edge_dim=16, attend_sparse_neighbors=True, num_neighbors=0,
                           max_sparse_neighbors=8), b=8, n=512, edges='tokens', adj=4),
    'cfg5': dict(ctor=dict(dim=512, heads=8, dim_head=64, depth=6, num_degrees=4, num_neighbors=32), b=8, n=2048),
    # reduced-width variants for quick iteration (NOT the headline)
    'cfg2_d128': dict(ctor=dict(dim=128, heads=8, dim_head=16, depth=6, num_degrees=4, num_neighbors=16), b=4, n=1024),
    'cfg2_depth1': dict(ctor=dict(dim=512, heads=8, dim_head=64, depth=1, num_degrees=4, num_neighbors=16), b=4, n=1024),
    # weights-sensitivity experiment: Fourier-encoded distances make the radial functions rougher (higher rank of the radial model)
    'cfg2_depth1_fourier': dict(ctor=dict(dim=512, heads=8, dim_head=64, depth=1, num_degrees=4, num_neighbors=16, fourier_encode_dist=True,
                                          rel_dist_num_fourier_features=4), b=4, n=1024),
}


def conv_list(ctor):
    """[(fiber_in, fiber_out)] of every ConvSE3 in the model (reference S:1074-1113): conv_in, 2 per attention block, conv_out."""
    dim = ctor['dim']
    nd = ctor['num_degrees']
    hid_attn = ctor.get('heads', 8) * ctor.get('dim_head', 24)
    f_in = [(d, dim) for d in range(ctor.get('input_degrees', 1))]
    f_hid = [(d, dim) for d in range(nd)]
    f_kv = [(d, hid_attn) for d in range(nd)]
    f_out = [(d, dim) for d in range(ctor.get('output_degrees', 1))]
    convs = [(f_in, f_hid)]
    for _ in range(ctor.get('depth', 2)):
        convs += [(f_hid, f_kv), (f_hid, f_kv)]
    convs.append((f_hid, f_out))
    return convs


def conv_flops(f_in, f_out, edges):
    """Algorithmic FLOPs of one ConvSE3 on `edges` edges (SURVEY.md 8d): radial last layer 2*128 per R element +
    contraction 2*(2lo+1) per R element."""
    tot = 0
    for di, ci in f_in:
        for do, co in f_out:
            f = 2 * min(di, do) + 1
            tot += edges * co * ci * f * (2 * 128 + 2 * (2 * do + 1))
    return tot


def forward_flops(wl):
    c = wl['ctor']
    edges = wl['b'] * wl['n'] * neighbours(wl)
    return sum(conv_flops(fi, fo, edges) for fi, fo in conv_list(c))


def neighbours(wl):
    c = wl['ctor']
    k = int(min(c.get('num_neighbors', float('inf')), wl['n'] - 1))
    if c.get('attend_sparse_neighbors'):
        k += int(min(c.get('max_sparse_neighbors', 0), 2 * wl.get('adj', 0)))
    return k


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p['hbm_gbs'], bf16_burst=p['bf16_tflops'], bf16_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source='fallback (B200_PROFILING.md)')


DUMP_BYTES = 64 << 20


def output_arrays(out):
    """The forward's return value (one tensor, or a dict degree -> tensor) as host arrays named for --dump-outputs."""
    import numpy as np
    host = lambda t: t.detach().cpu().numpy() if hasattr(t, 'detach') else np.asarray(t)
    if isinstance(out, dict):
        return {f'type{d}': host(t) for d, t in out.items()}
    return {'out': host(out)}


def dump_outputs(arrays, path):
    """Write every array as path/<name>.npy, float64 kept and anything else as float32.  Past DUMP_BYTES in all, each array
    keeps the same fraction of its rows (rows = the flattened batch x point axes), drawn once from a fixed seed and kept in
    order, so that runs of the same arguments still sample the same points."""
    import numpy as np
    arrays = {k: (a if a.dtype == np.float64 else a.astype(np.float32)) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            rows = a.reshape(-1, *a.shape[2:]) if a.ndim > 2 else a.reshape(-1)
            keep = max(1, len(rows) * DUMP_BYTES // total)
            a = rows[np.sort(np.random.default_rng(0).choice(len(rows), keep, replace=False))]
        np.save(os.path.join(path, f'{name}.npy'), a)


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline: the numpy oracle on a bounded, width-preserving sample
# ------------------------------------------------------------------------------------------------------------------
class CpuSample:
    """ONE hidden->hidden ConvSE3 (pool=False: the K or V projection, >96 % of the forward's work) of the workload's widths,
    evaluated by the oracle on a small random edge set.  prepare() builds weights/inputs once; run() is the timed part."""

    def __init__(self, wl, target_flops=3e11, seed=0):
        import numpy as np
        from oracle import se3_oracle as O
        self.O, self.wl = O, wl
        c = wl['ctor']
        nd, dim = c['num_degrees'], c['dim']
        hid = c.get('heads', 8) * c.get('dim_head', 24)
        k = neighbours(wl)
        e_dim = c.get('edge_dim') or 0               # per-edge features next to the distance (BASELINE configs[3])
        self.f_in = [(d, dim) for d in range(nd)]
        self.f_out = [(d, hid) for d in range(nd)]
        per_edge = conv_flops(self.f_in, self.f_out, 1)
        edges = max(k, int(target_flops / per_edge))
        n = max(k + 1, (edges + k - 1) // k)
        rng = np.random.default_rng(seed)
        P = {}
        for di, ci in self.f_in:
            for do, co in self.f_out:
                f = 2 * min(di, do) + 1
                pp = f'to_v.kernel_unary.({di},{do}).rp.'
                P[pp + 'net.0.weight'] = rng.standard_normal((128, 1 + e_dim), dtype=np.float32)
                P[pp + 'net.0.bias'] = np.zeros(128, np.float32)
                P[pp + 'net.1.weight'] = np.ones(128, np.float32)
                P[pp + 'net.1.bias'] = np.zeros(128, np.float32)
                P[pp + 'net.3.weight'] = rng.standard_normal((128, 128), dtype=np.float32) / np.float32(11.3)
                P[pp + 'net.3.bias'] = np.zeros(128, np.float32)
                P[pp + 'net.4.weight'] = np.ones(128, np.float32)
                P[pp + 'net.4.bias'] = np.zeros(128, np.float32)
                w = rng.random((co * ci * f, 128), dtype=np.float32)
                w -= np.float32(0.5)
                w *= np.float32(2 / 11.3)
                P[pp + 'net.6.weight'] = w
                P[pp + 'net.6.bias'] = np.zeros(co * ci * f, np.float32)
        self.P = P
        coors = rng.standard_normal((1, n, 3)).astype(np.float32)
        self.feats = {str(d): rng.standard_normal((1, n, ci, 2 * d + 1)).astype(np.float32) for d, ci in self.f_in}
        self.graph = O.neighbor_graph(coors, None, num_neighbors=k)
        self.e_dim = e_dim
        if e_dim:
            self.graph['edges'] = rng.standard_normal((1, n, k, e_dim)).astype(np.float32)
        self.basis = O.get_basis(self.graph['rel_pos'], nd - 1)
        self.chunk = max(1, int(2 ** 28 // (hid * dim * (2 * (nd - 1) + 1))))
        self.E = n * k
        self.flops = conv_flops(self.f_in, self.f_out, self.E)
        self.desc = (f'oracle (numpy port of the reference algorithm) on one hidden->hidden ConvSE3 (to_v) at full widths '
                     f'(C_in={dim}, C_out={hid}, degrees {nd}, k={k}) over {self.E} edges; clouds/s extrapolated by algorithmic FLOPs '
                     f'({self.flops:.3e} sampled vs {forward_flops(wl) / wl["b"]:.3e} per cloud)')

    def run(self):
        # all host threads, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 for its workers)
        from threadpoolctl import threadpool_limits, threadpool_info
        with threadpool_limits(limits=os.cpu_count()):
            self.threads = max([p.get('num_threads', 1) for p in threadpool_info()] or [1])
            t0 = time.perf_counter()
            self.out = self.O.conv_se3(self.feats, self.graph, self.basis, self.P, 'to_v.', self.f_in, self.f_out, pool=False,
                                       self_interaction=False, edge_chunk=self.chunk)
            return time.perf_counter() - t0

    def gpu_parity(self, dev):
        """The same ConvSE3 (same weights, same inputs, full widths) through the product's production dispatch on the GPU --
        low-rank radial basis in edge-aligned frames, forced on for this small edge set -- against the oracle output of run()."""
        import numpy as np
        import torch
        from se3_transformer_pytorch_b200 import ops
        from se3_transformer_pytorch_b200.model import ConvSE3, Fiber, Geometry
        conv = ConvSE3(Fiber(self.f_in), Fiber(self.f_out), pool=False, self_interaction=False, edge_dim=self.e_dim)
        sd = {k[len('to_v.'):]: torch.from_numpy(v) for k, v in self.P.items()}
        conv.load_state_dict(sd)
        conv = conv.to(dev).eval()
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        g = self.graph
        inp = {d: t(v) for d, v in self.feats.items()}
        nd = len(self.f_in)
        prev = os.environ.get('SE3B200_LOWRANK_MIN_EDGES')
        os.environ['SE3B200_LOWRANK_MIN_EDGES'] = '0'
        ops.PROFILE = []
        try:
            with torch.no_grad():
                rel_pos = t(g['rel_pos'])
                basis = ops.basis_flat(rel_pos, nd - 1) + (Geometry(rel_pos, nd - 1),)
                out = conv(inp, (t(g['idx']), t(g['mask']), t(g['edges']) if self.e_dim else None), t(g['rel_dist']), basis)
            torch.cuda.synchronize()
        finally:
            kinds = sorted({p[0] for p in ops.PROFILE})
            ops.PROFILE = None
            if prev is None:
                del os.environ['SE3B200_LOWRANK_MIN_EDGES']
            else:
                os.environ['SE3B200_LOWRANK_MIN_EDGES'] = prev
        worst = 0.0
        for d, ref in self.out.items():
            got = out[d].cpu().numpy().astype(np.float64)
            worst = max(worst, float(np.abs(got - ref).max() / np.abs(ref).max()))
        return {'rel_err': worst, 'edges': int(self.E), 'vs': 'oracle', 'tolerance': 1e-4, 'kernels': kinds,
                'what': 'one hidden->hidden ConvSE3 at the workload widths: GPU production dispatch vs the numpy oracle on the same weights and edges '
                        '(max over output degrees of max|gpu - oracle| / max|oracle|)'}

    def clouds_per_s(self, seconds):
        return (self.flops / seconds) / (forward_flops(self.wl) / self.wl['b'])


def run_reference(args, wl, rank, world):
    """--impl reference: the reference algorithm's CPU restatement (oracle port) on the host cores, rank 0 only."""
    if rank != 0:
        return
    import numpy as np  # noqa: F401
    sample = CpuSample(wl, target_flops=args.cpu_flops)
    for _ in range(min(args.warmup, 1)):
        sample.run()
    times = [sample.run() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(output_arrays(sample.out), args.dump_outputs)
    sec = sum(times) / len(times)
    value = sample.clouds_per_s(sec)
    desc = sample.desc
    line = {
        'impl': 'reference', 'metric': 'point-clouds/sec fwd', 'value': value, 'unit': 'clouds/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': args.workload, **{k: v for k, v in wl['ctor'].items()}, 'batch_per_gpu': wl['b'], 'n_points': wl['n']},
        'cpu_baseline': {'value': value, 'unit': 'clouds/s', 'cores': sample.threads, 'kind': 'port', 'sample': desc},
        'e2e': {'value': value, 'unit': 'clouds/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.gpu_index}', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        with open(self.path) as f:
            for ln in f:
                parts = [p.strip() for p in ln.split(',')]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    smax.append(float(parts[2]))
                    power.append(float(parts[3]))
                except ValueError:
                    continue
                for nm, val in zip(names, parts[5:9]):
                    if val.lower().startswith('active'):
                        reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(smax), 'power_w_max': max(power), 'samples': len(sm),
                'reasons': sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args, wl, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from se3_transformer_pytorch_b200 import SE3Transformer, ops
    from se3_transformer_pytorch_b200.parallel import all_gather_batch

    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    torch.manual_seed(1234 + rank)
    t_build = time.perf_counter()
    with torch.device(dev):
        model = SE3Transformer(**wl['ctor'])
    model.eval()
    if args.global_batch:
        assert args.global_batch % world == 0, '--global-batch must be divisible by the number of GPUs'
        wl = dict(wl, b=args.global_batch // world)
    if args.radial_scale != 1.0:
        # weights-sensitivity experiment: a less smooth radial MLP (first-layer weights scaled up) needs a higher rank
        with torch.no_grad():
            for m in model.conv_modules():
                for pc in m.kernel_unary.values():
                    pc.rp.net['0'].weight.mul_(args.radial_scale)
    lowrank = ops.lowrank_enabled(wl['b'] * wl['n'] * neighbours(wl)) and not wl['ctor'].get('edge_dim')
    # tensor-core operand images (low-rank plan for distances <= 16 where the radial functions are distance-only, the
    # direct K=128 image otherwise); fp32 masters of net.6 released (inference)
    model.pack_weights(free_master=True, max_distance=16.0 if lowrank else None)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build
    weights_gb = torch.cuda.memory_allocated(dev) / 1e9
    b, n, dim = wl['b'], wl['n'], wl['ctor']['dim']
    fwd_kw = wl.get('fwd', {})
    g = torch.Generator().manual_seed(99 + rank)
    h_feats = torch.randn(b, n, dim, generator=g).pin_memory()
    h_coors = torch.randn(b, n, 3, generator=g).pin_memory()
    h_mask = torch.ones(b, n, dtype=torch.bool).pin_memory()
    if wl.get('edges') == 'tokens':                      # BASELINE configs[3]: edge tokens + band adjacency (|i - j| <= adj bonded neighbours)
        seq = torch.arange(n)
        fwd_kw = dict(fwd_kw, edges=torch.randint(0, wl['ctor']['num_edge_tokens'], (b, n, n), generator=g).to(dev),
                      adj_mat=((seq[:, None] - seq[None, :]).abs() <= wl['adj']).to(dev))

    graphed = None
    if args.cuda_graph:
        graphed = model.graphed(h_feats, h_coors, h_mask, **fwd_kw)

    def step_resident(inputs):
        out = graphed(*inputs) if graphed is not None else model(*inputs, **fwd_kw)
        if world > 1:
            out = all_gather_batch(out, b * world)
        return out

    def step_e2e():
        if graphed is not None:
            inputs = (h_feats, h_coors, h_mask)        # the graph's static input buffers are the H2D destination
        else:
            inputs = (h_feats.to(dev, non_blocking=True), h_coors.to(dev, non_blocking=True), h_mask.to(dev, non_blocking=True))
        out = step_resident(inputs)
        host = {k: v.cpu() for k, v in out.items()} if isinstance(out, dict) else out.cpu()
        return host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), res

    for _ in range(max(args.warmup, 3)):
        step_e2e()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # (1) end to end through the public API with host buffers
    ms_e2e, host_out = timed(step_e2e, args.steps)
    # (2) inputs resident in HBM; per-kernel CUDA-event brackets for the roofline
    dev_inputs = (h_feats.to(dev), h_coors.to(dev), h_mask.to(dev))
    launches0 = ops.LAUNCHES
    ops.PROFILE = []
    if args.profile_range:
        torch.cuda.cudart().cudaProfilerStart()
    ms_res, last_out = timed(lambda: step_resident(dev_inputs), args.steps)
    if args.profile_range:
        torch.cuda.cudart().cudaProfilerStop()
    prof, ops.PROFILE = ops.PROFILE, None
    launches = ops.LAUNCHES - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(output_arrays(last_out), args.dump_outputs)
    del last_out

    kern = {}
    detail = {}
    for name, s_ev, e_ev, fl, nb, tag, mma, fma in prof:
        ms = s_ev.elapsed_time(e_ev)
        d = kern.setdefault(name, dict(ms=0.0, flops=0, bytes=0, launches=0, mma=0, fma=0))
        d['ms'] += ms
        d['flops'] += fl
        d['mma'] += mma
        d['fma'] += fma
        d['bytes'] += nb
        d['launches'] += 1
        if tag:
            t = detail.setdefault(tag, dict(ms=0.0, flops=0, launches=0, mma=0))
            t['ms'] += ms
            t['flops'] += fl
            t['mma'] += mma
            t['launches'] += 1
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()         # before rank 0 spends a minute on the CPU baseline
    if rank != 0:
        return
    peaks = load_peaks()
    clouds = b * world * args.steps
    value = clouds / (ms_res / 1e3)
    e2e = clouds / (ms_e2e / 1e3)
    h2d = h_feats.numel() * 4 + h_coors.numel() * 4 + h_mask.numel()
    d2h = sum(v.numel() * 4 for v in host_out.values()) if isinstance(host_out, dict) else host_out.numel() * 4
    top = max(kern.items(), key=lambda kv: kv[1]['ms'])[0] if kern else None
    ncu = {}
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        with open(tpath) as f:
            ncu = json.load(f)
    roof = None
    if top:
        d = kern[top]
        nd = ncu.get(top) if isinstance(ncu.get(top), dict) else {}
        if d['mma'] > 0:
            # tensor-bound kernel: what the tensor cores really ISSUE (every fp16 pass of the 3-pass fp32-parity split counted)
            # per CUDA-event second, against the measured sustained cuBLAS bf16 rate (fp16 and bf16 share the pipe rate)
            ach = d['mma'] / (d['ms'] / 1e3) / 1e12
            roof = {'kernel': top, 'bound': 'tensor', 'achieved': ach, 'peak': peaks['bf16_sustained'], 'unit': 'TFLOP/s',
                    'frac': ach / peaks['bf16_sustained'], 'traffic': nd.get('dram_bytes_per_launch'),
                    'peak_source': peaks['source'] + ', sustained cuBLAS bf16', 'avg_launch_ms': d['ms'] / d['launches'],
                    'share_of_step': d['ms'] / ms_res,
                    'issued_fp32_fma_tflops': d['fma'] / (d['ms'] / 1e3) / 1e12,
                    'tensor_pipe_pct_ncu': nd.get('sm__pipe_tensor_cycles_active_pct'),
                    'algorithmic_bytes_per_launch': d['bytes'] / d['launches'],
                    'algorithmic_speedup': {
                        'reference_formulation_tflops': d['flops'] / (d['ms'] / 1e3) / 1e12,
                        'vs_issued': d['flops'] / max(d['mma'], 1),
                        'note': 'FLOPs of the reference formulation (SURVEY 8d: 2*128 radial GEMM + 2*(2lo+1) contraction per radial weight) per second; '
                                'NOT a hardware fraction: the low-rank radial basis + edge-aligned frames evaluate the same result with fewer operations'},
                    'note': 'achieved = ISSUED tensor-core FLOPs (3 fp16 passes x 2*M*N*K, CUDA events on the launching stream, all launches of the '
                            'timed steps) / time; frac = achieved / measured sustained cuBLAS bf16 TFLOP/s (MEASURED_PEAKS.json); tensor_pipe_pct_ncu and '
                            'traffic come from the committed ncu capture of the same kernel (profiles/traffic.json)',
                    'ncu_detail': nd or None}
        else:
            ach = d['bytes'] / (d['ms'] / 1e3) / 1e9
            roof = {'kernel': top, 'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'],
                    'traffic': nd.get('dram_bytes_per_launch'), 'peak_source': peaks['source']}
    hbm_kernels = {}
    for name, d in kern.items():
        if d['mma'] == 0 and d['bytes'] > 0 and d['ms'] > 0:
            ach = d['bytes'] / (d['ms'] / 1e3) / 1e9
            hbm_kernels[name] = {'achieved_GBs': ach, 'frac_of_hbm_peak': ach / peaks['hbm_gbs'], 'ms_per_step': d['ms'] / args.steps,
                                 'launches_per_step': d['launches'] / args.steps, 'bytes': 'algorithmic, no layout padding'}
    timed_ms = sum(v['ms'] for v in kern.values()) / args.steps
    khist = {}
    for m in model.conv_modules():
        for pair, pp in ((m._packed or {}).get('lr') or {}).get('pairs', {}).items():
            khist[str(pp['Kp'])] = khist.get(str(pp['Kp']), 0) + 1
    cpu, parity = None, None
    if not args.no_cpu_baseline and world == 1:          # reported at N = 1 only (the reference arm covers every N)
        sample = CpuSample(wl, target_flops=args.cpu_flops)
        dt = sample.run()
        cpu = {'value': sample.clouds_per_s(dt), 'unit': 'clouds/s', 'cores': sample.threads, 'kind': 'port', 'sample': sample.desc,
               'sample_seconds': dt}
        del model
        torch.cuda.empty_cache()
        parity = sample.gpu_parity(dev)
    line = {
        'metric': 'point-clouds/sec fwd', 'value': value, 'unit': 'clouds/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_res / args.steps, 'higher_is_better': True, 'scaling': 'strong' if args.global_batch else 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': args.workload, **wl['ctor'], 'batch_per_gpu': b, 'global_batch': b * world, 'n_points': n,
                   'parallelism': f'dp{world} (batch sharded, replicated weights, one all-gather of outputs)',
                   'cache': f'inputs larger than L2: every step streams the {weights_gb:.1f} GB of weight images and the per-layer T / K / V tensors (several GB each)', 'weights_resident_gb': weights_gb, 'random_init': True, 'cuda_graph': bool(args.cuda_graph), 'lowrank_radial': bool(lowrank),
                   'flops_per_cloud': forward_flops(wl) / b, 'model_build_s': t_build, 'radial_scale': args.radial_scale},
        'e2e': {'value': e2e, 'unit': 'clouds/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': ms_e2e / args.steps},
        'gpu_launches': launches,
        'clocks': clocks,
        'roofline': roof,
        'hbm_kernels': hbm_kernels,
        'kernel_ms_per_step': {k: v['ms'] / args.steps for k, v in sorted(kern.items(), key=lambda kv: -kv[1]['ms'])},
        'untimed_share_of_step': 1.0 - timed_ms / (ms_res / args.steps),
        'pairwise_detail': {k: {'ms_per_launch': v['ms'] / v['launches'], 'issued_mma_tflops': v['mma'] / v['ms'] / 1e9,
                                'reference_formulation_tflops': v['flops'] / v['ms'] / 1e9, 'launches': v['launches']}
                            for k, v in sorted(detail.items())},
        'lowrank_K_histogram': khist,
        'weights_sensitivity': ncu.get('weights_sensitivity'),
        'parity': parity,
        'cpu_baseline': cpu,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--cpu-flops', type=float, default=3e11, help='size of the bounded CPU sample (algorithmic FLOPs)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--global-batch', type=int, default=0, help='STRONG scaling: fixed global batch split over the ranks (default: weak scaling, the workload batch per rank)')
    ap.add_argument('--radial-scale', type=float, default=1.0, help='weights-sensitivity experiment: scale RadialFunc.net.0.weight (rougher radial functions, higher rank)')
    ap.add_argument('--cuda-graph', action='store_true', help='replay the forward from a CUDA graph (launch-bound small workloads)')
    ap.add_argument('--profile-range', action='store_true', help='cudaProfilerStart/Stop around the resident timed steps (for ncu --profile-from-start off)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the output of the last timed step as DIR/<name>.npy (float32/float64, '
                                                          'at most 64 MB in all: a fixed, seeded sample of the points beyond that)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, wl, rank, world)
        return
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    run_ours(args, wl, rank, local_rank, world)


if __name__ == '__main__':
    main()
