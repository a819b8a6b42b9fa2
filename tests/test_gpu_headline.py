"""Parity of the BENCHMARKED path at the BENCHMARKED shape (BASELINE.json configs[1] widths: dim 512, heads 8, dim_head 64,
num_degrees 4, k = 16, >= 16384 edges so that the production dispatch -- low-rank radial basis in edge-aligned frames --
is the one that runs), where the CPU reference cannot run in full (SURVEY.md 8d: ~79 h):

  * the oracle (numpy restatement of S:203-268, 450-519) evaluates the K / V projections and the attention output of the
    first attention block at FULL width on the edges of a few sampled query nodes, from the same weights and the same
    block input; the GPU's K, V and attention output on those edges / nodes must agree within 1e-4 relative (north_star);
  * the whole model must agree with its own fp32 SIMT path (no tensor cores, no low-rank plan, no aligned frames).
"""
import os

import numpy as np
import pytest
import torch

from helpers import rel_err
from oracle import se3_oracle as O

pytestmark = pytest.mark.gpu
DEV = 'cuda'
TOL = 1e-4


def _state_np(module, prefix):
    return {prefix + k: v.detach().cpu().numpy() for k, v in module.state_dict().items()}


def _capture_attention(model, feats, coors, mask):
    """Run the model, recording what the first attention block saw and produced (block input after prenorm, graph, K, V,
    attention output before to_out) and the kernel kinds launched."""
    from se3_transformer_pytorch_b200 import model as M, ops
    rec = {}
    attn = model.net.blocks[0][0].attn
    orig_conv, orig_attn_op, orig_knn = M.conv_forward, ops.attention, ops.knn

    def conv_spy(convs, inp, edge_info, rel_dist, basis, **kw):
        outs = orig_conv(convs, inp, edge_info, rel_dist, basis, **kw)
        if len(convs) == 2 and convs[0] is attn.to_k and 'k' not in rec:
            rec['inp'] = {d: t.clone() for d, t in inp.items()}
            # degrees >= 1 stay in the edge-aligned frame for the attention kernel (AlignedKV): to_global() is the same rotate-back
            rec['fused_rotate'] = any(isinstance(t, M.AlignedKV) for t in outs[0].values())
            rec['k'] = {d: basis[2].to_global(t).clone() for d, t in outs[0].items()}
            rec['v'] = {d: basis[2].to_global(t).clone() for d, t in outs[1].items()}
        return outs

    def attn_spy(q, k, v, **kw):
        out = orig_attn_op(q, k, v, **kw)
        if 'k' in rec and len(rec.setdefault('attn_out', {})) < len(rec['k']):
            rec['attn_out'][str((q.shape[-1] - 1) // 2)] = out.clone()
        return out

    def knn_spy(*a, **kw):
        res = orig_knn(*a, **kw)
        rec['graph'] = res
        return res

    M.conv_forward, ops.attention, ops.knn = conv_spy, attn_spy, knn_spy
    ops.PROFILE = []
    try:
        out = model(feats, coors, mask)
        torch.cuda.synchronize()
    finally:
        M.conv_forward, ops.attention, ops.knn = orig_conv, orig_attn_op, orig_knn
        prof, ops.PROFILE = ops.PROFILE, None
    rec['kinds'] = [p[0] for p in prof]
    return out, rec


def _oracle_block(rec, P_attn, nodes, nd, dim, heads, dim_head):
    """Oracle K, V, attention output (before to_out) of the sampled query nodes from the recorded block input."""
    idx, nmask, rel_pos, rel_dist = (t.cpu().numpy() for t in rec['graph'])
    graph = O.subgraph(dict(idx=idx, mask=nmask, rel_pos=rel_pos, rel_dist=rel_dist, edges=None), nodes)
    basis = O.get_basis(graph['rel_pos'], nd - 1)
    inp = {d: t.cpu().numpy() for d, t in rec['inp'].items()}
    fiber = [(d, dim) for d in range(nd)]
    kv_fiber = [(d, heads * dim_head) for d in range(nd)]
    kw = dict(pool=False, self_interaction=False, edge_chunk=64)
    K = O.conv_se3(inp, graph, basis, P_attn, 'to_k.', fiber, kv_fiber, **kw)
    V = O.conv_se3(inp, graph, basis, P_attn, 'to_v.', fiber, kv_fiber, **kw)
    P_no_out = {k: v for k, v in P_attn.items() if not k.startswith('to_out.')}
    # attention_se3 recomputes K / V internally; feed it the ones above instead (same code, half the CPU time)
    orig = O.conv_se3
    O.conv_se3 = lambda feats, g, b, P, prefix, *a, **k: K if prefix == 'to_k.' else V
    try:
        A = O.attention_se3(inp, graph, basis, P_no_out, '', fiber, heads=heads, dim_head=dim_head, attend_self=True, nodes=nodes)
    finally:
        O.conv_se3 = orig
    return K, V, A


@pytest.mark.parametrize('k_nbr,n', [(16, 1024), (32, 2048)])
def test_production_path_matches_oracle_at_headline_width(k_nbr, n):
    """cfg2 shape (N = 1024, k = 16: E = 16384 per cloud) and cfg5 shape (N = 2048, k = 32: E = 65536), one cloud, depth 1."""
    from se3_transformer_pytorch_b200 import SE3Transformer, ops
    if not ops.tc_supported(DEV, 512, 7):
        pytest.skip('needs sm_100')
    nd, dim, heads, dim_head = 4, 512, 8, 64
    torch.manual_seed(0)
    with torch.device(DEV):
        model = SE3Transformer(dim=dim, heads=heads, dim_head=dim_head, depth=1, num_degrees=nd, num_neighbors=k_nbr).eval()
    attn = model.net.blocks[0][0].attn
    P_attn = _state_np(attn, '')                                 # fp32 masters of this block -> host (12 GB), before they are released
    g = torch.Generator().manual_seed(3)
    feats = torch.randn(1, n, dim, generator=g).to(DEV)
    coors = torch.randn(1, n, 3, generator=g).to(DEV)
    mask = torch.ones(1, n, dtype=torch.bool, device=DEV)
    assert ops.lowrank_enabled(n * k_nbr)
    # the bench's configuration: images packed up front, fp32 masters of net.6 released
    model.pack_weights(free_master=True, max_distance=16.0)
    out, rec = _capture_attention(model, feats, coors, mask)
    kinds = set(rec['kinds'])
    assert kinds & {'zgemm', 'pairwise_lr'}, kinds               # the low-rank tensor-core kernel ran ...
    assert rec['fused_rotate'] and 'rotgather' in kinds, kinds   # ... in edge-aligned frames, rotate-back fused into attention
    assert 'pairwise_tc' not in kinds and 'pairwise_simt' not in kinds, kinds
    rng = np.random.default_rng(0)
    nodes = np.sort(rng.choice(n, size=256 // k_nbr, replace=False))     # 256 edges at full width
    K, V, A = _oracle_block(rec, P_attn, nodes, nd, dim, heads, dim_head)
    for d in map(str, range(nd)):
        for name, ref, got in (('K', K, rec['k']), ('V', V, rec['v']), ('attention', A, rec['attn_out'])):
            err = rel_err(got[d][:, nodes].cpu().numpy(), ref[d])
            assert err < TOL, f'{name} degree {d}: rel err {err:.3e} vs oracle on {256} sampled edges'


def test_production_path_matches_simt_whole_model():
    """Whole model at cfg2 widths, depth 1, E = 16384: production dispatch vs the fp32 SIMT kernels on the same weights."""
    from se3_transformer_pytorch_b200 import SE3Transformer, ops
    if not ops.tc_supported(DEV, 512, 7):
        pytest.skip('needs sm_100')
    torch.manual_seed(1)
    with torch.device(DEV):
        model = SE3Transformer(dim=512, heads=8, dim_head=64, depth=1, num_degrees=4, output_degrees=2, num_neighbors=16).eval()
    g = torch.Generator().manual_seed(4)
    n = 1024
    feats = torch.randn(1, n, 512, generator=g).to(DEV)
    coors = torch.randn(1, n, 3, generator=g).to(DEV)
    mask = torch.ones(1, n, dtype=torch.bool, device=DEV)
    ops.PROFILE = []
    try:
        out = model(feats, coors, mask)
    finally:
        prof, ops.PROFILE = ops.PROFILE, None
    kinds = {p[0] for p in prof}
    assert kinds & {'zgemm', 'pairwise_lr'} and 'rotgather' in kinds, kinds
    os.environ['SE3B200_FORCE_SIMT'] = '1'
    try:
        for m in model.conv_modules():
            m._packed = None
        ref = model(feats, coors, mask)
    finally:
        del os.environ['SE3B200_FORCE_SIMT']
    for d in ('0', '1'):
        err = rel_err(out[d].cpu().numpy(), ref[d].cpu().numpy())
        assert err < TOL, f'degree {d}: {err:.3e}'
    # the production path captures in a CUDA graph (no host synchronisation inside the forward; the plan's run-time check is a
    # device-side flag read after the replay): replay == eager, bit for bit, also for new inputs of the same shape
    for m in model.conv_modules():
        m._packed = None
    eager = model(feats, coors, mask)
    graphed = model.graphed(feats, coors, mask)
    rep = graphed(feats, coors, mask)
    assert all(torch.equal(rep[d], eager[d]) for d in eager)
    feats2, coors2 = feats.flip(1).contiguous(), coors.flip(1).contiguous()
    rep2 = {d: t.clone() for d, t in graphed(feats2, coors2, mask).items()}
    eager2 = model(feats2, coors2, mask)
    assert all(torch.equal(rep2[d], eager2[d]) for d in eager2)


@pytest.mark.parametrize('radial', ['mlp', 'table'])
def test_plan_guard_bounds_the_output_error(radial, monkeypatch):
    """(radial = 'mlp': per-edge radial MLP + residual guard, SE3B200_NO_UTABLE=1; 'table': the default, radial coordinates
    interpolated from the plan's table, whose guard is the tabulated distance range.)
    The run-time guard of the low-rank plan is on the radial trunk outputs (max |g - gmean - U V^T| <= 1e-5 max |g| on the edges
    of the forward), the contract on the outputs (1e-4).  Drive a model with released masters (plan built for distances <= 2) with
    growing point clouds until the guard rejects the input: every ACCEPTED forward -- including the ones whose residual sits just
    below the guard -- must match the direct K = 128 kernels of an identical model within 1e-4, and the first rejected one must
    raise LowRankPlanMiss instead of returning a degraded result.  The (residual, output error) pairs are recorded."""
    import json
    from se3_transformer_pytorch_b200 import SE3Transformer, ops, model as M
    if not ops.tc_supported(DEV, 128, 1):
        pytest.skip('needs sm_100')
    if radial == 'mlp':
        monkeypatch.setenv('SE3B200_NO_UTABLE', '1')
    ctor = dict(dim=128, heads=2, dim_head=64, depth=1, num_degrees=3, output_degrees=2, num_neighbors=8)
    torch.manual_seed(5)
    with torch.device(DEV):
        direct = SE3Transformer(**ctor).eval()
    torch.manual_seed(5)
    with torch.device(DEV):
        planned = SE3Transformer(**ctor).eval()
    os.environ['SE3B200_LOWRANK_MIN_EDGES'] = '0'
    try:
        planned.pack_weights(free_master=True, max_distance=2.0)
    finally:
        del os.environ['SE3B200_LOWRANK_MIN_EDGES']
    g = torch.Generator().manual_seed(9)
    n = 96
    feats = torch.randn(1, n, 128, generator=g).to(DEV)
    base = torch.randn(1, n, 3, generator=g).to(DEV) * 0.25
    mask = torch.ones(1, n, dtype=torch.bool, device=DEV)
    rows, accepted, rejected = [], 0, 0
    for scale in (1.0, 2.0, 3.0, 4.0, 4.2, 4.4, 4.5, 4.6, 4.7, 4.8, 4.9, 5.0, 6.0, 10.0, 40.0):
        coors = base * scale
        os.environ['SE3B200_NO_LOWRANK'] = '1'
        try:
            ref = direct(feats, coors, mask)
        finally:
            del os.environ['SE3B200_NO_LOWRANK']
        try:
            out = planned(feats, coors, mask)
        except M.LowRankPlanMiss:
            rejected += 1
            rows.append(dict(scale=scale, residual=M.LAST_PLAN_RESIDUAL, accepted=False))
            continue
        accepted += 1
        err = max(rel_err(out[d].cpu().numpy(), ref[d].cpu().numpy()) for d in ('0', '1'))
        rows.append(dict(scale=scale, residual=M.LAST_PLAN_RESIDUAL, accepted=True, output_rel_err=err))
        assert M.LAST_PLAN_RESIDUAL <= M.ConvSE3.LR_RUNTIME_TOL
        assert err < TOL, f'scale {scale}: residual {M.LAST_PLAN_RESIDUAL:.2e} was accepted but the output is off by {err:.2e}'
    os.makedirs('gpurun_out', exist_ok=True)
    with open(f'gpurun_out/plan_guard_{radial}.jsonl', 'w') as f:
        for r in rows:
            f.write(json.dumps(r) + '\n')
    print(rows)
    assert accepted >= 2, rows          # (whether some scale is rejected depends on the weights; rejected ones never return a result)


def test_bench_dumps_the_same_outputs_whatever_the_step_count(tmp_path):
    """bench.py --dump-outputs on the GPU arm: the last timed forward's output, float32, the same for every run of a workload
    (seeded weights and inputs) whatever --steps is."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for steps in (1, 3):
        r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--workload', 'cfg1', '--steps', str(steps), '--warmup', '1',
                            '--no-cpu-baseline', '--dump-outputs', str(tmp_path / str(steps))], capture_output=True, text=True,
                           timeout=600, cwd=root)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])
        assert line['steps'] == steps
        dumps.append(np.load(tmp_path / str(steps) / 'out.npy'))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (1, 32, 64) and np.isfinite(dumps[0]).all()
    assert rel_err(dumps[1], dumps[0]) < 1e-6
