"""CPU checks of ConvSE3's kernel routes: every CUDA op that conv_forward can reach is replaced by a float64 torch emulation of
its contract (include/se3b200.h), so the host logic -- route choice, plan images, edge chunking, launch order -- runs without a
device.  The kernels themselves have their own GPU tests."""
import json
import os

import numpy as np
import pytest
import torch

TRACES = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'conv_route_traces.json')


def _gather_rows(x, idx, e0, e1):
    bb, nn, Ci, Q = x.shape
    return x.reshape(bb * nn, Ci, Q)[(idx + torch.arange(bb).view(-1, 1, 1) * nn).reshape(-1)][e0:e1].double()


def _edge_range(idx, tile_begin, tile_count):
    from se3_transformer_pytorch_b200 import ops
    E = idx.numel()
    if tile_count is None:
        tile_count = (E + ops.TILE_E - 1) // ops.TILE_E - tile_begin
    return tile_begin * ops.TILE_E, min(E, (tile_begin + tile_count) * ops.TILE_E)


def emulated_ops():
    """{ops name: float64 emulation}."""
    from se3_transformer_pytorch_b200 import ops
    import torch.nn.functional as F

    def radial_trunk(feat, params, num_pairs):
        # params rows: net.0 W^T | b | LayerNorm w | b | net.3 W^T | b | LayerNorm w | b (RadialFunc.trunk_params)
        M = ops.RADIAL_MID
        feat = feat.double()
        in_dim = feat.shape[1]
        out = []
        for p in params.double():
            sizes = [in_dim * M, M, M, M, M * M, M, M, M]
            w0, b0, l1w, l1b, w3, b3, l4w, l4b = torch.split(p, sizes)
            h = F.gelu(F.layer_norm(feat @ w0.view(in_dim, M) + b0, (M,), l1w, l1b))
            out.append(F.gelu(F.layer_norm(h @ w3.view(M, M) + b3, (M,), l4w, l4b)))
        return torch.stack(out).float()

    def radial_trunk_u(feat, params, V, gmean, ones_col, stats, want_g=False):
        g = radial_trunk(feat, params, params.shape[0]).double()
        gc = g - gmean.double()[:, None, :]
        U = torch.bmm(gc, V.double())
        resid = (gc - torch.bmm(U, V.double().transpose(1, 2))).abs().amax(dim=(1, 2))
        stats[:, 0] = torch.maximum(stats[:, 0], resid.float())
        stats[:, 1] = torch.maximum(stats[:, 1], g.abs().amax(dim=(1, 2)).float())
        U[torch.arange(params.shape[0]), :, ones_col.long()] = 1.0
        return U.float(), (g.float() if want_g else None)

    def radial_table(dist, table, Dmax, ones_col, stats):
        # 4-point Lagrange interpolation of the plan's U(d) table (se3_radial_table_fwd)
        d = dist.reshape(-1).double()
        assert float(d.max()) <= Dmax
        Gn, KT = table.shape[1], table.shape[2]
        t = d * (Gn - 1) / Dmax
        i0 = t.floor().long().clamp(1, Gn - 3)
        f = (t - i0).unsqueeze(-1)
        w = (-f * (f - 1) * (f - 2) / 6, (f + 1) * (f - 1) * (f - 2) / 2, -(f + 1) * f * (f - 2) / 2, (f + 1) * f * (f - 1) / 6)
        U = torch.zeros(table.shape[0], d.numel(), 64, dtype=torch.float64)
        U[:, :, :KT] = sum(w[j] * table.double()[:, i0 - 1 + j] for j in range(4))
        U[torch.arange(table.shape[0]), :, ones_col.long()] = 1.0
        return U.float()

    def rotgather(x, idx, D, tile_begin=0, tile_count=None, out=None):
        e0, e1 = _edge_range(idx, tile_begin, tile_count)
        xj = _gather_rows(x, idx, e0, e1)
        return xj if D is None else torch.einsum('eqn,eiq->ein', D[e0:e1].double(), xj)      # x'[n] = sum_q D[q,n] x[q]

    def edge_scale(feats, idx, max_degree):
        return torch.full((idx.numel(),), 4.0)

    def zgemm_image(parts, Co, mode):
        per_seg = (lambda Ci: 3 * (Ci // 4)) if mode == 3 else (lambda Ci: Ci * min(mode, 2) // 4)
        return [(Fp.double(), Ci) for Fp, Ci in parts], sum((Fp.shape[1] // 16) * per_seg(Ci) for Fp, Ci in parts)

    def zgemm(segs, w_img, sx, E, Co, mode, out, out_edge_stride, comp_off, flush_stages=0, alg_flops=0, tag=''):
        mode = min(mode, 2)                                    # mode 3 = mode 2 evaluated with three products per complex one
        assert out_edge_stride == out.shape[1] * out.shape[2] and sx.shape == (E,)
        planes = out.view(E, -1, Co)                           # component-major rows: plane index = comp_off / Co
        res = [torch.zeros(E, Co, dtype=torch.float64) for _ in range(mode)]
        si = 0
        for Fp, Ci in w_img:
            Kp = Fp.shape[1]
            Fv = Fp.reshape(Co, Ci, mode, Kp)
            for kc in range(Kp // 16):
                U, X, Ci_s, ncomp, cplus, cminus = segs[si]
                si += 1
                assert Ci_s == Ci and X.shape == (E, Ci, ncomp) and U.shape[0] == E
                w = torch.einsum('ek,oifk->eoif', U[:, :16].double(), Fv[..., 16 * kc:16 * kc + 16])
                if mode == 1:
                    res[0] += torch.einsum('eoi,ei->eo', w[..., 0], X[:, :, cplus])
                else:
                    a, bb_ = w[..., 0], w[..., 1]
                    res[0] += torch.einsum('eoi,ei->eo', a, X[:, :, cplus]) - torch.einsum('eoi,ei->eo', bb_, X[:, :, cminus])
                    res[1] += torch.einsum('eoi,ei->eo', bb_, X[:, :, cplus]) + torch.einsum('eoi,ei->eo', a, X[:, :, cminus])
        assert si == len(segs)
        for c in range(mode):
            planes[:, comp_off[c] // Co, :] = res[c].float()

    def tbuild_blocks(x, idx, blocks, P, F, tile_begin=0, tile_count=None, out=None):
        E = idx.numel()
        e0, e1 = _edge_range(idx, tile_begin, tile_count)
        blk = blocks.reshape(E, P, x.shape[3], F)[e0:e1].double()
        return torch.einsum('epqf,eiq->eifp', blk, _gather_rows(x, idx, e0, e1))    # T[e,i,f,p]

    def tbuild(x, idx, basis_pair, d_in, d_out, tile_begin=0, tile_count=None, out=None):
        E = idx.numel()
        P, Q, F = 2 * d_out + 1, 2 * d_in + 1, 2 * min(d_in, d_out) + 1
        e0, e1 = _edge_range(idx, tile_begin, tile_count)
        return torch.einsum('epqf,eiq->eifp', basis_pair.reshape(E, P, Q, F)[e0:e1].double(), _gather_rows(x, idx, e0, e1))

    def gather_tiles(x, idx, tile_begin=0, tile_count=None, out=None):
        e0, e1 = _edge_range(idx, tile_begin, tile_count)
        return _gather_rows(x, idx, e0, e1).unsqueeze(2)                             # [e, i, f = 1, q]

    def fold_basis(S, basis_pair, E, Co, P, Q, F, out, accumulate, component_major=False, name='fold_basis'):
        res = torch.einsum('epqf,feqo->eop' if component_major else 'epqf,feoq->eop', basis_pair.reshape(E, P, Q, F).double(), S.double())
        out.copy_((out.double() + res if accumulate else res).float())

    def pack_lowrank(Fp, Co, Ci, F, Kp):
        assert Fp.shape == (Co * Ci * F, Kp) and Fp.dtype == torch.float32 and Fp.is_contiguous()
        return Fp.double().clone()                                                   # "image" = F' itself

    def pairwise_lr(U, img, T, E, Co, Ci, F, P, Kp, out, accumulate, alg_P=None, alg_units=None):
        assert T.shape == (E, Ci, F, P) and out.shape[0] == E
        R = (U[:, :Kp].double() @ img.t()).reshape(E, Co, Ci, F)                    # bias rides on the ones column of U
        res = torch.einsum('eoif,eifp->eop', R, T).reshape(out.shape)
        out.copy_((out.double() + res if accumulate else res).float())

    def pack_w3(W3, b3, Co, Ci, F):
        return torch.cat([W3.detach().double(), b3.detach().double()[:, None]], dim=1)   # "image" = [W3 | b3]

    def pairwise_tc(g, w_img, T, E, Co, Ci, F, P, out, accumulate):
        pairwise_simt(g, w_img[:, :-1], w_img[:, -1], T, E, Co, Ci, F, P, out, accumulate)

    def pairwise_simt(g, W3, b3, T, E, Co, Ci, F, P, out, accumulate):
        R = (g.double() @ W3.detach().double().t() + b3.detach().double()).reshape(E, Co, Ci, F)
        res = torch.einsum('eoif,eifp->eop', R, T).reshape(out.shape)
        out.copy_((out.double() + res if accumulate else res).float())

    def rotate_back(parts, D, E, Co, lo, out):
        P = 2 * lo + 1
        v = torch.zeros((E, Co, P), dtype=torch.float64)
        if parts[0] is not None:
            v[:, :, lo] = parts[0].reshape(E, Co).double()
        for m in range(1, lo + 1):
            if parts[m] is not None:
                v[:, :, lo + m], v[:, :, lo - m] = parts[m][:, :, 0].double(), parts[m][:, :, 1].double()
        out.copy_(torch.einsum('epn,eon->eop', D.reshape(E, P, P).double(), v).float())

    def masked_mean(x, mask):
        # x [nodes, K, ...], mask [nodes, K] or None: sum / clamp(count, 1), zero where nothing is left (utils.py:72-80)
        w = torch.ones(x.shape[:2], dtype=torch.float64) if mask is None else mask.double()
        cnt = w.sum(1)
        s = (x.double() * w.view(*w.shape, *([1] * (x.dim() - 2)))).sum(1)
        return torch.where(cnt.view(-1, *([1] * (s.dim() - 1))) > 0, s / cnt.clamp(min=1).view(-1, *([1] * (s.dim() - 1))), 0.0)

    def pool(x, mask):
        b, n, k = x.shape[:3]
        return masked_mean(x.reshape(b * n, k, *x.shape[3:]), None if mask is None else mask.reshape(b * n, k)).float().view(
            b, n, *x.shape[3:])

    def rotate_pool(Op, D, mask, self_add, nodes, K, Co, lo, out):
        v = Op.double().transpose(1, 2)                                             # [e, Co, P]
        if D is not None:
            v = torch.einsum('epn,eon->eop', D.double(), v)
        res = masked_mean(v.reshape(nodes, K, Co, 2 * lo + 1), None if mask is None else mask.reshape(nodes, K))
        out.copy_((res + (0 if self_add is None else self_add.double())).float())

    return dict(radial_trunk=radial_trunk, radial_trunk_u=radial_trunk_u, radial_table=radial_table, rotgather=rotgather,
                edge_scale=edge_scale, zgemm_image=zgemm_image, zgemm=zgemm, tbuild_blocks=tbuild_blocks, tbuild=tbuild,
                gather_tiles=gather_tiles, fold_basis=fold_basis, pack_lowrank=pack_lowrank, pairwise_lr=pairwise_lr, pack_w3=pack_w3,
                pairwise_tc=pairwise_tc, pairwise_simt=pairwise_simt, rotate_back=rotate_back, pool=pool, rotate_pool=rotate_pool)


def install(mp):
    """Install the emulation (and a CPU stand-in for the sm_100 checks) with a clean set of SE3B200_* switches.  Returns a
    function building seeded inputs (inp, edge_info, rel_dist, basis)."""
    from oracle import se3_oracle as O
    from se3_transformer_pytorch_b200 import ops, model as M
    for key in list(os.environ):
        if key.startswith('SE3B200_'):
            mp.delenv(key)
    mp.setenv('SE3B200_HOST_FRAMES', '1')                    # float64 torch frames (the device kernel has its own GPU test)
    mp.setenv('SE3B200_LOWRANK_MIN_EDGES', '0')
    mp.setattr(torch.cuda, 'get_device_capability', lambda device=None: (10, 0))
    mp.setattr(torch.cuda, 'is_current_stream_capturing', lambda: False)
    for name, fn in emulated_ops().items():
        mp.setattr(ops, name, fn)
    bases = {}
    mp.setattr(ops, 'basis_pairs', lambda flat, plan, E: bases[E])

    def make_inputs(b=1, n=40, k=8, L=2, C=32, geometry=True, seed=0):
        torch.manual_seed(seed)
        coors = torch.randn(b, n, 3)
        idx = torch.stack([torch.randperm(n - 1)[:k] for _ in range(b * n)]).reshape(b, n, k)
        idx = idx + (idx >= torch.arange(n).view(1, n, 1)).long()                    # neighbours != self
        rel_pos = (coors[:, :, None, :] - coors[torch.arange(b).view(b, 1, 1), idx]).reshape(b, n, k, 3)  # x_i - x_j (S:1222)
        rel_dist = rel_pos.norm(dim=-1)
        inp = {str(d): torch.randn(b, n, C, 2 * d + 1) for d in range(L + 1)}
        E = b * n * k
        Bo = O.get_basis(rel_pos.reshape(E, 3).double().numpy(), L)
        bases[E] = {(di, do): torch.from_numpy(np.asarray(Bo[f'{di},{do}'])).reshape(-1) for di in range(L + 1) for do in range(L + 1)}
        basis = (torch.zeros(0), None) + ((M.Geometry(rel_pos, L),) if geometry else ())
        nmask = torch.rand(b, n, k) > 0.2
        return inp, (idx, nmask, None), rel_dist, basis, Bo

    return make_inputs


@pytest.fixture
def make_inputs(monkeypatch):
    return install(monkeypatch)


def test_lowrank_plan_image_selection(make_inputs, monkeypatch):
    """Host logic of ConvSE3.lowrank_plan: distance-only radial trunks factor with rank <= 31, every pair of an all-eligible
    ConvSE3 gets edge-aligned images (one per |m|, F = 1 or 2 weight columns), a ConvSE3 with an ineligible pair keeps the
    global-frame images for the pairs it does cover."""
    from se3_transformer_pytorch_b200 import ops, model as M
    calls = []
    pack = ops.pack_lowrank

    def fake_pack(Fp, Co, Ci, F, Kp):
        calls.append((Co, Ci, F, Kp))
        return pack(Fp, Co, Ci, F, Kp)

    monkeypatch.setattr(ops, 'pack_lowrank', fake_pack)
    torch.manual_seed(0)
    fin, fout = M.Fiber([(0, 32), (1, 32), (2, 32)]), M.Fiber([(0, 32), (1, 32), (2, 32)])
    conv = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)
    plan = conv.lowrank_plan(4.0)
    assert set(plan['pairs']) == set(conv.pairs)
    for (di, do), pp in plan['pairs'].items():
        assert pp['r'] <= 31 and pp['Kp'] in (16, 32)
        assert pp.get('img') is None and pp.get('imgs_f') is None and len(pp['al_imgs']) == 1 + min(di, do)
    assert sorted(c[2] for c in calls) == [1] * 9 + [2] * 5          # 9 pairs: one m = 0 image each; sum of min(di,do) = 5
    calls.clear()
    conv2 = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)
    conv2.kernel_unary['(2,2)'].rp.net['6'].weight.data[0, 0] = 1e5          # outside the fp16 range: not tensor-core eligible
    plan2 = conv2.lowrank_plan(4.0)
    assert (2, 2) not in plan2['pairs'] and len(plan2['pairs']) == 8
    assert all(pp.get('al_imgs') is None and (pp.get('img') is not None or pp.get('imgs_f') is not None) for pp in plan2['pairs'].values())
    assert conv2.lowrank_plan(3.0) is plan2                          # cached while the distance range is covered


@pytest.mark.parametrize('frame', ['zgemm', 'aligned', 'global'])
def test_lowrank_conv_dispatch_on_cpu_emulation(make_inputs, monkeypatch, frame):
    """conv_forward's low-rank dispatch -- the one-GEMM production path (DESIGN.md 4.5: rotated gather, K segments per input
    degree and 16-column block of U, component planes, rotate-back), the R-first edge-aligned path (4.4) and the global frame
    with input-side contraction (4.2-4.3) (plan images, per-(l_in, m) tiles, (+m,-m) buffers, rotate-back, edge chunking)
    against the reference order of operations (kernel = R . B first, S:336-343, with the oracle's basis)."""
    from se3_transformer_pytorch_b200 import ops, model as M

    b, n, k, C = 1, 40, 8, (128 if frame == 'zgemm' else 32)      # the one-GEMM kernel takes C_out % 128 == 0
    L = 2
    fin, fout = M.Fiber([(d, C) for d in range(L + 1)]), M.Fiber([(d, C) for d in range(L + 1)])
    if frame == 'global':
        monkeypatch.setenv('SE3B200_NO_ALIGNED', '1')
    monkeypatch.setattr(M, 'T_WORKSPACE_BYTES', ops.t_numel(1, C, 2, 2) * 4 if frame != 'zgemm' else 9 * C * ops.TILE_E * 4)  # one edge tile per chunk -> 3 chunks
    launched = []
    zgemm = ops.zgemm
    monkeypatch.setattr(ops, 'zgemm', lambda *a, **kw: (launched.append(kw['tag']), zgemm(*a, **kw)))
    inp, (idx, _, _), rel_dist, basis, Bo = make_inputs(b, n, k, L, C)

    torch.manual_seed(0)
    conv = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)
    nmask = torch.ones(b, n, k, dtype=torch.bool)
    with torch.no_grad():
        out = M.conv_forward([conv], inp, (idx, nmask, None), rel_dist, basis)[0]

    assert (len(launched) == 3 * (1 + 2 + 3)) == (frame == 'zgemm')       # 3 edge chunks x one launch per (degree_out, |m|)
    # reference order of operations in float64
    E = b * n * k
    feat = rel_dist.reshape(E, 1).double()
    worst = 0.0
    for do in range(L + 1):
        ref = np.zeros((E, C, 2 * do + 1))
        for di in range(L + 1):
            pc = conv.kernel_unary[f'({di},{do})']
            lin = pc.rp.net['6']
            g = pc.rp.trunk64(feat)
            R = (g @ lin.weight.double().t() + lin.bias.double()).reshape(E, C, C, pc.num_freq).detach().numpy()
            xj = inp[str(di)].reshape(n, C, 2 * di + 1)[idx.reshape(-1)].double().numpy()
            ref += np.einsum('eoif,epqf,eiq->eop', R, np.asarray(Bo[f'{di},{do}']), xj)
        got = out[str(do)].reshape(E, C, 2 * do + 1).numpy()
        worst = max(worst, float(np.abs(got - ref).max() / np.abs(ref).max()))
    assert worst < 2e-5, worst


# ---- launch traces ----------------------------------------------------------------------------------------------------
def _encode(v):
    """Launch arguments as JSON: integers, flags and tags as they are, tensors by shape, None kept, anything else by type."""
    if v is None or isinstance(v, (bool, int, str)):
        return v
    if torch.is_tensor(v):
        return list(v.shape)
    if isinstance(v, (list, tuple)):
        return [_encode(x) for x in v]
    return type(v).__name__


def _fibers(C, L=2):
    from se3_transformer_pytorch_b200 import model as M
    return M.Fiber([(d, C) for d in range(L + 1)]), M.Fiber([(d, C) for d in range(L + 1)])


def _conv(C, seed=1, **kw):
    from se3_transformer_pytorch_b200 import model as M
    torch.manual_seed(seed)
    kw = dict(dict(pool=False, self_interaction=False), **kw)
    return M.ConvSE3(*_fibers(C), edge_dim=0, **kw)


def _forward(convs, args, keep_aligned=False):
    from se3_transformer_pytorch_b200 import model as M
    inp, edge_info, rel_dist, basis = args[:4]
    with torch.no_grad():
        return M.conv_forward(convs, inp, edge_info, rel_dist, basis, keep_aligned=keep_aligned)


def _case_zgemm(mk, mp):
    _forward([_conv(128)], mk(C=128))


def _case_zgemm_chunks(mk, mp):
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(128)], mk(C=128))


def _case_zgemm_no_utable(mk, mp):
    mp.setenv('SE3B200_NO_UTABLE', '1')
    _forward([_conv(128)], mk(C=128))


def _case_aligned_chunks(mk, mp):
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(32)], mk())


def _case_global_chunks(mk, mp):
    mp.setenv('SE3B200_NO_ALIGNED', '1')
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(32)], mk())


def _case_kv_keep_aligned(mk, mp):
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    outs = _forward([_conv(128, seed=1), _conv(128, seed=2)], mk(C=128), keep_aligned=True)
    assert all(type(t).__name__ == 'AlignedKV' for o in outs for d, t in o.items() if d != '0')


def _case_kv_split_routes(mk, mp):
    """to_k was blocked from its low-rank plan after a miss, to_v was not: the two take different routes in one call."""
    to_k, to_v = _conv(128, seed=1), _conv(128, seed=2)
    to_k._lr_blocked = True
    _forward([to_k, to_v], mk(C=128), keep_aligned=True)


def _case_kv_mixed_aligned_global(mk, mp):
    to_k, to_v = _conv(32, seed=1), _conv(32, seed=2)
    to_k.kernel_unary['(2,2)'].rp.net['6'].weight.data[0, 0] = 1e5           # one pair outside the fp16 range
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([to_k, to_v], mk())


def _case_pooled_self_zgemm(mk, mp):
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(128, pool=True, self_interaction=True)], mk(C=128))


def _case_pooled_self_zgemm_unfused(mk, mp):
    """Edge chunks that split neighbour lists (128 % 6 != 0): no fused pooling epilogue."""
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(128, pool=True, self_interaction=True)], mk(k=6, C=128))


def _case_pooled_self_aligned(mk, mp):
    _forward([_conv(32, pool=True, self_interaction=True)], mk())


def _case_pooled_self_direct(mk, mp):
    mp.setenv('SE3B200_NO_LOWRANK', '1')
    _forward([_conv(32, pool=True, self_interaction=True)], mk())


def _case_one_ineligible_pair(mk, mp):
    conv = _conv(32)
    conv.kernel_unary['(2,2)'].rp.net['6'].weight.data[0, 0] = 1e5
    _forward([conv], mk())


def _case_direct_tc(mk, mp):
    mp.setenv('SE3B200_NO_LOWRANK', '1')
    mp.setattr('se3_transformer_pytorch_b200.model.T_WORKSPACE_BYTES', 1)
    _forward([_conv(32)], mk())


def _case_direct_simt_no_geometry(mk, mp):
    mp.setenv('SE3B200_FORCE_SIMT', '1')
    _forward([_conv(32)], mk(geometry=False))


def _case_below_lowrank_min_edges(mk, mp):
    mp.setenv('SE3B200_LOWRANK_MIN_EDGES', '100000')
    _forward([_conv(32)], mk())


def _case_zgemm_plan_then_no_zgemm(mk, mp):
    conv, args = _conv(128), mk(C=128)
    _forward([conv], args)
    mp.setenv('SE3B200_NO_ZGEMM', '1')
    _forward([conv], args)


def _case_aligned_plan_then_no_aligned(mk, mp):
    conv, args = _conv(32), mk()
    _forward([conv], args)
    mp.setenv('SE3B200_NO_ALIGNED', '1')
    _forward([conv], args)


def _case_aligned_plan_without_geometry(mk, mp):
    with pytest.raises(RuntimeError, match='Geometry'):
        _forward([_conv(32)], mk(geometry=False))


def _case_free_master(mk, mp):
    conv, args = _conv(128), mk(C=128)
    conv.pack_weights(free_master=True, max_distance=float(args[2].max()) * 1.25)
    _forward([conv], args)


def _case_free_master_below_min_edges(mk, mp):
    conv, args = _conv(32), mk()
    conv.pack_weights(free_master=True, max_distance=float(args[2].max()) * 1.25)
    mp.setenv('SE3B200_LOWRANK_MIN_EDGES', '100000')
    _forward([conv], args)


def _case_capture_with_deferred_check(mk, mp):
    conv, args = _conv(128), mk(C=128)
    _forward([conv], args)                                      # the warm-up forward builds the plan
    mp.setattr(torch.cuda, 'is_current_stream_capturing', lambda: True)
    args[3][2].deferred = []
    _forward([conv], args)
    assert len(args[3][2].deferred) == 1


TRACE_CASES = {name[len('_case_'):]: fn for name, fn in globals().items() if name.startswith('_case_')}


def record_trace(case, mp):
    """Run one case with every emulated op wrapped in a recorder: [(op name, arguments)] in launch order."""
    from se3_transformer_pytorch_b200 import ops
    mk = install(mp)
    trace = []
    for name in emulated_ops():
        fn = getattr(ops, name)
        mp.setattr(ops, name, lambda *a, _n=name, _f=fn, **kw: (trace.append([_n, _encode(a), {k: _encode(v) for k, v in sorted(kw.items())}]),
                                                                _f(*a, **kw))[1])
    TRACE_CASES[case](mk, mp)
    return json.loads(json.dumps(trace))


@pytest.mark.parametrize('case', sorted(TRACE_CASES))
def test_conv_route_launch_trace(monkeypatch, case):
    """The ordered launches of conv_forward (and of the plan it builds) -- op, sizes, accumulate flags, tile ranges, tags --
    match the recorded trace of each route: one GEMM per (degree_out, |m|), the R-first edge-aligned kernels, the global-frame
    low-rank and direct kernels, and their mixtures."""
    with open(TRACES) as f:
        expected = json.load(f)[case]
    got = record_trace(case, monkeypatch)
    assert len(got) == len(expected)
    for i, (g, e) in enumerate(zip(got, expected)):
        assert g == e, f'launch {i}'
