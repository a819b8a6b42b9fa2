"""CPU-only checks: host logic, state_dict layout, C-ABI surface.  No kernel is launched here."""
import ctypes
import os
import re

import pytest
import torch

from helpers import MODEL_CASES, BIG_CASES, Z_CASES, load_case, state_keys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('name', MODEL_CASES + BIG_CASES + Z_CASES)
def test_state_dict_layout_matches_reference(name):
    """Same parameter names and shapes as the reference (SURVEY.md A.6): load_state_dict interchange."""
    from se3_transformer_pytorch_b200 import SE3Transformer
    _, cfg = load_case(name)
    model = SE3Transformer(**cfg['ctor'])
    mine = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert mine == state_keys(name)


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads on a GPU-less box and exports everything include/se3b200.h declares."""
    from se3_transformer_pytorch_b200 import build, ops
    path = build.build()
    handle = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, 'include', 'se3b200.h')).read()
    declared = set(re.findall(r'\b(se3_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations parsed'
    for sym in declared:
        assert hasattr(handle, sym), f'{sym} declared in se3b200.h but not exported'
    assert declared == set(ops.EXPORTED_SYMBOLS)
    assert ops.lib().se3_abi_version() == 1


def test_build_stamp_survives_a_move_of_the_tree(tmp_path):
    """The GPU box runs a copy of the repository under another path and must load the library that was built here: the
    staleness digest may depend on file names and contents only (it once hashed absolute paths, so every box rebuilt and
    the ranks of a torchrun launch raced on the link step)."""
    import importlib.util
    import shutil
    import se3_transformer_pytorch_b200.build as B
    root = os.path.dirname(B.PKG)
    dst = tmp_path / 'moved'
    shutil.copytree(os.path.join(B.PKG, 'csrc'), dst / 'pkg' / 'csrc')
    shutil.copytree(os.path.join(root, 'include'), dst / 'include')
    shutil.copy(os.path.join(B.PKG, 'build.py'), dst / 'pkg' / 'build.py')
    spec = importlib.util.spec_from_file_location('moved_build', dst / 'pkg' / 'build.py')
    M = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(M)
    assert M.PKG != B.PKG and M._digest() == B._digest()
    B.build()
    assert B.is_current()                  # the in-tree library matches the sources


def test_constructor_assertions_match_reference():
    from se3_transformer_pytorch_b200 import SE3Transformer
    with pytest.raises(AssertionError):          # reference S:1048
        SE3Transformer(dim=8)
    with pytest.raises(AssertionError):          # reference S:1008
        SE3Transformer(dim=8, num_degrees=2, num_edge_tokens=4)
    with pytest.raises(AssertionError):          # reference S:1069
        SE3Transformer(dim=8, num_degrees=2, causal=True, attend_self=False)
    with pytest.raises(AssertionError):          # reference S:416
        SE3Transformer(dim=8, num_degrees=2, linear_proj_keys=True, tie_key_values=True)
    for flag in ('reversible', 'use_egnn', 'differentiable_coors'):
        with pytest.raises(NotImplementedError):
            SE3Transformer(dim=8, num_degrees=2, **{flag: True})


def test_no_cpu_fallback():
    """The product path must fail loudly without CUDA tensors."""
    from se3_transformer_pytorch_b200 import SE3Transformer
    model = SE3Transformer(dim=8, heads=2, dim_head=4, depth=1, num_degrees=2, num_neighbors=4)
    with pytest.raises(RuntimeError, match='CUDA'):
        model(torch.randn(1, 8, 8), torch.randn(1, 8, 3), torch.ones(1, 8).bool())


def test_forward_assertions_match_reference():
    from se3_transformer_pytorch_b200 import SE3Transformer
    model = SE3Transformer(dim=8, heads=2, dim_head=4, depth=1, num_degrees=2, num_neighbors=4, global_feats_dim=4)
    with pytest.raises(AssertionError):          # reference S:1136
        model(torch.randn(1, 8, 8), torch.randn(1, 8, 3))
    model = SE3Transformer(dim=8, heads=2, dim_head=4, depth=1, num_degrees=2, num_neighbors=4, attend_sparse_neighbors=True)
    with pytest.raises(AssertionError):          # reference S:1151
        model(torch.randn(1, 8, 8), torch.randn(1, 8, 3))


def test_basis_plan_shapes():
    from se3_transformer_pytorch_b200 import ops
    plan = ops.BasisPlan(3, 'cpu')
    assert len(plan.pairs) == 16 and plan.rows_per_edge == 1092      # SURVEY.md 8a row a5
    assert plan.col.numel() == 1132                                   # non-zeros of the 44 Q_J tables (SURVEY.md App. B)


def test_aligned_frames_reproduce_the_reference_basis():
    """Host math of the edge-aligned formulation (DESIGN.md 4.4), on CPU against the oracle: harmonics, Wigner matrices
    from rotated sample points, the (a, -b; b, a) structure of the basis on the axis, and the identity
    B(r) = D_lo B(a) D_li^T including coincident points (r = 0 -> the reference evaluates the basis on the axis)."""
    import numpy as np
    import torch
    from oracle import se3_oracle as O
    from se3_transformer_pytorch_b200 import aligned as AL
    torch.manual_seed(0)
    L = 3
    d = torch.randn(64, 3, dtype=torch.float64)
    d[0] = 0.0
    d[1] = torch.tensor([0.0, -2.0, 0.0])            # opposite to the axis
    d[2] = torch.tensor([0.0, 3.0, 0.0])
    unit = d / d.norm(dim=-1, keepdim=True).clamp(min=1e-300)
    Y = AL.real_sh64(unit[1:], 2 * L)
    Yo = O.real_spherical_harmonics(unit[1:].numpy(), 2 * L)
    assert max(float(np.abs(Y[l].numpy() - Yo[l]).max()) for l in range(2 * L + 1)) < 1e-12
    fr = AL.EdgeFrames(d.reshape(1, 1, -1, 3), L)
    Bo = O.get_basis(d.numpy(), L)
    Ba = O.get_basis(np.array([AL.AXIS]), L)
    for li in range(L + 1):
        for lo in range(L + 1):
            c0, ca, cb = AL.aligned_coeffs(li, lo)       # asserts the block structure internally
            ba = np.asarray(Ba[f'{li},{lo}'])[0]
            assert np.allclose(c0.numpy(), ba[lo, li, :], atol=1e-7)
            pred = np.einsum('epr,rsf,eqs->epqf', fr.D[lo].double().numpy(), ba, fr.D[li].double().numpy())
            ref = np.asarray(Bo[f'{li},{lo}'])
            assert np.abs(pred - ref).max() < 2e-6 * max(1.0, np.abs(ref).max()), (li, lo)


def test_lowrank_plan_image_selection(monkeypatch):
    """Host logic of ConvSE3.lowrank_plan on CPU (the CUDA packer is stubbed): distance-only radial trunks factor with rank
    <= 31, every pair of an all-eligible ConvSE3 gets edge-aligned images (one per |m|, F = 1 or 2 weight columns), a
    ConvSE3 with an ineligible pair keeps the global-frame images for the pairs it does cover."""
    import torch
    from se3_transformer_pytorch_b200 import ops, model as M
    calls = []

    def fake_pack(Fp, Co, Ci, F, Kp):
        assert Fp.shape == (Co * Ci * F, Kp) and Fp.dtype == torch.float32 and Fp.is_contiguous()
        calls.append((Co, Ci, F, Kp))
        return torch.zeros(1)

    monkeypatch.setattr(ops, 'pack_lowrank', fake_pack)
    monkeypatch.delenv('SE3B200_NO_ALIGNED', raising=False)
    torch.manual_seed(0)
    fin, fout = M.Fiber([(0, 32), (1, 32), (2, 32)]), M.Fiber([(0, 32), (1, 32), (2, 32)])
    monkeypatch.setattr(M.ConvSE3, 'tc_eligible', lambda self, di, do: True)
    conv = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)
    plan = conv.lowrank_plan(4.0)
    assert set(plan['pairs']) == set(conv.pairs)
    for (di, do), pp in plan['pairs'].items():
        assert pp['r'] <= 31 and pp['Kp'] in (16, 32)
        assert pp['img'] is None and pp['imgs_f'] is None and len(pp['al_imgs']) == 1 + min(di, do)
    assert sorted(c[2] for c in calls) == [1] * 9 + [2] * 5          # 9 pairs: one m = 0 image each; sum of min(di,do) = 5
    calls.clear()
    monkeypatch.setattr(M.ConvSE3, 'tc_eligible', lambda self, di, do: (di, do) != (2, 2))
    conv2 = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)
    plan2 = conv2.lowrank_plan(4.0)
    assert (2, 2) not in plan2['pairs'] and len(plan2['pairs']) == 8
    assert all(pp.get('al_imgs') is None and (pp['img'] is not None or pp['imgs_f'] is not None) for pp in plan2['pairs'].values())
    assert conv2.lowrank_plan(3.0) is plan2                          # cached while the distance range is covered


@pytest.mark.parametrize('frame', ['zgemm', 'aligned', 'global'])
def test_lowrank_conv_dispatch_on_cpu_emulation(monkeypatch, frame):
    """conv_forward's low-rank dispatch -- the one-GEMM production path (DESIGN.md 4.5: rotated gather, K segments per input
    degree and 16-column block of U, component planes, rotate-back), the R-first edge-aligned path (4.4) and the global frame
    with input-side contraction (4.2-4.3) (plan images, per-(l_in, m) tiles, (+m,-m) buffers, rotate-back, edge chunking)
    with every CUDA op replaced by a float64 torch emulation of its contract, against the reference order of operations
    (kernel = R . B first, S:336-343, with the oracle's basis).  Host logic only: the CUDA kernels have their own GPU tests."""
    import numpy as np
    import torch
    from oracle import se3_oracle as O
    from se3_transformer_pytorch_b200 import ops, model as M

    torch.manual_seed(0)
    b, n, k, C = 1, 40, 8, (128 if frame == 'zgemm' else 32)      # the one-GEMM kernel takes C_out % 128 == 0
    L = 2
    fin, fout = M.Fiber([(d, C) for d in range(L + 1)]), M.Fiber([(d, C) for d in range(L + 1)])
    if frame in ('aligned', 'zgemm'):
        monkeypatch.delenv('SE3B200_NO_ALIGNED', raising=False)
    else:
        monkeypatch.setenv('SE3B200_NO_ALIGNED', '1')
    monkeypatch.delenv('SE3B200_NO_ZGEMM', raising=False)
    monkeypatch.setenv('SE3B200_HOST_FRAMES', '1')               # float64 torch frames (the device kernel has its own GPU test)
    monkeypatch.setattr(M.ConvSE3, 'tc_eligible', lambda self, di, do: True)
    monkeypatch.setattr(ops, 'lowrank_enabled', lambda E: True)
    monkeypatch.setattr(torch.cuda, 'is_current_stream_capturing', lambda: False)
    monkeypatch.setattr(M, 'T_WORKSPACE_BYTES', ops.t_numel(1, C, 2, 2) * 4 if frame != 'zgemm' else 9 * C * ops.TILE_E * 4)  # one edge tile per chunk -> 3 chunks
    monkeypatch.setattr(ops, 'pack_lowrank', lambda Fp, Co, Ci, F, Kp: Fp.double().clone())  # "image" = F' itself

    conv = M.ConvSE3(fin, fout, edge_dim=0, pool=False, self_interaction=False)

    def radial_trunk(feat, params, num_pairs):
        return torch.stack([conv.kernel_unary[f'({di},{do})'].rp.trunk64(feat.double()) for di, do in conv.pairs]).float()

    def radial_trunk_u(feat, params, V, gmean, ones_col, stats, want_g=False):
        g = radial_trunk(feat, params, len(conv.pairs)).double()
        gc = g - gmean.double()[:, None, :]
        U = torch.bmm(gc, V.double())
        resid = (gc - torch.bmm(U, V.double().transpose(1, 2))).abs().amax(dim=(1, 2))
        stats[:, 0] = torch.maximum(stats[:, 0], resid.float())
        stats[:, 1] = torch.maximum(stats[:, 1], g.abs().amax(dim=(1, 2)).float())
        U[torch.arange(len(conv.pairs)), :, ones_col.long()] = 1.0
        return U.float(), (g.float() if want_g else None)

    def radial_table(dist, table, Dmax, ones_col, stats):
        # float64 restatement of se3_radial_table_fwd: 4-point Lagrange interpolation of the plan's U(d) table
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
        E = idx.numel()
        e0, e1 = tile_begin * ops.TILE_E, min(E, (tile_begin + tile_count) * ops.TILE_E)
        xj = gather_rows(x, idx, e0, e1)
        return xj if D is None else torch.einsum('eqn,eiq->ein', D[e0:e1].double(), xj)      # x'[n] = sum_q D[q,n] x[q]

    def edge_scale(feats, idx, max_degree):
        return torch.full((idx.numel(),), 4.0)

    def zgemm_image(parts, Co, mode):
        per_seg = (lambda Ci: 3 * (Ci // 4)) if mode == 3 else (lambda Ci: Ci * min(mode, 2) // 4)
        return [(Fp.double(), Ci) for Fp, Ci in parts], sum((Fp.shape[1] // 16) * per_seg(Ci) for Fp, Ci in parts)

    launched = []

    def zgemm(segs, w_img, sx, E, Co, mode, out, out_edge_stride, comp_off, flush_stages=0, alg_flops=0, tag=''):
        launched.append(tag)
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
        bb, nn, Ci, Q = x.shape
        E = idx.numel()
        e0, e1 = tile_begin * ops.TILE_E, min(E, (tile_begin + tile_count) * ops.TILE_E)
        xj = x.reshape(bb * nn, Ci, Q)[(idx + torch.arange(bb).view(-1, 1, 1) * nn).reshape(-1)][e0:e1].double()
        blk = blocks.reshape(E, P, Q, F)[e0:e1].double()
        return torch.einsum('epqf,eiq->eifp', blk, xj)                             # T[e,i,f,p]

    def gather_rows(x, idx, e0, e1):
        bb, nn, Ci, Q = x.shape
        return x.reshape(bb * nn, Ci, Q)[(idx + torch.arange(bb).view(-1, 1, 1) * nn).reshape(-1)][e0:e1].double()

    def tbuild(x, idx, basis_pair, d_in, d_out, tile_begin=0, tile_count=None, out=None):
        E = idx.numel()
        P, Q, F = 2 * d_out + 1, 2 * d_in + 1, 2 * min(d_in, d_out) + 1
        e0, e1 = tile_begin * ops.TILE_E, min(E, (tile_begin + tile_count) * ops.TILE_E)
        return torch.einsum('epqf,eiq->eifp', basis_pair.reshape(E, P, Q, F)[e0:e1].double(), gather_rows(x, idx, e0, e1))

    def gather_tiles(x, idx, tile_begin=0, tile_count=None, out=None):
        E = idx.numel()
        e0, e1 = tile_begin * ops.TILE_E, min(E, (tile_begin + tile_count) * ops.TILE_E)
        return gather_rows(x, idx, e0, e1).unsqueeze(2)                             # [e, i, f = 1, q]

    def fold_basis(S, basis_pair, E, Co, P, Q, F, out, accumulate, component_major=False, name='fold_basis'):
        res = torch.einsum('epqf,feqo->eop' if component_major else 'epqf,feoq->eop', basis_pair.reshape(E, P, Q, F).double(), S.double())
        out.copy_((out.double() + res if accumulate else res).float())

    def pairwise_lr(U, img, T, E, Co, Ci, F, P, Kp, out, accumulate, alg_P=None, out_strides=None, p_off=None, alg_units=None):
        assert out_strides is None and T.shape == (E, Ci, F, P) and out.shape[0] == E
        R = (U[:, :Kp].double() @ img.t()).reshape(E, Co, Ci, F)                    # bias rides on the ones column of U
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

    for name, fn in (('radial_trunk', radial_trunk), ('tbuild_blocks', tbuild_blocks), ('pairwise_lr', pairwise_lr),
                     ('rotate_back', rotate_back), ('tbuild', tbuild), ('gather_tiles', gather_tiles), ('fold_basis', fold_basis),
                     ('radial_trunk_u', radial_trunk_u), ('radial_table', radial_table), ('rotgather', rotgather), ('edge_scale', edge_scale), ('zgemm_image', zgemm_image),
                     ('zgemm', zgemm)):
        monkeypatch.setattr(ops, name, fn)

    coors = torch.randn(b, n, 3)
    idx = torch.stack([torch.randperm(n - 1)[:k] for _ in range(b * n)]).reshape(b, n, k)
    idx = idx + (idx >= torch.arange(n).view(1, n, 1)).long()                        # neighbours != self
    rel_pos = coors[0][:, None, :] - coors[0][idx[0]]                                # x_i - x_j   (S:1222)
    rel_pos = rel_pos.reshape(b, n, k, 3)
    rel_dist = rel_pos.norm(dim=-1)
    inp = {str(d): torch.randn(b, n, C, 2 * d + 1) for d in range(L + 1)}

    E = b * n * k
    Bo = O.get_basis(rel_pos.reshape(E, 3).double().numpy(), L)
    monkeypatch.setattr(ops, 'basis_pairs', lambda flat, plan, E_: {(di, do): torch.from_numpy(np.asarray(Bo[f'{di},{do}'])).reshape(-1)
                                                                     for di in range(L + 1) for do in range(L + 1)})
    basis = (torch.zeros(0), None, M.Geometry(rel_pos, L))
    nmask = torch.ones(b, n, k, dtype=torch.bool)
    with torch.no_grad():
        out = M.conv_forward([conv], inp, (idx, nmask, None), rel_dist, basis)[0]

    assert (len(launched) == 3 * (1 + 2 + 3)) == (frame == 'zgemm')       # 3 edge chunks x one launch per (degree_out, |m|)
    # reference order of operations in float64
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


def _run_bench(extra, env=None):
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ, **(env or {}))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--workload', 'cfg1', '--steps', '1',
                        '--warmup', '0', '--cpu-flops', '1e8'] + extra, capture_output=True, text=True, timeout=300, env=e, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith('{')]
    return [json.loads(ln) for ln in lines]


def test_reference_arm_prints_the_contract_line_on_cpu():
    """bench.py --impl reference: the oracle on the host cores, no GPU needed; one JSON line with the contract's keys."""
    (line,) = _run_bench([])
    assert line['impl'] == 'reference' and line['metric'] == 'point-clouds/sec fwd' and line['unit'] == 'clouds/s'
    assert line['higher_is_better'] is True and line['n_gpus'] == 1 and line['steps'] == 1 and line['gpu_launches'] == 0
    assert line['value'] > 0 and abs(line['e2e']['value'] - line['value']) < 1e-12
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    cb = line['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and 'ConvSE3' in cb['sample'] and cb['value'] == line['value']
    assert line['config']['workload'] == 'cfg1'


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs and prints the reference arm; the other ranks exit 0 without work."""
    assert _run_bench(['--gpus', '2'], env={'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'}) == []


def test_reference_arm_dumps_the_same_outputs_whatever_the_step_count(tmp_path):
    """--dump-outputs writes the last timed step's output as float .npy files; the inputs come from fixed seeds, so runs with
    other step counts write the same arrays."""
    import numpy as np
    dumps = []
    for steps in (1, 2):
        (line,) = _run_bench(['--steps', str(steps), '--dump-outputs', str(tmp_path / str(steps))])
        assert line['steps'] == steps
        dumps.append({f: np.load(tmp_path / str(steps) / f) for f in sorted(os.listdir(tmp_path / str(steps)))})
    assert sorted(dumps[0]) == ['type0.npy', 'type1.npy']
    for f, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all() and np.abs(a).max() > 0
        np.testing.assert_allclose(dumps[1][f], a, rtol=1e-5, atol=0)


def test_bench_rejects_zero_steps():
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and '--steps' in r.stderr


def test_dump_outputs_samples_the_same_points_within_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 64 << 10)
    rng = np.random.default_rng(1)
    arrays = {'type0': rng.random((4, 1024, 8, 1)), 'type1': rng.random((4, 1024, 8, 3)).astype(np.float16)}
    for d in ('a', 'b'):
        bench.dump_outputs(arrays, str(tmp_path / d))
    got = {f: np.load(tmp_path / 'a' / f) for f in ('type0.npy', 'type1.npy')}
    assert got['type0.npy'].dtype == np.float64 and got['type1.npy'].dtype == np.float32
    assert sum(a.nbytes for a in got.values()) <= 64 << 10
    rows0 = got['type0.npy'].reshape(len(got['type0.npy']), -1)
    all0 = arrays['type0'].reshape(4096, -1)
    assert len(rows0) > 1 and all(any((r == all0).all(1)) for r in rows0)       # whole rows of the output, not mixtures
    for f, a in got.items():
        assert np.array_equal(np.load(tmp_path / 'b' / f), a)


def test_concurrent_builds_do_not_race(tmp_path):
    """One process per GPU: every rank may find the library missing at the same moment.  Three processes build a moved copy of
    the sources at once; the file lock lets one of them compile, the others wait and load the finished library (a rank once
    dlopen'ed a half-linked file: 'invalid ELF header')."""
    import shutil
    import subprocess
    import sys
    import se3_transformer_pytorch_b200.build as B
    root = os.path.dirname(B.PKG)
    dst = tmp_path / 'moved'
    shutil.copytree(os.path.join(B.PKG, 'csrc'), dst / 'pkg' / 'csrc')
    shutil.copytree(os.path.join(root, 'include'), dst / 'include')
    shutil.copy(os.path.join(B.PKG, 'build.py'), dst / 'pkg' / 'build.py')
    code = ('import importlib.util, ctypes, sys\n'
            f'spec = importlib.util.spec_from_file_location("moved_build", r"{dst / "pkg" / "build.py"}")\n'
            'M = importlib.util.module_from_spec(spec); spec.loader.exec_module(M)\n'
            'h = ctypes.CDLL(M.build()); assert h.se3_abi_version() > 0; print("loaded")\n')
    procs = [subprocess.Popen([sys.executable, '-c', code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for _ in range(3)]
    outs = [p.communicate(timeout=900) for p in procs]
    for p, (out, err) in zip(procs, outs):
        assert p.returncode == 0 and 'loaded' in out, err[-2000:]
    assert not [f for f in os.listdir(dst / 'pkg') if f.endswith('.tmp')]
