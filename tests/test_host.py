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
