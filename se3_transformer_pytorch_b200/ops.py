"""ctypes binding of libse3b200.so (C ABI in include/se3b200.h) for torch CUDA tensors.

PyTorch is plumbing here: it owns device memory and the current stream; every op below hands raw device pointers
and the stream handle to the hand-written sm_100a kernels.  There is NO CPU fallback: calling an op with a
non-CUDA tensor, or without the compiled library, raises.
"""
import ctypes
import os
import threading

import numpy as np
import torch

from . import build as _build

_PKG = os.path.dirname(os.path.abspath(__file__))
_lib = None
_lock = threading.Lock()

c_void_p, c_int, c_int64, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float

_SIGNATURES = {
    'se3_last_error': (ctypes.c_char_p, []),
    'se3_abi_version': (c_int, []),
    'se3_knn_fwd': (c_int, [c_void_p] * 4 + [c_int, c_int, c_int, c_float, c_int] + [c_void_p] * 4 + [c_void_p]),
    'se3_gather_pairs_fwd': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_basis_fwd': (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 5 + [c_int, c_void_p, c_void_p]),
    'se3_radial_trunk_fwd': (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'se3_tbuild_fwd': (c_int, [c_void_p] * 3 + [c_int] * 7 + [c_int64, c_int64, c_void_p, c_void_p]),
    'se3_pairwise_simt_fwd': (c_int, [c_void_p] * 4 + [c_int64] + [c_int] * 5 + [c_void_p, c_void_p]),
    'se3_w3_image_bytes': (c_int64, [c_int, c_int, c_int]),
    'se3_pack_w3': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_pairwise_tc_fwd': (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 5 + [c_void_p, c_void_p]),
    'se3_pairwise_tc_debug': (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 5 + [c_void_p, c_void_p, c_void_p]),
    'se3_lowrank_image_bytes': (c_int64, [c_int, c_int, c_int, c_int]),
    'se3_pack_lowrank': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_pairwise_lr_fwd': (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 6 + [c_void_p, c_void_p]),
    'se3_pairwise_lr_trace': (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 6 + [c_void_p, c_void_p, c_void_p]),
    'se3_fold_basis_fwd': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_fold_basis_cm_fwd': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_rotate_back_fwd': (c_int, [c_void_p] * 5 + [c_int64, c_int, c_int, c_void_p, c_void_p]),
    'se3_radial_trunk_u_fwd': (c_int, [c_void_p, c_int64, c_int, c_int] + [c_void_p] * 8),
    'se3_radial_table_fwd': (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    'se3_frames_fwd': (c_int, [c_void_p, c_int64, c_int] + [c_void_p] * 5),
    'se3_rotgather_fwd': (c_int, [c_void_p] * 3 + [c_int] * 5 + [c_int64, c_int64, c_void_p, c_void_p]),
    'se3_rotate_pool_fwd': (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_linear_tc_fwd': (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_pow2_scale_fwd': (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    'se3_rowabsmax_fwd': (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    'se3_edge_scale_fwd': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_zgemm_tile_n': (c_int, [c_int, c_int]),
    'se3_zgemm_image_bytes': (c_int64, [c_int, c_int, c_int]),
    'se3_zgemm_pack': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'se3_zgemm_fwd': (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    'se3_pool_fwd': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    'se3_norm_fwd': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_float, c_int, c_void_p, c_void_p]),
    'se3_attn_aligned_fwd': (c_int, [c_void_p] * 4 + [c_int] + [c_void_p] * 7 + [c_int, c_void_p] + [c_int] * 7 + [c_float, c_void_p, c_void_p]),
    'se3_attn_fwd': (c_int, [c_void_p] * 10 + [c_int, c_void_p] + [c_int] * 7 + [c_float, c_void_p, c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    """Load (building if the sources changed) libse3b200.so.  Raises if it cannot be built/loaded."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                path = _build.build()
                handle = ctypes.CDLL(path)
                for name, (res, args) in _SIGNATURES.items():
                    fn = getattr(handle, name)       # AttributeError if the symbol is missing -> loud failure
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


LAUNCHES = 0          # number of libse3b200 kernel launches issued by this process (bench.py reports it)
PROFILE = None        # when a list: every launch appends (kernel, start_event, end_event, reference-formulation FLOPs,
                      # algorithmic (unpadded) bytes, tag, issued tensor-core FLOPs (every pass counted), issued fp32 FMA FLOPs)


def _check(rc):
    global LAUNCHES
    if rc != 0:
        raise RuntimeError('libse3b200: ' + lib().se3_last_error().decode())
    LAUNCHES += 1


class _timed:
    """CUDA-event bracket on the launching stream around one kernel launch (only when PROFILE is enabled)."""

    def __init__(self, name, flops=0, nbytes=0, tag='', mma=0, fma=0):
        self.name, self.flops, self.nbytes, self.tag, self.mma, self.fma = name, flops, nbytes, tag, mma, fma

    def __enter__(self):
        if PROFILE is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None and exc[0] is None:
            self.end.record()
            PROFILE.append((self.name, self.start, self.end, self.flops, self.nbytes, self.tag, self.mma, self.fma))
        return False


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError('se3_transformer_pytorch_b200 runs on CUDA (sm_100a) only: got a tensor on %s; '
                               'there is no CPU path' % t.device)


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f32(t):
    if t.dtype != torch.float32:
        raise RuntimeError(f'se3_transformer_pytorch_b200 computes in float32 (got {t.dtype})')
    return t.contiguous()


def _u8(t):
    return None if t is None else t.contiguous().view(torch.uint8) if t.dtype == torch.bool else t.contiguous().to(torch.uint8)


# ---------------------------------------------------------------------------------------------------------
# K1
# ---------------------------------------------------------------------------------------------------------
def knn(coors, k, valid_radius, node_mask=None, neighbor_mask=None, sparse_adj=None, causal=False):
    """Neighbour graph (reference se3_transformer_pytorch.py:1171-1294).
    Returns idx int64 [b,n,k], mask bool [b,n,k], rel_pos [b,n,k,3], rel_dist [b,n,k]."""
    _require_cuda(coors, node_mask, neighbor_mask, sparse_adj)
    coors = _f32(coors)
    b, n, _ = coors.shape
    # the kernel indexes the masks as [b, n] / [b, n, n]: broadcastable inputs ([n, n], [1, n, n]) are expanded here, anything
    # else is refused instead of being read out of bounds
    if node_mask is not None:
        if node_mask.shape != (b, n):
            raise ValueError(f'knn: node_mask must be [b, n] = {(b, n)}, got {tuple(node_mask.shape)}')
    pair = []
    for name, t in (('neighbor_mask', neighbor_mask), ('sparse_adj', sparse_adj)):
        if t is not None:
            if t.dim() == 2:
                t = t.unsqueeze(0)
            if t.shape[-2:] != (n, n) or t.shape[0] not in (1, b):
                raise ValueError(f'knn: {name} must be [n, n], [1, n, n] or [b, n, n] with b, n = {(b, n)}, got {tuple(t.shape)}')
            t = t.expand(b, n, n)
        pair.append(t)
    neighbor_mask, sparse_adj = pair
    idx = torch.empty((b, n, k), dtype=torch.int64, device=coors.device)
    mask = torch.empty((b, n, k), dtype=torch.uint8, device=coors.device)
    rel_pos = torch.empty((b, n, k, 3), dtype=torch.float32, device=coors.device)
    rel_dist = torch.empty((b, n, k), dtype=torch.float32, device=coors.device)
    nm, nbm, sa = _u8(node_mask), _u8(neighbor_mask), _u8(sparse_adj)
    valid_radius = float(min(valid_radius, 3.0e38))
    nbytes = 12 * b * n + 25 * b * n * k + sum(t.numel() for t in (nm, nbm, sa) if t is not None)
    with torch.cuda.device(coors.device), _timed('knn', nbytes=nbytes):
        _check(lib().se3_knn_fwd(_p(coors), _p(nm), _p(nbm), _p(sa), b, n, k, valid_radius, int(bool(causal)),
                                 _p(idx), _p(mask), _p(rel_pos), _p(rel_dist), _stream()))
    return idx, mask.view(torch.bool), rel_pos, rel_dist


def gather_pairs(pair_feat, idx):
    """pair_feat [b,n,n,e] -> [b,n,k,e] (reference utils.py:56-70 at S:1293-1294)."""
    _require_cuda(pair_feat, idx)
    pair_feat = _f32(pair_feat)
    b, n, _, e = pair_feat.shape
    k = idx.shape[-1]
    out = torch.empty((b, n, k, e), dtype=torch.float32, device=pair_feat.device)
    with torch.cuda.device(pair_feat.device):
        _check(lib().se3_gather_pairs_fwd(_p(pair_feat), _p(idx.contiguous()), b, n, k, e, _p(out), _stream()))
    return out


# ---------------------------------------------------------------------------------------------------------
# K2
# ---------------------------------------------------------------------------------------------------------
_QJ = None


def qj_table(J, d_in, d_out):
    """Q_J tables (reference basis.py:123-138), shipped as data generated by the reference routine so that the sign
    convention matches trained reference weights (SURVEY.md finding 6)."""
    global _QJ
    if _QJ is None:
        _QJ = dict(np.load(os.path.join(_PKG, 'data', 'qj_tables.npz')))
    return _QJ[f'{J}_{d_in}_{d_out}']


MAX_DEGREE = 5


class BasisPlan:
    """CSR view of all Q_J tables for one max_degree + the per-pair output layout."""
    _cache = {}

    def __init__(self, max_degree, device):
        if max_degree > MAX_DEGREE:
            raise ValueError(f'max_degree {max_degree} > {MAX_DEGREE} (Q_J tables shipped up to degree {MAX_DEGREE})')
        self.max_degree = max_degree
        self.pairs = [(di, do) for di in range(max_degree + 1) for do in range(max_degree + 1)]
        row_ptr, col, val = [0], [], []
        pair_row0, pair_base = [0], []
        base = 0
        for di, do in self.pairs:
            P, Q, F = 2 * do + 1, 2 * di + 1, 2 * min(di, do) + 1
            tabs = [qj_table(abs(di - do) + f, di, do) for f in range(F)]
            for pq in range(P * Q):
                for f in range(F):
                    J = abs(di - do) + f
                    row = tabs[f][pq]
                    thr = 1e-6 * np.abs(tabs[f]).max()
                    for m in np.nonzero(np.abs(row) > thr)[0]:
                        col.append(J * J + int(m))
                        val.append(float(row[m]))
                    row_ptr.append(len(col))
            pair_base.append(base)
            base += P * Q * F
            pair_row0.append(pair_row0[-1] + P * Q * F)
        self.rows_per_edge = base
        self.pair_base = pair_base
        self.pair_rows = [pair_row0[i + 1] - pair_row0[i] for i in range(len(self.pairs))]
        mk = lambda a, dt: torch.tensor(a, dtype=dt, device=device)
        self.row_ptr, self.col, self.val = mk(row_ptr, torch.int32), mk(col, torch.int32), mk(val, torch.float32)
        self.pair_row0, self.pair_base_t = mk(pair_row0, torch.int32), mk(pair_base, torch.int32)

    @classmethod
    def get(cls, max_degree, device):
        key = (max_degree, str(device))
        if key not in cls._cache:
            cls._cache[key] = cls(max_degree, device)
        return cls._cache[key]


def basis_flat(rel_pos, max_degree):
    """rel_pos [..., 3] -> (flat fp32 buffer, plan); pair p lives at flat[base_p*E : (base_p+rows_p)*E] as [E, rows_p]."""
    _require_cuda(rel_pos)
    rel_pos = _f32(rel_pos)
    E = rel_pos.numel() // 3
    plan = BasisPlan.get(max_degree, rel_pos.device)
    out = torch.empty(plan.rows_per_edge * E, dtype=torch.float32, device=rel_pos.device)
    with torch.cuda.device(rel_pos.device), _timed('basis', nbytes=E * (12 + 4 * plan.rows_per_edge)):
        _check(lib().se3_basis_fwd(_p(rel_pos), E, max_degree, _p(plan.row_ptr), _p(plan.col), _p(plan.val),
                                   _p(plan.pair_row0), _p(plan.pair_base_t), len(plan.pairs), _p(out), _stream()))
    return out, plan


def get_basis(r_ij, max_degree, differentiable=False):
    """Drop-in for the reference get_basis (basis.py:153-205): {'di,do': [..., 1, 2do+1, 1, 2di+1, f]} (forward only)."""
    flat, plan = basis_flat(r_ij, max_degree)
    E = r_ij.numel() // 3
    lead = tuple(r_ij.shape[:-1])
    out = {}
    for (di, do), base, rows in zip(plan.pairs, plan.pair_base, plan.pair_rows):
        out[f'{di},{do}'] = flat[base * E:(base + rows) * E].view(*lead, 1, 2 * do + 1, 1, 2 * di + 1, 2 * min(di, do) + 1)
    return out


def basis_pairs(flat, plan, E):
    """{(di,do): [E, P, Q, F] view} on the flat buffer."""
    out = {}
    for (di, do), base, rows in zip(plan.pairs, plan.pair_base, plan.pair_rows):
        out[(di, do)] = flat[base * E:(base + rows) * E]
    return out


# ---------------------------------------------------------------------------------------------------------
# K3 / K4
# ---------------------------------------------------------------------------------------------------------
RADIAL_MID = 128
TILE_E, TILE_O, TILE_IF = 128, 32, 4


def trunk_param_stride(in_dim):
    return in_dim * RADIAL_MID + 3 * RADIAL_MID + RADIAL_MID * RADIAL_MID + 3 * RADIAL_MID


def radial_trunk(feat, params, num_pairs):
    """feat [E, in_dim], params [num_pairs, trunk_param_stride] -> g [pairs, E, 128] fp32."""
    _require_cuda(feat, params)
    feat = _f32(feat)
    E, in_dim = feat.shape
    g = torch.empty((num_pairs, E, RADIAL_MID), dtype=torch.float32, device=feat.device)
    with torch.cuda.device(feat.device), _timed('radial_trunk', flops=2 * E * num_pairs * RADIAL_MID * (in_dim + RADIAL_MID),
                                                 nbytes=4 * (feat.numel() + params.numel() + g.numel())):
        _check(lib().se3_radial_trunk_fwd(_p(feat), E, in_dim, num_pairs, _p(params), _p(g), _stream()))
    return g


def t_numel(num_tiles, Ci, F, P):
    nifb = (Ci * F + TILE_IF - 1) // TILE_IF
    ph = (P + 3) // 4
    return num_tiles * nifb * TILE_IF * ph * TILE_E * 4


def tbuild(x, idx, basis_pair, d_in, d_out, tile_begin=0, tile_count=None, out=None):
    """x [b,n,Ci,2di+1], idx [b,n,k], basis_pair flat [E*P*Q*F] -> T (tile layout, see include/se3b200.h)."""
    _require_cuda(x, idx, basis_pair)
    x = _f32(x)
    b, n, Ci, Q = x.shape
    k = idx.shape[-1]
    P, F = 2 * d_out + 1, 2 * min(d_in, d_out) + 1
    E = b * n * k
    n_tiles = (E + TILE_E - 1) // TILE_E
    if tile_count is None:
        tile_count = n_tiles - tile_begin
    numel = t_numel(tile_count, Ci, F, P)
    if out is None or out.numel() < numel:
        out = torch.empty(numel, dtype=torch.float32, device=x.device)
    Ec = min(E - tile_begin * TILE_E, tile_count * TILE_E)       # edges of this call; bytes WITHOUT the layout padding of T
    nbytes = 4 * Ec * (Ci * F * P + P * Q * F + Ci * Q) + 8 * Ec
    with torch.cuda.device(x.device), _timed('tbuild', flops=2 * Ec * Ci * F * P * Q, nbytes=nbytes):
        _check(lib().se3_tbuild_fwd(_p(x), _p(idx.contiguous()), _p(basis_pair), b, n, k, Ci, P, Q, F, tile_begin, tile_count,
                                    _p(out), _stream()))
    return out


_IDENTITY_BASIS = {}


def gather_tiles(x, idx, tile_begin=0, tile_count=None, out=None):
    """Neighbour features in the T tile layout: X[e,i,q] = x[b, idx[e], i, q] (se3_tbuild_fwd with an identity basis,
    P := Q, F := 1); the right-hand operand of the input-side contraction."""
    _require_cuda(x, idx)
    x = _f32(x)
    b, n, Ci, Q = x.shape
    k = idx.shape[-1]
    E = b * n * k
    key = (E, Q, x.device)
    if key not in _IDENTITY_BASIS:
        _IDENTITY_BASIS.clear()
        _IDENTITY_BASIS[key] = torch.eye(Q, dtype=torch.float32, device=x.device).repeat(E, 1, 1).reshape(-1).contiguous()
    eye = _IDENTITY_BASIS[key]
    n_tiles = (E + TILE_E - 1) // TILE_E
    if tile_count is None:
        tile_count = n_tiles - tile_begin
    numel = t_numel(tile_count, Ci, 1, Q)
    if out is None or out.numel() < numel:
        out = torch.empty(numel, dtype=torch.float32, device=x.device)
    Ec = min(E - tile_begin * TILE_E, tile_count * TILE_E)
    nbytes = 4 * Ec * (2 * Ci * Q) + 8 * Ec
    with torch.cuda.device(x.device), _timed('tbuild', flops=2 * Ec * Ci * Q * Q, nbytes=nbytes):
        _check(lib().se3_tbuild_fwd(_p(x), _p(idx.contiguous()), _p(eye), b, n, k, Ci, Q, Q, 1, tile_begin, tile_count, _p(out), _stream()))
    return out


def tbuild_blocks(x, idx, blocks, P, F, tile_begin=0, tile_count=None, out=None):
    """se3_tbuild_fwd with caller-supplied per-edge blocks [E,P,Q,F] (flat): T[e,i,f,p] = sum_q blocks[e,p,q,f] x[b, idx[e], i, q]."""
    _require_cuda(x, idx, blocks)
    x = _f32(x)
    b, n, Ci, Q = x.shape
    k = idx.shape[-1]
    E = b * n * k
    assert blocks.numel() == E * P * Q * F
    n_tiles = (E + TILE_E - 1) // TILE_E
    if tile_count is None:
        tile_count = n_tiles - tile_begin
    numel = t_numel(tile_count, Ci, F, P)
    if out is None or out.numel() < numel:
        out = torch.empty(numel, dtype=torch.float32, device=x.device)
    Ec = min(E - tile_begin * TILE_E, tile_count * TILE_E)
    nbytes = 4 * Ec * (Ci * F * P + P * Q * F + Ci * Q) + 8 * Ec
    with torch.cuda.device(x.device), _timed('tbuild', flops=2 * Ec * Ci * F * P * Q, nbytes=nbytes):
        _check(lib().se3_tbuild_fwd(_p(x), _p(idx.contiguous()), _p(blocks), b, n, k, Ci, P, Q, F, tile_begin, tile_count, _p(out), _stream()))
    return out


def fold_basis(S, basis_pair, E, Co, P, Q, F, out, accumulate, component_major=False, name='fold_basis'):
    """out [E,Co,P] (+)= sum_{f,q} basis_pair[e,p,q,f] S[f,e,o,q]; S [F,E,Co,Q] (or [F,E,Q,Co] if component_major),
    basis_pair the [E,P,Q,F] rows of these edges."""
    _require_cuda(S, basis_pair, out)
    assert S.is_contiguous() and basis_pair.is_contiguous() and out.is_contiguous()
    nbytes = 4 * (S.numel() + basis_pair.numel() + out.numel() * (2 if accumulate else 1))
    with torch.cuda.device(out.device), _timed(name, flops=2 * E * Co * P * Q * F, nbytes=nbytes):
        fn = lib().se3_fold_basis_cm_fwd if component_major else lib().se3_fold_basis_fwd
        _check(fn(_p(S), _p(basis_pair), E, Co, P, Q, F, int(accumulate), _p(out), _stream()))


def rotate_back(parts, D, E, Co, lo, out):
    """out [E,Co,2lo+1] = D_lo(e) out'(e): parts[0] [E,Co] (m = 0), parts[m] [E,Co,2] (components +m, -m) or None."""
    _require_cuda(D, out)
    ptrs = [(_p(t) if t is not None else None) for t in (list(parts) + [None] * 4)[:4]]
    P = 2 * lo + 1
    nbytes = 4 * (2 * E * Co * P + E * P * P)
    with torch.cuda.device(out.device), _timed('rotate_back', flops=2 * E * Co * P * P, nbytes=nbytes):
        _check(lib().se3_rotate_back_fwd(*ptrs, _p(D), E, Co, lo, _p(out), _stream()))


def pairwise_simt(g, W3, b3, T, E, Co, Ci, F, P, out, accumulate):
    _require_cuda(g, W3, b3, T, out)
    with torch.cuda.device(out.device), _timed('pairwise_simt', flops=2 * E * Co * Ci * F * (RADIAL_MID + P), fma=2 * E * Co * Ci * F * (RADIAL_MID + P)):
        _check(lib().se3_pairwise_simt_fwd(_p(g), _p(W3), _p(b3), _p(T), E, Co, Ci, F, P, int(accumulate), _p(out), _stream()))


def w3_image_bytes(Co, Ci, F):
    return lib().se3_w3_image_bytes(Co, Ci, F)


def pack_w3(W3, b3, Co, Ci, F):
    _require_cuda(W3, b3)
    nbytes = w3_image_bytes(Co, Ci, F)
    if nbytes < 0:
        raise RuntimeError(f'pack_w3: unsupported shape Co={Co} Ci={Ci} F={F}')
    img = torch.empty(nbytes, dtype=torch.uint8, device=W3.device)
    with torch.cuda.device(W3.device):
        _check(lib().se3_pack_w3(_p(_f32(W3)), _p(_f32(b3)), Co, Ci, F, _p(img), _stream()))
    return img


def pairwise_tc(g, w_img, T, E, Co, Ci, F, P, out, accumulate, dump=None):
    _require_cuda(g, w_img, T, out)
    # algorithmic work: the radial GEMM (2*128 per R element) + the contraction with T (2*P per R element)
    flops = 2 * E * Co * Ci * F * (RADIAL_MID + P)
    nbytes = w_img.numel() + 4 * E * Ci * F * P + 4 * E * Co * P * (2 if accumulate else 1)
    with torch.cuda.device(out.device), _timed('pairwise_tc', flops=flops, nbytes=nbytes, tag=f'P{P}F{F}Ci{Ci}Co{Co}',
                                               mma=2 * E * Co * Ci * F * 3 * RADIAL_MID, fma=2 * E * Co * Ci * F * P):
        if dump is None:
            _check(lib().se3_pairwise_tc_fwd(_p(g), _p(w_img), _p(T), E, Co, Ci, F, P, int(accumulate), _p(out), _stream()))
        else:
            _check(lib().se3_pairwise_tc_debug(_p(g), _p(w_img), _p(T), E, Co, Ci, F, P, int(accumulate), _p(out), _p(dump),
                                               _stream()))


def pack_lowrank(Fp, Co, Ci, F, Kp):
    """Fp [Co*Ci*F, Kp] fp32 (W3 V | b3 | 0) -> tensor-core operand image for pairwise_lr."""
    _require_cuda(Fp)
    nbytes = lib().se3_lowrank_image_bytes(Co, Ci, F, Kp)
    if nbytes < 0:
        raise RuntimeError(f'pack_lowrank: unsupported shape Co={Co} Ci={Ci} F={F}')
    img = torch.empty(nbytes, dtype=torch.uint8, device=Fp.device)
    with torch.cuda.device(Fp.device):
        _check(lib().se3_pack_lowrank(_p(_f32(Fp)), Co, Ci, F, Kp, _p(img), _stream()))
    return img


def pairwise_lr(U, w_img, T, E, Co, Ci, F, P, Kp, out, accumulate, alg_P=None, alg_units=None):
    """Low-rank radial path: U [E,64] fp32 (G V | 1 | 0), w_img from pack_lowrank."""
    _require_cuda(U, w_img, T, out)
    # algorithmic work of the reference formulation (SURVEY.md 8d): 2*128 (radial GEMM) + 2P (contraction) per R element;
    # executed work: the GEMM has K = Kp instead of 128
    # (alg_P: the launch is one frequency of an input-side contraction whose reference formulation has P = alg_P)
    # (alg_units: reference-formulation FLOPs per (edge, o, i) that this launch stands for, when it is not F*(2*128 + 2P))
    flops = 2 * E * Co * Ci * F * (RADIAL_MID + (alg_P if alg_P is not None else P))
    if alg_units is not None:
        flops = E * Co * Ci * alg_units
    # issued: 3 fp16 MMA passes of K = Kp per R element on the tensor cores, P fp32 FMAs per R element on the SIMT pipe
    nbytes = w_img.numel() + 4 * E * Ci * F * P + 4 * E * Co * P * (2 if accumulate else 1)
    tag = f'P{P}F{F}Ci{Ci}Co{Co}K{Kp}' + (f'(in-side of P{alg_P})' if alg_P is not None else '')
    with torch.cuda.device(out.device), _timed('pairwise_lr', flops=flops, nbytes=nbytes, tag=tag,
                                               mma=2 * E * Co * Ci * F * 3 * Kp, fma=2 * E * Co * Ci * F * P):
        _check(lib().se3_pairwise_lr_fwd(_p(U), _p(w_img), _p(T), E, Co, Ci, F, P, Kp, int(accumulate), _p(out), _stream()))


# ---------------------------------------------------------------------------------------------------------
# production path: low-rank radial basis + edge-aligned frames as one GEMM per (degree_out, |m|)  (csrc/zgemm.cu, aligned.cu)
# ---------------------------------------------------------------------------------------------------------
class ZSeg(ctypes.Structure):
    _fields_ = [('U', c_void_p), ('X', c_void_p), ('Ci', c_int), ('ncomp', c_int), ('cplus', c_int), ('cminus', c_int)]


def radial_trunk_u(feat, params, V, gmean, ones_col, stats, want_g=False):
    """Trunk + radial coordinates: feat [E,in_dim], params [pairs, stride], V [pairs,128,64] fp32, gmean [pairs,128] fp32 (centre of
    the pair's radial curve), ones_col [pairs] int32, stats [pairs,2] fp32 (accumulates (max residual, max |g|)) ->
    U [pairs,E,64] = ((g - gmean) V | 1 | 0) (, g [pairs,E,128])."""
    _require_cuda(feat, params, V, gmean, ones_col, stats)
    assert gmean.shape == (params.shape[0], RADIAL_MID) and gmean.is_contiguous() and gmean.dtype == torch.float32
    feat = _f32(feat)
    E, in_dim = feat.shape
    num_pairs = params.shape[0]
    assert V.shape == (num_pairs, RADIAL_MID, 64) and V.is_contiguous() and ones_col.dtype == torch.int32 and stats.is_contiguous()
    U = torch.empty((num_pairs, E, 64), dtype=torch.float32, device=feat.device)
    g = torch.empty((num_pairs, E, RADIAL_MID), dtype=torch.float32, device=feat.device) if want_g else None
    flops = 2 * E * num_pairs * RADIAL_MID * (in_dim + RADIAL_MID + 2 * 64)
    with torch.cuda.device(feat.device), _timed('radial_trunk', flops=flops, nbytes=4 * (feat.numel() + params.numel() + V.numel() + U.numel())):
        _check(lib().se3_radial_trunk_u_fwd(_p(feat), E, in_dim, num_pairs, _p(params), _p(V), _p(gmean), _p(ones_col), _p(g), _p(U), _p(stats), _stream()))
    return U, g


def radial_table(dist, table, Dmax, ones_col, stats):
    """Radial coordinates by table lookup: dist [E] fp32, table [pairs, G, KT] fp32 (U(d) on the uniform grid of [0, Dmax]),
    ones_col [pairs] int32, stats [pairs, 2] (out-of-range flag) -> U [pairs, E, 64]."""
    _require_cuda(dist, table, ones_col, stats)
    dist = _f32(dist).reshape(-1)
    E = dist.numel()
    num_pairs, G, KT = table.shape
    assert table.is_contiguous() and table.dtype == torch.float32 and ones_col.dtype == torch.int32
    U = torch.empty((num_pairs, E, 64), dtype=torch.float32, device=dist.device)
    with torch.cuda.device(dist.device), _timed('radial_table', flops=8 * E * num_pairs * KT, nbytes=4 * (E + U.numel() + 4 * E * num_pairs * KT)):
        _check(lib().se3_radial_table_fwd(_p(dist), E, _p(table), G, KT, float(Dmax), _p(ones_col), num_pairs, _p(U), _p(stats), _stream()))
    return U


_FRAME_TABLES = {}


def _frame_tables(lmax, device):
    key = (lmax, str(device))
    if key not in _FRAME_TABLES:
        from . import aligned
        xs_t, pin_t, keep = [None], [None], []
        ns = [0]
        for l in range(1, lmax + 1):
            xs, pin = aligned._samples(l, device)
            xs, pin = xs.contiguous(), pin.contiguous()
            keep += [xs, pin]
            xs_t.append(xs.data_ptr()); pin_t.append(pin.data_ptr()); ns.append(xs.shape[0])
        mk = lambda vals: (c_void_p * (lmax + 1))(*[c_void_p(v) if v else None for v in vals])
        _FRAME_TABLES[key] = (mk(xs_t), mk(pin_t), (c_int * (lmax + 1))(*ns), keep)
    return _FRAME_TABLES[key]


def frames(rel_pos, lmax):
    """Wigner matrices of the edge frames: rel_pos [...,3] -> [None, D_1 [E,3,3], ..., D_lmax] fp32 (float64 arithmetic inside)."""
    _require_cuda(rel_pos)
    rel_pos = _f32(rel_pos).reshape(-1, 3)
    E = rel_pos.shape[0]
    D = [None] + [torch.empty((E, 2 * l + 1, 2 * l + 1), dtype=torch.float32, device=rel_pos.device) for l in range(1, lmax + 1)]
    if lmax >= 1:
        xs, pin, ns, _ = _frame_tables(lmax, rel_pos.device)
        dptr = (c_void_p * (lmax + 1))(*[c_void_p(t.data_ptr()) if t is not None else None for t in D])
        with torch.cuda.device(rel_pos.device), _timed('frames', nbytes=E * (12 + 4 * sum((2 * l + 1) ** 2 for l in range(1, lmax + 1)))):
            _check(lib().se3_frames_fwd(_p(rel_pos), E, lmax, xs, pin, ns, dptr, _stream()))
    return D


def rotgather(x, idx, D, tile_begin=0, tile_count=None, out=None):
    """x [b,n,Ci,Q], idx [b,n,k], D [E,Q,Q] (None for Q = 1) -> X [tile_count, Ci, Q, 128]: rotated neighbour features."""
    _require_cuda(x, idx, D)
    x = _f32(x)
    b, n, Ci, Q = x.shape
    k = idx.shape[-1]
    E = b * n * k
    n_tiles = (E + TILE_E - 1) // TILE_E
    if tile_count is None:
        tile_count = n_tiles - tile_begin
    numel = tile_count * Ci * Q * TILE_E
    if out is None or out.numel() < numel:
        out = torch.empty(numel, dtype=torch.float32, device=x.device)
    Ec = min(E - tile_begin * TILE_E, tile_count * TILE_E)
    nbytes = 4 * Ec * (2 * Ci * Q + (Q * Q if Q > 1 else 0)) + 8 * Ec
    with torch.cuda.device(x.device), _timed('rotgather', flops=2 * Ec * Ci * Q * Q, nbytes=nbytes):
        _check(lib().se3_rotgather_fwd(_p(x), _p(idx.contiguous()), _p(D), b, n, k, Ci, Q, tile_begin, tile_count, _p(out), _stream()))
    return out


def rotate_pool(Op, D, mask, self_add, nodes, K, Co, lo, out):
    """Pooled ConvSE3 epilogue fused with the rotate-back: Op [nodes*K, 2lo+1, Co], D [nodes*K, P, P] or None (lo = 0),
    mask [nodes*K] bool or None, self_add [nodes, Co, P] or None -> out [nodes, Co, P]."""
    _require_cuda(Op, D, mask, self_add, out)
    P = 2 * lo + 1
    assert Op.is_contiguous() and out.is_contiguous() and (self_add is None or self_add.is_contiguous())
    nbytes = 4 * (Op.numel() + out.numel() * (2 if self_add is not None else 1) + (nodes * K * P * P if lo else 0)) + nodes * K
    with torch.cuda.device(out.device), _timed('rotate_pool', flops=2 * nodes * K * Co * P * P, nbytes=nbytes):
        _check(lib().se3_rotate_pool_fwd(_p(Op), _p(D), _p(_u8(mask)), _p(self_add), nodes, K, Co, lo, _p(out), _stream()))


def edge_scale(feats, idx, max_degree):
    """Power-of-two scale per edge from the largest |component| of the neighbour's features (all degrees): [E] fp32."""
    b, n, k = idx.shape
    first = True
    nodemax = torch.empty(b * n, dtype=torch.float32, device=idx.device)
    with torch.cuda.device(idx.device):
        for t in feats.values():
            t = _f32(t)
            _check(lib().se3_rowabsmax_fwd(_p(t), b * n, t.shape[2] * t.shape[3], int(not first), _p(nodemax), _stream()))
            first = False
        sx = torch.empty(b * n * k, dtype=torch.float32, device=idx.device)
        _check(lib().se3_edge_scale_fwd(_p(nodemax), _p(idx.contiguous()), b, n, k, max_degree, _p(sx), _stream()))
    return sx


def linear_supported(D, Eo, device):
    """Shapes the tensor-core LinearSE3 kernel takes."""
    if os.environ.get('SE3B200_NO_LINEAR_TC') or os.environ.get('SE3B200_FORCE_SIMT'):
        return False
    return D % 64 == 0 and Eo % 128 == 0 and torch.cuda.get_device_capability(device)[0] == 10


def linear_image(W):
    """W [D, Eo] fp32 (LinearSE3.weights[degree]) -> tensor-core operand image of W^T for linear_tc."""
    _require_cuda(W)
    D, Eo = W.shape
    Fp = _f32(W.detach().t()).contiguous().reshape(Eo * (D // 16), 16)
    nbytes = lib().se3_zgemm_image_bytes(Eo, 4, D // 64)
    if nbytes < 0:
        raise RuntimeError(f'linear_image: unsupported shape D={D} Eo={Eo}')
    img = torch.empty(nbytes, dtype=torch.uint8, device=W.device)
    with torch.cuda.device(W.device):
        _check(lib().se3_zgemm_pack(_p(Fp), 16, 0, Eo, D // 16, 4, D // 64, 0, _p(img), _stream()))
    return img


def linear_tc(x, img, Eo, res=None):
    """LinearSE3 on the tensor cores: x [b,n,D,M] (reference layout, read in place) -> [b,n,Eo,M] (+ res)."""
    _require_cuda(x, img, res)
    x = _f32(x)
    b, n, D, M = x.shape
    nodes = b * n
    out = torch.empty((b, n, Eo, M), dtype=torch.float32, device=x.device)
    if res is not None:
        res = _f32(res)
        assert res.shape == out.shape
    with torch.cuda.device(x.device):
        rowmax = torch.empty(nodes, dtype=torch.float32, device=x.device)
        sx = torch.empty(nodes, dtype=torch.float32, device=x.device)
        _check(lib().se3_rowabsmax_fwd(_p(x), nodes, D * M, 0, _p(rowmax), _stream()))
        _check(lib().se3_pow2_scale_fwd(_p(rowmax), nodes, 14, _p(sx), _stream()))
        nbytes = img.numel() + 4 * (2 * x.numel() + out.numel() * (2 if res is not None else 1))
        with _timed('linear', flops=2 * nodes * M * D * Eo, nbytes=nbytes, mma=2 * nodes * M * D * Eo * 3, tag=f'linear D{D}E{Eo}M{M}'):
            _check(lib().se3_linear_tc_fwd(_p(x), _p(img), _p(res), _p(sx), nodes, D, Eo, M, _p(out), _stream()))
    return out


def zgemm_tile_n(Co, mode):
    return lib().se3_zgemm_tile_n(Co, mode)


def zgemm_image(parts, Co, mode):
    """parts: [(Fp [Co*Ci*F, Kp] fp32, Ci)] in K order (one entry per input degree; Kp / 16 sub-segments each; F = 1 for mode 1,
    rows (o, i, (a, b)) for modes 2 and 3) -> (uint8 image, total_stages)."""
    F = 1 if mode == 1 else 2
    per_seg = (lambda Ci: 3 * (Ci // 4)) if mode == 3 else (lambda Ci: Ci * F // 4)
    stages = [(Fp.shape[1] // 16) * per_seg(Ci) for Fp, Ci in parts]
    S = sum(stages)
    nbytes = lib().se3_zgemm_image_bytes(Co, mode, S)
    if nbytes < 0:
        raise RuntimeError(f'zgemm_image: unsupported shape Co={Co} mode={mode}')
    dev = parts[0][0].device
    img = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s0 = 0
    with torch.cuda.device(dev):
        for Fp, Ci in parts:
            _require_cuda(Fp)
            Fp = _f32(Fp)
            Kp = Fp.shape[1]
            assert Fp.shape[0] == Co * Ci * F and Kp % 16 == 0 and (Ci * F) % 4 == 0
            for kc in range(Kp // 16):
                _check(lib().se3_zgemm_pack(_p(Fp), Kp, 16 * kc, Co, Ci * F, mode, S, s0, _p(img), _stream()))
                s0 += per_seg(Ci)
    return img, S


def zgemm(segs, w_img, sx, E, Co, mode, out, out_edge_stride, comp_off, flush_stages=0, alg_flops=0, tag=''):
    """segs: [(U [E,64] view (row stride 64; column offset folded into the pointer), X buffer, Ci, ncomp, cplus, cminus)]."""
    _require_cuda(w_img, sx, out)
    arr = (ZSeg * len(segs))()
    Ktot = 0
    for i, (U, X, Ci, ncomp, cplus, cminus) in enumerate(segs):
        _require_cuda(U, X)
        assert U.dtype == torch.float32 and U.stride(-1) == 1 and (U.dim() == 1 or U.stride(0) == 64)
        arr[i] = ZSeg(U.data_ptr(), X.data_ptr(), Ci, ncomp, cplus, cminus)
        Ktot += Ci * (1, 2, 3)[mode - 1] * 16
    N = zgemm_tile_n(Co, mode)
    # issued tensor-core FLOPs: 3 fp16 passes of 2 M N K; mode 2 feeds two accumulators from every B tile, mode 3 has three
    # weight sets with one accumulator each
    mma = 2 * E * Co * Ktot * 3 * (2 if mode == 2 else 1)
    planes = 1 if mode == 1 else 2
    nbytes = w_img.numel() + 4 * E * Co * planes + sum(4 * E * s[2] * (planes + 16) for s in segs)
    with torch.cuda.device(out.device), _timed('zgemm', flops=alg_flops, nbytes=nbytes, tag=tag or f'mode{mode}N{N}K{Ktot}', mma=mma):
        _check(lib().se3_zgemm_fwd(arr, len(segs), _p(w_img), _p(sx), E, Co, mode, _p(out), out_edge_stride, comp_off[0],
                                   comp_off[1] if len(comp_off) > 1 else 0, flush_stages, _stream()))


# max-abs residual of the radial basis relative to max|G|.  The fp32 trunk itself carries ~6e-7..1e-6 of rounding noise
# against float64, so 1e-6 keeps the truncation below what fp32 can resolve; at the headline width (depth-2 slice of cfg2)
# the output differs from the fp32 SIMT path by 1.6e-5 with 1e-6 and by 1.5e-5 with 2e-7 or with the direct K = 128 kernel
# (tools/lr_tol_check.py).  With 1e-6, 96 % of the cfg2 pairs need rank <= 15 (K = 16) instead of 26 % with 2e-7.
LOWRANK_TOL = 1e-6


def lowrank_basis(G64, tol=None, ranks=(15, 31, 47, 63)):
    """Affine low-rank model of the curve G64 [S, 128] (float64 samples of a radial trunk along its input curve):
    returns (r, V [128, r] float64 orthonormal, mean [128] float64) for the smallest listed rank with
    max|(G - mean) - ((G - mean) V) V^T| <= tol * max|G|, else None.  The mean costs nothing downstream: W3 mean joins the bias
    column of F' (the ones column of U), and centring lowers the rank the tolerance needs by one (measured on 120 random
    trunks: ranks 14/15/16/17 for 26/52/22/1 % without, 13/14/15/16 with), so that ~99 % instead of ~78 % of the pairs fit K = 16.
    QR + SVD of the triangular factor (no Gram matrix, so the small singular directions stay accurate)."""
    if tol is None:
        tol = float(os.environ.get('SE3B200_LOWRANK_TOL', LOWRANK_TOL))
    G64 = G64.detach()
    mean = G64.mean(dim=0)
    H = G64 - mean
    Rm = torch.linalg.qr(H, mode='r').R              # Q is never needed
    # SVD of the 128 x 128 triangular factor on the host: 128 KB to move, ~1 ms of LAPACK, instead of the hundreds of small
    # launches of the iterative device SVD per (degree_in, degree_out) pair at plan time
    Vh = torch.linalg.svd(Rm.cpu())[2].to(G64.device)
    gmax = float(G64.abs().max())
    for r in ranks:
        V = Vh[:r].t().contiguous()
        res = float((H - (H @ V) @ V.t()).abs().max())
        if res <= tol * gmax:
            return r, V, mean
    return None


def lowrank_enabled(E):
    if os.environ.get('SE3B200_NO_LOWRANK'):
        return False
    return E >= int(os.environ.get('SE3B200_LOWRANK_MIN_EDGES', 16384))


def tc_supported(device, Co, P):
    """The tcgen05 kernel needs sm_100 and Co % 32 == 0, degree_out <= 3."""
    if os.environ.get('SE3B200_FORCE_SIMT'):
        return False
    if Co % TILE_O != 0 or P > 7:
        return False
    return torch.cuda.get_device_capability(device)[0] == 10


def pool(x, mask):
    """masked mean over axis 2 of x [b,n,k,...] with mask [b,n,k] (reference utils.py:72-80)."""
    _require_cuda(x, mask)
    x = _f32(x)
    b, n, k = x.shape[:3]
    C = x[0, 0, 0].numel()
    out = torch.empty((b, n) + tuple(x.shape[3:]), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed('pool', nbytes=4 * (x.numel() + out.numel()) + b * n * k):
        _check(lib().se3_pool_fwd(_p(x), _p(_u8(mask)), b * n, k, C, _p(out), _stream()))
    return out


# ---------------------------------------------------------------------------------------------------------
# K5
# ---------------------------------------------------------------------------------------------------------
def attention(q, k, v, *, heads, dim_head, scale, nmask=None, k_idx=None, self_k=None, self_v=None, null_k=None, null_v=None,
              global_k=None, global_v=None, kv_heads=None, D=None, k_aligned=False):
    """One degree of AttentionSE3 / OneHeadedKVAttentionSE3 (reference S:476-517, 612-652).
    q [b,n,H*Dh,M]; k,v [b,n,K,Ckv,M] (k may be node level [b,n,Ckv,M] with k_idx [b,n,K]).
    With D [b*n*K, M, M] (edge frames): v (and k if k_aligned) are the edge-aligned, component-major [b,n,K,M,Ckv] outputs of
    zgemm and the rotation back to the global frame is fused into the kernel (se3_attn_aligned_fwd)."""
    _require_cuda(q, k, v, D)
    q, k, v = _f32(q), _f32(k), _f32(v)
    b, n, _, M = q.shape
    K = v.shape[2]
    kv_heads = heads if kv_heads is None else kv_heads
    G = 0 if global_k is None else global_k.shape[1]
    cont = lambda t: None if t is None else _f32(t)
    self_k, self_v, null_k, null_v, global_k, global_v = map(cont, (self_k, self_v, null_k, null_v, global_k, global_v))
    out = torch.empty_like(q)
    nm = _u8(nmask)
    ki = None if k_idx is None else k_idx.contiguous()
    J = K + G + (self_k is not None) + (null_k is not None)
    nbytes = 4 * (2 * q.numel() + 2 * b * n * J * heads * dim_head * M)
    if D is not None:
        assert M > 1 and D.is_contiguous() and D.numel() == b * n * K * M * M and v.shape[3] == M
        nbytes += 4 * D.numel()
        with torch.cuda.device(q.device), _timed('attention', flops=4 * b * n * J * heads * dim_head * M * (1 + M), nbytes=nbytes):
            _check(lib().se3_attn_aligned_fwd(_p(q), _p(k), _p(v), _p(D), int(bool(k_aligned)), _p(ki), _p(self_k), _p(self_v), _p(null_k),
                                              _p(null_v), _p(global_k), _p(global_v), G, _p(nm), b, n, K, heads, dim_head, M, kv_heads,
                                              float(scale), _p(out), _stream()))
        return out
    with torch.cuda.device(q.device), _timed('attention', flops=4 * b * n * J * heads * dim_head * M, nbytes=nbytes):
        _check(lib().se3_attn_fwd(_p(q), _p(k), _p(v), _p(ki), _p(self_k), _p(self_v), _p(null_k), _p(null_v), _p(global_k),
                                  _p(global_v), G, _p(nm), b, n, K, heads, dim_head, M, kv_heads, float(scale), _p(out), _stream()))
    return out


def norm_se3(x, scale, eps, use_gelu):
    """NormSE3 with a per-channel scale (reference S:130-152): x [b,n,C,M] -> same shape."""
    _require_cuda(x, scale)
    x = _f32(x)
    C, M = x.shape[-2], x.shape[-1]
    out = torch.empty_like(x)
    with torch.cuda.device(x.device), _timed('norm', nbytes=8 * x.numel()):
        _check(lib().se3_norm_fwd(_p(x), _p(_f32(scale).reshape(-1)), x.numel() // M, C, M, float(eps), int(use_gelu), _p(out), _stream()))
    return out
