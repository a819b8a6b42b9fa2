"""Host-side mirror of the reference's module tree for the SE(3) attention hot path.

Same constructor, forward signature, assertions and state_dict key/shape layout as
lucidrains/se3-transformer-pytorch v0.9.0 (se3_transformer_pytorch.py:936-1375; SURVEY.md Appendix A.6), so
`ours.load_state_dict(reference.state_dict())` works.  The hot path -- neighbour graph, spherical-harmonic / CG basis,
radial trunk, pairwise tensor product (tcgen05), pooling, attention -- runs in the hand-written sm_100a kernels of
libse3b200.so through `ops`; the cheap glue around it (embeddings, LinearSE3 GEMMs, NormSE3, residuals) stays torch.

Forward only: everything runs under torch.no_grad().  CUDA only: there is no CPU fallback.
"""
import os
from math import sqrt

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from . import aligned as _aligned


def exists(v):
    return v is not None


def default(v, d):
    return v if exists(v) else d


def to_order(degree):
    return 2 * degree + 1


class Fiber:
    """Ordered list of (degree, channels) (reference S:20-59)."""

    def __init__(self, structure):
        if isinstance(structure, dict):
            structure = list(structure.items())
        self.structure = [(int(d), int(c)) for d, c in structure]

    @staticmethod
    def create(num_degrees, dim):
        dims = dim if isinstance(dim, tuple) else (dim,) * num_degrees
        return Fiber([(d, c) for d, c in zip(range(num_degrees), dims)])

    @property
    def degrees(self):
        return [d for d, _ in self.structure]

    @property
    def dims(self):
        return list(dict.fromkeys(c for _, c in self.structure))

    def __getitem__(self, degree):
        return dict(self.structure)[degree]

    def __iter__(self):
        return iter(self.structure)

    def shared(self, other):
        """(degree, dim_self, dim_other) for degrees present in both (reference S:52-59)."""
        od = dict(other.structure)
        return [(d, c, od[d]) for d, c in self.structure if d in od]


def forward_only_guard(what, modules, tensors=()):
    """The kernels have no backward (SURVEY.md 8f row 4).  Called with autograd recording and anything that wants a gradient,
    they would silently return tensors cut off from the graph (radial weights and inputs without gradients, the torch glue
    with): fail loudly instead.  SE3Transformer.forward itself runs under torch.no_grad()."""
    if not torch.is_grad_enabled():
        return
    wants = any(t is not None and torch.is_tensor(t) and t.requires_grad for t in tensors) or \
        any(p.requires_grad for m in modules for p in m.parameters())
    if wants:
        raise RuntimeError(f'{what} is forward only (no backward kernels): call it under torch.no_grad() / torch.inference_mode(), '
                           'or use the reference implementation for training')


def residual_add(x, res):
    return {d: (t + res[d] if d in res else t) for d, t in x.items()}


class LinearSE3(nn.Module):
    """Per-degree channel mix (reference S:78-95).  Widths the tensor-core kernel takes (C_in % 64 == 0, C_out % 128 == 0) run
    on se3_linear_tc_fwd: the A operand is read in place from the reference layout, split to fp16 hi / lo on the fly (fp32
    parity), an optional residual is added in the epilogue; other widths are a plain cuBLAS GEMM."""

    def __init__(self, fiber_in, fiber_out):
        super().__init__()
        self.weights = nn.ParameterDict()
        for degree, dim_in, dim_out in fiber_in.shared(fiber_out):
            self.weights[str(degree)] = nn.Parameter(torch.randn(dim_in, dim_out) / sqrt(dim_in))
        self._images = {}

    def image(self, degree):
        w = self.weights[degree]
        ver = (w._version, w.data_ptr())
        hit = self._images.get(degree)
        if hit is None or hit[0] != ver:
            ok = float(w.detach().abs().max()) < 6.0e4              # fp16 range of the hi / lo split
            hit = (ver, ops.linear_image(w) if ok else None)
            self._images[degree] = hit
        return hit[1]

    def forward(self, x, residual=None):
        out = {}
        for degree, w in self.weights.items():
            t = x[degree]                                            # [b, n, d, m]
            res = residual.get(degree) if residual is not None else None
            if t.is_cuda and t.dtype == torch.float32 and not torch.is_grad_enabled() and ops.linear_supported(w.shape[0], w.shape[1], t.device):
                img = self.image(degree)
                if img is not None:
                    out[degree] = ops.linear_tc(t, img, w.shape[1], res=res)
                    continue
            y = torch.matmul(t.transpose(-1, -2), w).transpose(-1, -2).contiguous()
            out[degree] = y if res is None else y + res
        return out                                                   # (degrees only in `residual` are dropped, as ResidualSE3 S:67-76)


class NormSE3(nn.Module):
    """Norm nonlinearity (reference S:97-152)."""

    def __init__(self, fiber, nonlin=None, gated_scale=False, eps=1e-12):
        super().__init__()
        self.fiber = fiber
        self.nonlin = nonlin if nonlin is not None else nn.GELU()
        self.eps = eps
        self.transform = nn.ModuleDict()
        for degree, chan in fiber:
            pd = nn.ParameterDict()
            if gated_scale:
                pd['w_gate'] = nn.Parameter(torch.empty(chan, chan).uniform_(-1e-3, 1e-3))
            else:
                pd['scale'] = nn.Parameter(torch.ones(1, 1, chan))
            self.transform[str(degree)] = pd

    def forward(self, features):
        out = {}
        for degree, t in features.items():
            pd = self.transform[degree]
            fused = 'scale' in pd and t.is_cuda and t.dtype == torch.float32 and isinstance(self.nonlin, (nn.GELU, nn.Identity)) \
                and not (isinstance(self.nonlin, nn.GELU) and self.nonlin.approximate != 'none')
            if fused:                                    # one fused kernel (libse3b200: se3_norm_fwd)
                out[degree] = ops.norm_se3(t, pd['scale'], self.eps, isinstance(self.nonlin, nn.GELU))
                continue
            norm = t.norm(dim=-1, keepdim=True).clamp(min=self.eps)
            phase = t / norm
            pd = self.transform[degree]
            tr = norm.squeeze(-1)
            scale = pd['scale'] if 'scale' in pd else torch.matmul(tr, pd['w_gate'])
            tr = self.nonlin(tr * scale)
            out[degree] = (tr.unsqueeze(-1) * phase).view(*t.shape)
        return out


class RadialFunc(nn.Module):
    """Parameter holder for the radial MLP (reference S:270-299).  `net` keeps the reference's Sequential indices
    (0 Linear, 1 LayerNorm, 3 Linear, 4 LayerNorm, 6 Linear) so state_dict keys match; evaluation happens in the
    fused kernels, never here."""

    def __init__(self, num_freq, in_dim, out_dim, edge_dim=0, mid_dim=ops.RADIAL_MID):
        super().__init__()
        assert mid_dim == ops.RADIAL_MID
        self.num_freq, self.in_dim, self.out_dim, self.edge_dim = num_freq, in_dim, out_dim, edge_dim
        self.net = nn.ModuleDict({
            '0': nn.Linear(edge_dim + 1, mid_dim),
            '1': nn.LayerNorm(mid_dim),
            '3': nn.Linear(mid_dim, mid_dim),
            '4': nn.LayerNorm(mid_dim),
            '6': nn.Linear(mid_dim, num_freq * in_dim * out_dim),
        })

    def trunk64(self, feat):
        """The trunk (net.0 .. net.5) in float64 with torch ops: used off the hot path, to sample the curve g(d) when the
        low-rank plan of a pair is built."""
        n = self.net
        h = F.linear(feat.double(), n['0'].weight.double(), n['0'].bias.double())
        h = F.gelu(F.layer_norm(h, (h.shape[-1],), n['1'].weight.double(), n['1'].bias.double()))
        h = F.linear(h, n['3'].weight.double(), n['3'].bias.double())
        return F.gelu(F.layer_norm(h, (h.shape[-1],), n['4'].weight.double(), n['4'].bias.double()))

    def trunk_params(self):
        n = self.net
        return torch.cat([n['0'].weight.t().reshape(-1), n['0'].bias, n['1'].weight, n['1'].bias,
                          n['3'].weight.t().reshape(-1), n['3'].bias, n['4'].weight, n['4'].bias])


class PairwiseConv(nn.Module):
    """Holder for one (degree_in, degree_out) radial profile (reference S:301-343)."""

    def __init__(self, degree_in, nc_in, degree_out, nc_out, edge_dim=0):
        super().__init__()
        self.degree_in, self.degree_out, self.nc_in, self.nc_out = degree_in, degree_out, nc_in, nc_out
        self.num_freq = to_order(min(degree_in, degree_out))
        self.d_out = to_order(degree_out)
        self.rp = RadialFunc(self.num_freq, nc_in, nc_out, edge_dim)


# upper bound on the T workspace (bytes); larger convolutions are evaluated in edge chunks
T_WORKSPACE_BYTES = int(8 * 2 ** 30)


class ConvSE3(nn.Module):
    """Tensor-field-network layer (reference S:154-268) on the fused kernels."""

    def __init__(self, fiber_in, fiber_out, self_interaction=True, pool=True, edge_dim=0, fourier_encode_dist=False,
                 num_fourier_features=4, splits=4):
        super().__init__()
        self.fiber_in, self.fiber_out = fiber_in, fiber_out
        self.edge_dim = edge_dim
        self.self_interaction = self_interaction
        self.num_fourier_features = num_fourier_features
        self.fourier_encode_dist = fourier_encode_dist
        self.splits = splits          # accepted for API parity; chunking is by T_WORKSPACE_BYTES instead
        edge_dim += 0 if not fourier_encode_dist else num_fourier_features * 2
        self.in_dim = edge_dim + 1
        self.kernel_unary = nn.ModuleDict()
        self.pairs = []
        for di, mi in fiber_in:
            for do, mo in fiber_out:
                self.kernel_unary[f'({di},{do})'] = PairwiseConv(di, mi, do, mo, edge_dim=edge_dim)
                self.pairs.append((di, do))
        self.pool = pool
        if self_interaction:
            assert self.pool, 'must pool edges if followed with self interaction'
            self.self_interact = LinearSE3(fiber_in, fiber_out)
        self._packed = None
        self.free_master = False

    # ---- packed weights ---------------------------------------------------------------------------------
    def _param_version(self):
        v = []
        for p in self.kernel_unary.parameters():
            v.append((p._version, p.data_ptr()))
        return tuple(v)

    def packed(self):
        """Trunk parameter pack [pairs, stride] (built lazily, rebuilt when weights change) + a cache of the tensor-core
        images of net.6 for the direct (K = 128) kernel, filled on demand by w3_image()."""
        ver = None if self.free_master else self._param_version()
        if self._packed is not None and (self.free_master or self._packed['version'] == ver):
            return self._packed
        with torch.no_grad():
            trunk = torch.stack([self.kernel_unary[f'({di},{do})'].rp.trunk_params() for di, do in self.pairs]).contiguous()
        self._packed = dict(version=ver, trunk=trunk, images={}, tc_ok={})
        return self._packed

    def tc_eligible(self, di, do):
        """The tcgen05 kernels take this pair: sm_100, C_out % 32 == 0, degree_out <= 3 and operands inside the fp16 range
        of the hi/lo split (|g| <= sqrt(127) max|ln.w| + max|ln.b| after LayerNorm + GELU)."""
        pk = self.packed()
        if (di, do) not in pk['tc_ok']:
            pc = self.kernel_unary[f'({di},{do})']
            ok = ops.tc_supported(pk['trunk'].device, pc.nc_out, pc.d_out)
            if ok and (di, do) not in pk['images']:
                lin, ln = pc.rp.net['6'], pc.rp.net['4']
                g_bound = 11.3 * float(ln.weight.abs().max()) + float(ln.bias.abs().max())
                ok = g_bound < 6.0e4 and (lin.weight.numel() == 0 or float(lin.weight.abs().max()) < 6.0e4)
            pk['tc_ok'][(di, do)] = ok
        return pk['tc_ok'][(di, do)]

    def w3_image(self, di, do):
        pk = self.packed()
        if (di, do) not in pk['images']:
            pc = self.kernel_unary[f'({di},{do})']
            lin = pc.rp.net['6']
            if lin.weight.numel() == 0:
                raise RuntimeError(f'ConvSE3 pair ({di},{do}): the fp32 net.6 weights were released by pack_weights(free_master=True) and '
                                   'only the low-rank image was kept, but this forward needs the direct (K = 128) image (low-rank path '
                                   'switched off or not applicable); rebuild the model or pack with free_master=False')
            with torch.no_grad():
                pk['images'][(di, do)] = ops.pack_w3(lin.weight, lin.bias, pc.nc_out, pc.nc_in, pc.num_freq)
        return pk['images'][(di, do)]

    # ---- low-rank radial path ----------------------------------------------------------------------------
    LR_GRID = 16384          # float64 samples of g(d) per pair when a plan is built
    LR_RUNTIME_TOL = 1e-5    # sanity bound on max|G - (G V) V^T| / max|G| of the fp32 trunk outputs of a forward

    def encode_dist(self, rd):
        """[..., 1] distances -> radial-MLP input (reference utils.py:96-104 when fourier_encode_dist)."""
        if not self.fourier_encode_dist:
            return rd
        scales = 2 ** torch.arange(self.num_fourier_features, device=rd.device, dtype=rd.dtype)
        xs = rd / scales
        return torch.cat([xs.sin(), xs.cos(), rd], dim=-1)

    def lowrank_plan(self, d_max):
        """Per pair: orthonormal V [128, r] spanning the curve g(d), d in [0, D], and the tensor-core images of
        F'' = [W3 V | b3 | 0] for the route the ConvSE3 will take.  Depends on the weights and on D only: built once (and again
        if weights change or a forward brings a larger distance).  Only for distance-only radial functions (no extra edge
        features)."""
        pk = self.packed()
        plan = pk.get('lr')
        if plan is not None and plan['D'] >= d_max:
            return plan
        dev = pk['trunk'].device
        D = 1.25 * d_max
        with torch.no_grad():
            grid = torch.linspace(0.0, D, self.LR_GRID, device=dev, dtype=torch.float64).unsqueeze(-1)
            bases, ugrid = self.lowrank_bases(grid)
            covered = len(bases) == len(self.pairs)
            # the edge-aligned images serve a ConvSE3 only if EVERY pair has a plan (all launches of an output degree then
            # accumulate in the aligned frame); otherwise keep the global-frame images of 4.2-4.3 for the covered pairs
            route = GLOBAL
            if covered and use_aligned():
                route = ZGEMM if use_zgemm() and self.zgemm_eligible({pair: _kp(r) for pair, (r, _, _) in bases.items()}) else ALIGNED
            pairs, fps = {}, {}
            for (di, do), (r, V, gmean) in bases.items():
                Fp = self.fold_w3(di, do, r, V, gmean)
                pairs[(di, do)] = rec = dict(r=r, Kp=_kp(r), V=torch.zeros((ops.RADIAL_MID, 64), dtype=torch.float32, device=dev),
                                             gmean=gmean.float())
                rec['V'][:, :r] = V.float()
                if route == ZGEMM:               # concatenated over the input degrees into one GEMM image per (do, m) below
                    fps.update({(di, do, m): w for m, w in enumerate(self.aligned_weights(di, do, Fp))})
                elif route == ALIGNED:           # one image per |m| (DESIGN.md 4.4)
                    pc = self.kernel_unary[f'({di},{do})']
                    rec['al_imgs'] = [ops.pack_lowrank(w, pc.nc_out, pc.nc_in, 1 if m == 0 else 2, rec['Kp'])
                                      for m, w in enumerate(self.aligned_weights(di, do, Fp))]
                else:
                    rec.update(self.global_images(di, do, Fp))
                del Fp
            zplan = self.zgemm_images(fps) if route == ZGEMM else None
            utab = self.radial_table(ugrid, bases, grid, dev) if covered and use_utable() else None
            del ugrid, fps
            # per-pair operands of the radial kernels, stacked over all pairs of the ConvSE3 (zero for pairs without a plan)
            zero = torch.zeros((ops.RADIAL_MID, 64), dtype=torch.float32, device=dev)
            recs = [pairs.get(p, dict(V=zero, gmean=zero[:, 0], r=0)) for p in self.pairs]
            plan = dict(D=D, pairs=pairs, z=zplan, utab=utab, Vstack=torch.stack([p['V'] for p in recs]),
                        gmean=torch.stack([p['gmean'] for p in recs]), ones_col=torch.tensor([p['r'] for p in recs], dtype=torch.int32, device=dev),
                        have=torch.tensor([p in pairs for p in self.pairs], device=dev))
        pk['lr'] = plan
        return plan

    def lowrank_bases(self, grid):
        """{pair: (r, V, gmean)} low-rank bases of the trunk outputs on the grid, {pair: (U(d) on the grid, max|g|)}."""
        feat = self.encode_dist(grid)
        bases, ugrid = {}, {}
        for di, do in self.pairs:
            pc = self.kernel_unary[f'({di},{do})']
            if self.tc_eligible(di, do) and pc.rp.net['6'].weight.numel() > 0:
                G64 = pc.rp.trunk64(feat)
                basis = ops.lowrank_basis(G64)
                if basis is not None:
                    bases[(di, do)] = basis
                    ugrid[(di, do)] = ((G64 - basis[2]) @ basis[1], float(G64.abs().max()))     # U(d) on the grid, float64
                del G64
        return bases, ugrid

    def fold_w3(self, di, do, r, V, gmean):
        """F' = [W3 V | b3 + W3 gmean | 0] [Co*Ci*F, Kp] fp32, rows (o, i, f): the radial weights as a function of U."""
        lin = self.kernel_unary[f'({di},{do})'].rp.net['6']
        Fp = torch.zeros((lin.weight.shape[0], _kp(r)), dtype=torch.float32, device=V.device)
        Fp[:, :r] = (lin.weight.double() @ V).float()
        Fp[:, r] = (lin.bias.double() + lin.weight.double() @ gmean).float()      # affine model: W3 gmean joins the bias
        return Fp

    def aligned_weights(self, di, do, Fp):
        """The edge-aligned weights w0, (a_m, b_m), m = 1..min(di, do): constant combinations of the F frequencies (rows
        (o,i,f) of F'), as [Co*Ci, Kp] for m = 0 and [Co*Ci*2, Kp] (rows (o, i, (a, b))) otherwise."""
        pc = self.kernel_unary[f'({di},{do})']
        Kp = Fp.shape[1]
        Fv = Fp.view(pc.nc_out, pc.nc_in, pc.num_freq, Kp).double()
        c0, ca, cb = (t.to(Fp.device) for t in _aligned.aligned_coeffs(di, do))
        out = [torch.einsum('oifk,f->oik', Fv, c0).reshape(-1, Kp).float().contiguous()]
        for m in range(1, min(di, do) + 1):
            ab = torch.stack([torch.einsum('oifk,f->oik', Fv, ca[m - 1]), torch.einsum('oifk,f->oik', Fv, cb[m - 1])], dim=2)
            out.append(ab.reshape(-1, Kp).float().contiguous())
        return out

    def global_images(self, di, do, Fp):
        """Global frame (DESIGN.md 4.2-4.3): `img` (all frequencies) for the output-side contraction, `imgs_f` (one per
        frequency) for the input-side one; a single-frequency pair has both."""
        pc = self.kernel_unary[f'({di},{do})']
        Kp = Fp.shape[1]
        if input_side(di, do) and pc.num_freq > 1:
            Fv = Fp.view(pc.nc_out, pc.nc_in, pc.num_freq, Kp)
            return dict(imgs_f=[ops.pack_lowrank(Fv[:, :, f, :].reshape(-1, Kp).contiguous(), pc.nc_out, pc.nc_in, 1, Kp)
                                for f in range(pc.num_freq)])
        img = ops.pack_lowrank(Fp, pc.nc_out, pc.nc_in, pc.num_freq, Kp)
        return dict(img=img, imgs_f=[img]) if pc.num_freq == 1 else dict(img=img)

    def zgemm_images(self, fps):
        """{(do, m): one GEMM image over the input degrees di >= m (DESIGN.md 4.5)} from the aligned weights fps[(di, do, m)]."""
        zplan = {}
        for do, mo in self.fiber_out:
            for m in range(do + 1):
                degs = [(di, mi) for di, mi in self.fiber_in if di >= m]
                if not degs:
                    continue
                mode = 1 if m == 0 else z_mode_m()
                img, S = ops.zgemm_image([(fps.pop((di, do, m)), mi) for di, mi in degs], mo, mode)
                zplan[(do, m)] = dict(img=img, S=S, degs=degs, mode=mode)
        return zplan

    UTABLE_TOL = 5e-7        # max interpolation error of the tabulated radial coordinates relative to max|g| (float64, grid midpoints)

    def radial_table(self, ugrid, bases, grid, dev):
        """The radial coordinates U(d) = (g(d) - gmean) V of every pair tabulated on the plan's uniform distance grid (float64 ->
        fp32 [pairs, G, KT]); the forward interpolates them (se3_radial_table_fwd, 4-point Lagrange) instead of evaluating the MLP
        per edge.  Accepted only if the interpolant reproduces the float64 trunk at the grid MIDPOINTS to UTABLE_TOL (smooth
        radial functions pass by orders of magnitude; a rougher one falls back to se3_radial_trunk_u_fwd)."""
        Gn = grid.shape[0]
        KT = max(_kp(bases[p][0]) for p in self.pairs)
        tab = torch.zeros((len(self.pairs), Gn, KT), dtype=torch.float32, device=dev)
        mid = (grid[:-1] + grid[1:]) * 0.5
        featm = self.encode_dist(mid)
        worst = 0.0
        for pi, pair in enumerate(self.pairs):
            r, V, gmean = bases[pair]
            Ug, gmax = ugrid[pair]
            tab[pi, :, :r] = Ug.float()
            pc = self.kernel_unary[f'({pair[0]},{pair[1]})']
            exact = (pc.rp.trunk64(featm) - gmean) @ V                                      # [G-1, r] float64
            T = tab[pi, :, :r].double()
            i0 = torch.arange(Gn - 1, device=dev).clamp(1, Gn - 3)                          # as the kernel chooses its 4 nodes
            f = (torch.arange(Gn - 1, device=dev, dtype=torch.float64) + 0.5 - i0).unsqueeze(-1)
            w = (-f * (f - 1) * (f - 2) / 6, (f + 1) * (f - 1) * (f - 2) / 2, -(f + 1) * f * (f - 2) / 2, (f + 1) * f * (f - 1) / 6)
            interp = sum(w[j] * T[i0 - 1 + j] for j in range(4))
            worst = max(worst, float((interp - exact).abs().max()) / max(gmax, 1e-30))
        self.utable_error = worst
        return tab if worst <= self.UTABLE_TOL else None

    def zgemm_eligible(self, kps):
        """Shapes the one-GEMM kernel takes: every C_out a multiple of 128, every C_in a multiple of 4 (one stage = 64 K values),
        at most 16 K segments per launch (a pair with K = 16 j contributes j), and |g|_2 small enough for the fp16 operands
        (|Z| <= 2^10 |U|, |U_k| <= |g|_2 <= 11.32 (max|ln.w| + max|ln.b|))."""
        if any(mo % 128 for _, mo in self.fiber_out) or any(mi % 4 for _, mi in self.fiber_in):
            return False
        for do, _ in self.fiber_out:
            if sum(kps[(di, do)] // 16 for di, _ in self.fiber_in) > 16:
                return False
        for di, do in self.pairs:
            ln = self.kernel_unary[f'({di},{do})'].rp.net['4']
            if 11.32 * (float(ln.weight.abs().max()) + float(ln.bias.abs().max())) > 60.0:
                return False
        return True

    def pack_weights(self, free_master=False, max_distance=None):
        """Build the tensor-core weight images now.  With max_distance (an upper bound on the neighbour distances the model
        will see) and distance-only radial functions, the low-rank plan is built and pairs it covers need no direct
        (K = 128) image.  free_master=True then releases the fp32 net.6 weights of every imaged pair (inference only:
        state_dict() no longer holds them)."""
        covered = {}
        if max_distance is not None and self.edge_dim == 0 and not os.environ.get('SE3B200_NO_LOWRANK'):
            covered = self.lowrank_plan(float(max_distance) / 1.25)['pairs']
        for di, do in self.pairs:
            if self.tc_eligible(di, do) and (di, do) not in covered:
                self.w3_image(di, do)
        if free_master:
            pk = self.packed()
            self.free_master = True
            for key in list(pk['images']) + list(covered):
                lin = self.kernel_unary[f'({key[0]},{key[1]})'].rp.net['6']
                lin.weight.data = torch.empty(0, device=pk['trunk'].device)
        return self.packed()

    # ---- forward ----------------------------------------------------------------------------------------
    def edge_features(self, edge_info, rel_dist):
        _, _, edges = edge_info
        rd = self.encode_dist(rel_dist.unsqueeze(-1))
        feat = torch.cat((rd, edges), dim=-1) if exists(edges) else rd
        return feat.reshape(-1, feat.shape[-1]).contiguous()

    def forward(self, inp, edge_info, rel_dist=None, basis=None):
        return conv_forward([self], inp, edge_info, rel_dist, basis)[0]


def input_side(di, do):
    """Degree pairs evaluated with the input-side contraction on the low-rank path: out = B . (R x) instead of R (B x).
    The fused kernel then spends 2 l_in + 1 instead of 2 l_out + 1 FMAs per radial weight; worth it for l_in <= 1 < l_out
    and for l_in = 0 (measured: (0,3) 7.7 -> 2.6 ms, (1,3) 19.3 -> ~11.4 ms at cfg2 widths)."""
    return di < do and di <= 1 and not os.environ.get('SE3B200_NO_INPUT_SIDE')


def use_zgemm():
    """One GEMM per (degree_out, |m|) with the A operand generated on the fly (DESIGN.md 4.5) instead of the R-first kernels."""
    return not os.environ.get('SE3B200_NO_ZGEMM')


def use_utable():
    """Radial coordinates by table lookup (se3_radial_table_fwd) instead of the per-edge radial MLP (se3_radial_trunk_u_fwd)."""
    return not os.environ.get('SE3B200_NO_UTABLE')


def z_mode_m():
    """Kernel mode of the |m| > 0 launches: 3 = three real products per complex one (Gauss; 3/4 of the tensor-core work of mode 2)."""
    return 2 if os.environ.get('SE3B200_Z_MODE2') else 3


def use_aligned():
    """Edge-aligned evaluation of the low-rank path (DESIGN.md 4.4): 2 FMAs per radial weight instead of 2 l_out + 1."""
    return not os.environ.get('SE3B200_NO_ALIGNED')


class Geometry:
    """Per-forward edge geometry shared by every layer; the aligned frames are built on first use."""

    def __init__(self, rel_pos, max_degree):
        self.rel_pos, self.max_degree, self._frames = rel_pos, max_degree, None
        # run-time checks of the low-rank plans, as (ConvSE3, stats [pairs, 2]) : None = check inside every ConvSE3 (one host
        # synchronisation each); a list = the caller collects them and checks once per forward (SE3Transformer.forward)
        self.deferred = None
        self._dmax = None

    def d_max(self, rel_dist):
        if self._dmax is None:
            self._dmax = float(rel_dist.max())          # the one host synchronisation of the plan lookup, once per forward
        return self._dmax

    def to_global(self, akv):
        """AlignedKV -> [b, n, k, C, 2lo+1] in the global frame (the rotate-back the attention kernel otherwise fuses)."""
        if not isinstance(akv, AlignedKV):
            return akv
        b, n, k, P, C = akv.t.shape
        out = torch.empty((b * n * k, C, P), dtype=torch.float32, device=akv.t.device)
        rotate_to_global(akv.t.reshape(-1, P, C), self.frames().D[akv.lo], out)
        return out.view(b, n, k, C, P)

    def frames(self):
        """Per-edge Wigner matrices D_l(R_e) (se3_frames_fwd, float64 arithmetic on the device; SE3B200_HOST_FRAMES=1: the
        float64 torch restatement in aligned.py)."""
        if self._frames is None:
            if os.environ.get('SE3B200_HOST_FRAMES'):
                self._frames = _aligned.EdgeFrames(self.rel_pos, self.max_degree)
            else:
                self._frames = _aligned.EdgeFrames(self.rel_pos, self.max_degree, D=ops.frames(self.rel_pos, self.max_degree))
        return self._frames


def check_lowrank_stats(checks):
    """checks: [(ConvSE3, stats [pairs, 2] = (max |g - U V^T|, max |g|) of one forward)].  ONE host synchronisation for all of
    them; returns the ConvSE3 modules whose cached radial basis does not cover this forward's distances."""
    global LAST_PLAN_RESIDUAL
    if not checks:
        return []
    worst = torch.stack([torch.where(have, st[:, 0] / st[:, 1].clamp(min=1e-30), torch.zeros_like(st[:, 0])).max() for _, st, have in checks]).cpu()
    LAST_PLAN_RESIDUAL = float(worst.max())      # diagnostics / tests: how close the last checked forward came to the guard
    return [conv for (conv, _, _), w in zip(checks, worst.tolist()) if not (w <= conv.LR_RUNTIME_TOL)]


LAST_PLAN_RESIDUAL = None


class AlignedKV:
    """A ConvSE3 output of degree lo >= 1 still in the edge-aligned frame (DESIGN.md 4.5): t [b, n, k, 2lo+1, C], component
    major, out[e, c, :] = D_lo(e) t[e, :, c].  AttentionSE3 hands it to the attention kernel, which rotates on the fly;
    Geometry.to_global() materialises the reference-layout tensor [b, n, k, C, 2lo+1]."""

    def __init__(self, t, lo):
        self.t, self.lo = t, lo


class LowRankPlanMiss(RuntimeError):
    """The radial trunk outputs of a forward left the cached low-rank subspace (distances beyond the plan's range)."""


ZGEMM, ALIGNED, GLOBAL = 'zgemm', 'aligned', 'global'       # the routes of a ConvSE3 forward (conv_route, DESIGN.md 4)


def _kp(r):
    """K of the low-rank radial GEMM: r basis columns + the ones column, in steps of 16."""
    return 16 * ((r + 1 + 15) // 16)


def conv_route(conv, E, edge_info, rel_dist, geom, capturing):
    """The route of one ConvSE3 for this forward and what it needs: dict(route, lr = {pair: plan record} of the low-rank pairs,
    U / g = outputs of the radial kernels it launches, z = the one-GEMM images, outs = per-edge output buffers)."""
    pk = conv.packed()
    feat = conv.edge_features(edge_info, rel_dist)
    assert feat.shape[-1] == conv.in_dim, f'edge feature width {feat.shape[-1]} != {conv.in_dim}'
    tc_ok = {pair: conv.tc_eligible(*pair) for pair in conv.pairs}
    # low-rank radial path (distance-only radial functions): U = G V with the pair's cached basis, K = r+1 <= 64
    plan = None
    if os.environ.get('SE3B200_NO_LOWRANK') or conv.edge_dim != 0:
        pass
    elif conv.free_master and pk.get('lr') is not None:
        plan = pk['lr']                         # built by pack_weights(max_distance=...) before the masters went away:
                                                # the only image there is, whatever the edge count
    elif ops.lowrank_enabled(E) and any(tc_ok.values()) and not conv.free_master and not getattr(conv, '_lr_blocked', False):
        # while capturing: the plan the warm-up forwards built (the residual check below still covers it); otherwise cached,
        # it needs the distance range (one host sync per forward, in Geometry)
        plan = pk.get('lr') if capturing else conv.lowrank_plan(geom.d_max(rel_dist) if geom is not None else float(rel_dist.max()))
    st = dict(conv=conv, route=GLOBAL, tc_ok=tc_ok, lr={}, U=None, g=None, z=None,
              outs={do: torch.empty((E, mo, to_order(do)), dtype=torch.float32, device=feat.device) for do, mo in conv.fiber_out})
    if plan is not None and plan['pairs']:
        # trunk + U = G V + the residual statistics of the cached subspace on THIS forward's edges, one kernel
        covered = len(plan['pairs']) == len(conv.pairs)
        stats = torch.zeros((len(conv.pairs), 2), dtype=torch.float32, device=feat.device)
        if covered and plan['utab'] is not None and use_utable():
            # distance-only radial functions: U(d) interpolated from the plan's float64 table; the guard is the table's range
            st['U'] = ops.radial_table(rel_dist, plan['utab'], plan['D'], plan['ones_col'], stats)
        else:
            st['U'], st['g'] = ops.radial_trunk_u(feat, pk['trunk'], plan['Vstack'], plan['gmean'], plan['ones_col'], stats,
                                                  want_g=not covered)
        st['lr'] = dict(plan['pairs'])
        check = (conv, stats, plan['have'])
        if geom is not None and geom.deferred is not None:
            geom.deferred.append(check)          # checked once per forward by the caller
        elif check_lowrank_stats([check]):
            # the fp32 trunk outputs of this forward leave the cached subspace (distances beyond the plan's range)
            if conv.free_master:
                raise LowRankPlanMiss('low-rank radial plan does not cover this input; pack_weights(max_distance=...) was given too '
                                      'small a distance')
            st['lr'] = {}                        # evaluate this ConvSE3 with the direct K = 128 kernels
        if st['lr'] and covered and geom is not None:
            if plan['z'] is not None:
                st['route'], st['z'] = ZGEMM, plan['z']
            elif all('al_imgs' in pp for pp in st['lr'].values()):
                st['route'] = ALIGNED
    if st['route'] == GLOBAL and any('img' not in pp and 'imgs_f' not in pp for pp in st['lr'].values()):
        # the plan holds edge-aligned images only (DESIGN.md 4.4-4.5); they need the per-forward Geometry
        if geom is None:
            raise RuntimeError('ConvSE3 was called with a (flat, plan) basis: the edge-aligned low-rank plan needs the third element, '
                               'model.Geometry(rel_pos, max_degree), as SE3Transformer.forward passes it (or set SE3B200_NO_ALIGNED=1)')
        st['lr'] = {}                            # images that do not fit this route: direct kernels for this forward
    if st['route'] == GLOBAL and len(st['lr']) < len(conv.pairs) and st['g'] is None:
        st['g'] = ops.radial_trunk(feat, pk['trunk'], len(conv.pairs))       # the direct kernels consume g itself
    return st


def edge_chunks(E, bytes_per_tile):
    """[(first tile, tiles, first edge, edges)] of the edge chunks whose workspace fits T_WORKSPACE_BYTES."""
    n_tiles = (E + ops.TILE_E - 1) // ops.TILE_E
    per_chunk = max(1, min(n_tiles, T_WORKSPACE_BYTES // bytes_per_tile))
    return [(t0, min(per_chunk, n_tiles - t0), t0 * ops.TILE_E, min(E - t0 * ops.TILE_E, per_chunk * ops.TILE_E))
            for t0 in range(0, n_tiles, per_chunk)]


def rotate_to_global(t, D, out):
    """Edge-aligned outputs back to the global frame: out [E, C, P] = D(e) t[e], t [E, P, C] component major, D [E, P, P]."""
    E, P, C = t.shape
    ops.fold_basis(t.reshape(1, E, P, C), D.reshape(-1), E, C, P, P, 1, out, accumulate=False, component_major=True, name='rotate_back')


def conv_forward(convs, inp, edge_info, rel_dist, basis, keep_aligned=False):
    """Evaluate one or more ConvSE3 that share input features, graph and fibers (to_k / to_v of an attention block): each
    takes its route (conv_route); the convolutions on one route share its per-chunk gathers."""
    forward_only_guard('ConvSE3', convs, list(inp.values()) + [rel_dist])
    idx, nmask, _ = edge_info
    E = idx.numel()
    if isinstance(basis, dict):
        raise TypeError("ConvSE3 takes the basis as the tuple (flat buffer, BasisPlan, Geometry) that SE3Transformer.forward builds: "
                        "`ops.basis_flat(rel_pos, max_degree) + (model.Geometry(rel_pos, max_degree),)`; the dict returned by the "
                        "drop-in get_basis() is the reference's per-pair view of the same buffer and is not accepted here")
    geom = basis[2] if len(basis) > 2 else None
    capturing = torch.cuda.is_current_stream_capturing()
    states = []
    for conv in convs:
        assert conv.pairs == convs[0].pairs and conv.in_dim == convs[0].in_dim
        states.append(conv_route(conv, E, edge_info, rel_dist, geom, capturing))
    routed = {route: [st for st in states if st['route'] == route] for route in (ZGEMM, ALIGNED, GLOBAL)}
    if routed[ZGEMM]:
        eval_zgemm(routed[ZGEMM], inp, idx, nmask, geom, keep_aligned)
    workspace = eval_aligned(routed[ALIGNED], inp, idx, geom) if routed[ALIGNED] else None
    if routed[GLOBAL]:
        eval_global(routed[GLOBAL], inp, idx, ops.basis_pairs(basis[0], basis[1], E), workspace)
    return [conv_outputs(st, inp, idx, nmask) for st in states]


def eval_zgemm(states, inp, idx, nmask, geom, keep_aligned):
    """Production path (DESIGN.md 4.5): neighbour features rotated into the edge frame once per input degree and chunk, then
    ONE tensor-core GEMM per (conv, degree_out, |m|) over all input degrees, then the rotation back to the global frame."""
    c0 = states[0]['conv']
    b, n, k = idx.shape
    E, dev = b * n * k, idx.device
    frames = geom.frames()
    sx = ops.edge_scale(inp, idx, max(di for di, _ in c0.fiber_in))
    chunks = edge_chunks(E, sum(mi * to_order(di) for di, mi in c0.fiber_in) * ops.TILE_E * 4)
    # pooled convolutions (conv_in / conv_out): masked mean over the neighbours + self-interaction fused into the rotate-back
    # (needs edge chunks that hold whole neighbour lists)
    fuse_pool = len(chunks) == 1 or (chunks[0][1] * ops.TILE_E) % k == 0
    for st in states:
        conv = st['conv']
        if conv.pool and fuse_pool:
            st['pooled'] = {do: torch.empty((b * n, mo, to_order(do)), dtype=torch.float32, device=dev) for do, mo in conv.fiber_out}
            st['self'] = conv.self_interact(inp) if conv.self_interaction else {}
        elif keep_aligned:                          # the consumer (attention) rotates back on the fly: keep out' itself
            st['aligned_out'] = {do: torch.empty((E, to_order(do), mo), dtype=torch.float32, device=dev) for do, mo in conv.fiber_out if do > 0}
    nmask_flat = None if nmask is None else nmask.reshape(-1)
    for t0, tc, e0, ec in chunks:
        X = {di: ops.rotgather(inp[str(di)], idx, frames.D[di] if di > 0 else None, t0, tc) for di, _ in c0.fiber_in}
        for st in states:
            conv = st['conv']
            for do, mo in conv.fiber_out:
                P = to_order(do)
                full = all((do, m) in st['z'] for m in range(do + 1))
                if do == 0 and 'pooled' not in st:
                    Op = st['outs'][0][e0:e0 + ec]                   # [ec, mo, 1] is [ec, 1, mo]
                elif do in st.get('aligned_out', {}):
                    Op = st['aligned_out'][do][e0:e0 + ec]
                    if not full:
                        Op.zero_()
                else:
                    Op = (torch.empty if full else torch.zeros)((ec, P, mo), dtype=torch.float32, device=dev)
                for m in range(do + 1):
                    zp = st['z'].get((do, m))
                    if zp is None:
                        continue
                    segs, alg = [], 0
                    for di, mi in zp['degs']:
                        pi = conv.pairs.index((di, do))
                        for kc in range(st['lr'][(di, do)]['Kp'] // 16):
                            segs.append((st['U'][pi, e0:e0 + ec, 16 * kc:], X[di], mi, to_order(di), di + m, di - m))
                        alg += ec * mo * mi * 2 * (ops.RADIAL_MID + P) * (1 if m == 0 else 2)
                    ops.zgemm(segs, zp['img'], sx[e0:e0 + ec], ec, mo, zp['mode'], Op, P * mo, [(do + m) * mo, (do - m) * mo],
                              alg_flops=alg, tag=f'mode{zp["mode"]}lo{do}m{m}Co{mo}S{zp["S"]}')
                if 'pooled' in st:                  # rotate back + masked mean over k + self-interaction, one kernel
                    sa = st['self'].get(str(do))
                    ops.rotate_pool(Op, frames.D[do][e0:e0 + ec] if do > 0 else None, None if nmask_flat is None else nmask_flat[e0:e0 + ec],
                                    None if sa is None else sa.reshape(b * n, mo, P)[e0 // k:(e0 + ec) // k], ec // k, k, mo, do,
                                    st['pooled'][do][e0 // k:(e0 + ec) // k])
                elif do > 0 and do not in st.get('aligned_out', {}):    # (aligned_out stays in the edge frame for the attention kernel)
                    rotate_to_global(Op, frames.D[do][e0:e0 + ec], st['outs'][do][e0:e0 + ec])
        del X


def tbuild_chunks(conv, E):
    """Edge chunks in which the largest T block of the R-first kernels fits the workspace."""
    return edge_chunks(E, max(ops.t_numel(1, mi, to_order(min(di, do)), to_order(do)) * 4
                              for di, mi in conv.fiber_in for do, _ in conv.fiber_out))


def eval_aligned(states, inp, idx, geom):
    """R-first edge-aligned formulation (DESIGN.md 4.4): neighbour features rotated into the edge frame per (degree_in, |m|)
    and chunk, two output components per launch, then the rotation back.  Returns the T workspace."""
    c0 = states[0]['conv']
    E, dev = idx.numel(), idx.device
    workspace = None
    for t0, tc, e0, ec in tbuild_chunks(c0, E):
        frames = geom.frames()
        # out' of degree do lives in one dense buffer per |m|: [edges, C_out] for m = 0, [edges, C_out, 2] = (+m, -m) otherwise
        # (the kernel's native layout); first contribution overwrites, later input degrees accumulate
        outp = [{} for _ in states]
        for di, mi in c0.fiber_in:
            for m in range(di + 1):
                targets = [(do, mo) for do, mo in c0.fiber_out if do >= m]
                if not targets:
                    continue
                Pk = Fk = 1 if m == 0 else 2
                workspace = ops.tbuild_blocks(inp[str(di)], idx, frames.block(di, m), Pk, Fk, t0, tc, out=workspace)
                for do, mo in targets:
                    pi = c0.pairs.index((di, do))
                    for st, op in zip(states, outp):
                        lrp = st['lr'][(di, do)]
                        first = (do, m) not in op
                        if first:
                            op[(do, m)] = st['outs'][do][e0:e0 + ec] if do == 0 else torch.empty((ec, mo, Pk), dtype=torch.float32, device=dev)
                        ops.pairwise_lr(st['U'][pi, e0:e0 + ec], lrp['al_imgs'][m], workspace, ec, mo, mi, Fk, Pk, lrp['Kp'], op[(do, m)],
                                        accumulate=not first, alg_units=Fk * 2 * (ops.RADIAL_MID + to_order(do)))
        for st, op in zip(states, outp):
            for do, mo in c0.fiber_out:
                if do > 0:                      # back to the global frame: out = D_lo out'
                    ops.rotate_back([op.get((do, m)) for m in range(do + 1)], frames.D[do][e0:e0 + ec].reshape(-1), ec, mo, do,
                                    st['outs'][do][e0:e0 + ec])
                elif (0, 0) not in op:
                    st['outs'][0][e0:e0 + ec].zero_()
        del outp
    return workspace


def eval_global(states, inp, idx, bpairs, workspace=None):
    """Per pair in the global frame (DESIGN.md 4.1-4.3): T = gather x basis once per (pair, chunk), then per convolution the
    low-rank kernel (output- or input-side contraction) or the direct K = 128 kernel."""
    c0 = states[0]['conv']
    E, dev = idx.numel(), idx.device
    for t0, tc, e0, ec in tbuild_chunks(c0, E):
        gathered = {}                            # degree_in -> neighbour features of this chunk in tile layout
        for do, mo in c0.fiber_out:
            P = to_order(do)
            first = True
            for di, mi in c0.fiber_in:
                Fq = to_order(min(di, do))
                Q = to_order(di)
                in_side = [input_side(di, do) and 'imgs_f' in st['lr'].get((di, do), {}) for st in states]
                if any(in_side) and di not in gathered:
                    gathered[di] = ops.gather_tiles(inp[str(di)], idx, t0, tc)
                if not all(in_side):
                    workspace = ops.tbuild(inp[str(di)], idx, bpairs[(di, do)], di, do, t0, tc, out=workspace)
                pi = c0.pairs.index((di, do))
                for st, ins in zip(states, in_side):
                    conv = st['conv']
                    out = st['outs'][do][e0:e0 + ec]
                    if ins:
                        # S[f,e,o,q] = sum_i R[e,o,i,f] x[j(e),i,q], then out[e,o,p] (+)= sum_{f,q} B[e,p,q,f] S[f,e,o,q]
                        lrp = st['lr'][(di, do)]
                        S = torch.empty((Fq, ec, mo, Q), dtype=torch.float32, device=dev)
                        for f in range(Fq):
                            ops.pairwise_lr(st['U'][pi, e0:e0 + ec], lrp['imgs_f'][f], gathered[di], ec, mo, mi, 1, Q, lrp['Kp'], S[f],
                                            accumulate=False, alg_P=P)
                        ops.fold_basis(S, bpairs[(di, do)][e0 * P * Q * Fq:(e0 + ec) * P * Q * Fq], ec, mo, P, Q, Fq, out,
                                       accumulate=not first)
                        del S
                    elif (di, do) in st['lr']:
                        lrp = st['lr'][(di, do)]
                        ops.pairwise_lr(st['U'][pi, e0:e0 + ec], lrp['img'], workspace, ec, mo, mi, Fq, P, lrp['Kp'], out,
                                        accumulate=not first)
                    elif st['tc_ok'][(di, do)]:
                        ops.pairwise_tc(st['g'][pi, e0:e0 + ec], conv.w3_image(di, do), workspace, ec, mo, mi, Fq, P,
                                        out, accumulate=not first)
                    else:
                        lin = conv.kernel_unary[f'({di},{do})'].rp.net['6']
                        ops.pairwise_simt(st['g'][pi, e0:e0 + ec], lin.weight, lin.bias, workspace, ec, mo, mi, Fq, P, out,
                                          accumulate=not first)
                first = False


def conv_outputs(st, inp, idx, nmask):
    """The result of one ConvSE3: pooled, AlignedKV or per-edge outputs, plus the self-interaction residual."""
    conv = st['conv']
    b, n, k = idx.shape
    if 'pooled' in st:
        return {str(do): st['pooled'][do].view(b, n, mo, to_order(do)) for do, mo in conv.fiber_out}
    outputs = {}
    for do, mo in conv.fiber_out:
        if do in st.get('aligned_out', {}):
            outputs[str(do)] = AlignedKV(st['aligned_out'][do].view(b, n, k, to_order(do), mo), do)
            continue
        o = st['outs'][do].view(b, n, k, mo, to_order(do))
        outputs[str(do)] = ops.pool(o, nmask) if conv.pool else o
    if conv.self_interaction:
        outputs = residual_add(outputs, conv.self_interact(inp))
    return outputs


class FeedForwardSE3(nn.Module):
    """reference S:347-365"""

    def __init__(self, fiber, mult=4):
        super().__init__()
        hidden = Fiber([(d, c * mult) for d, c in fiber])
        self.project_in = LinearSE3(fiber, hidden)
        self.nonlin = NormSE3(hidden)
        self.project_out = LinearSE3(hidden, fiber)

    def forward(self, x, residual=None):
        return self.project_out(self.nonlin(self.project_in(x)), residual=residual)


class FeedForwardBlockSE3(nn.Module):
    """reference S:367-383"""

    def __init__(self, fiber, norm_gated_scale=False):
        super().__init__()
        self.prenorm = NormSE3(fiber, gated_scale=norm_gated_scale)
        self.feedforward = FeedForwardSE3(fiber)

    def forward(self, x):
        return self.feedforward(self.prenorm(x), residual=x)          # residual added in the epilogue of project_out


class AttentionSE3(nn.Module):
    """AttentionSE3 (reference S:387-519) and, with one_headed=True, OneHeadedKVAttentionSE3 (S:522-654)."""

    def __init__(self, fiber, dim_head=64, heads=8, attend_self=False, edge_dim=None, fourier_encode_dist=False,
                 rel_dist_num_fourier_features=4, use_null_kv=False, splits=4, global_feats_dim=None, linear_proj_keys=False,
                 tie_key_values=False, one_headed=False):
        super().__init__()
        hidden_dim = dim_head * heads
        self.fiber = fiber
        hidden_fiber = Fiber([(d, hidden_dim) for d, _ in fiber])
        kv_fiber = Fiber([(d, dim_head) for d, _ in fiber]) if one_headed else hidden_fiber
        project_out = not (heads == 1 and len(fiber.dims) == 1 and dim_head == fiber.dims[0])
        self.scale = dim_head ** -0.5
        self.heads, self.dim_head, self.one_headed = heads, dim_head, one_headed
        self.linear_proj_keys = linear_proj_keys
        conv_kw = dict(edge_dim=default(edge_dim, 0), pool=False, self_interaction=False, fourier_encode_dist=fourier_encode_dist,
                       num_fourier_features=rel_dist_num_fourier_features, splits=splits)
        self.to_q = LinearSE3(fiber, hidden_fiber)
        self.to_v = ConvSE3(fiber, kv_fiber, **conv_kw)
        assert not (linear_proj_keys and tie_key_values), 'you cannot do linear projection of keys and have shared key / values turned on at the same time'
        if linear_proj_keys:
            self.to_k = LinearSE3(fiber, kv_fiber)
        elif not tie_key_values:
            self.to_k = ConvSE3(fiber, kv_fiber, **conv_kw)
        else:
            self.to_k = None
        self.to_out = LinearSE3(hidden_fiber, fiber) if project_out else nn.Identity()
        self.use_null_kv = use_null_kv
        if use_null_kv:
            self.null_keys = nn.ParameterDict()
            self.null_values = nn.ParameterDict()
            for degree in fiber.degrees:
                shape = (dim_head, to_order(degree)) if one_headed else (heads, dim_head, to_order(degree))
                self.null_keys[str(degree)] = nn.Parameter(torch.zeros(*shape))
                self.null_values[str(degree)] = nn.Parameter(torch.zeros(*shape))
        self.attend_self = attend_self
        if attend_self:
            self.to_self_k = LinearSE3(fiber, kv_fiber)
            self.to_self_v = LinearSE3(fiber, kv_fiber)
        self.accept_global_feats = exists(global_feats_dim)
        if self.accept_global_feats:
            gin = Fiber.create(1, global_feats_dim)
            gout = Fiber.create(1, kv_fiber[0])
            self.to_global_k = LinearSE3(gin, gout)
            self.to_global_v = LinearSE3(gin, gout)

    def forward(self, features, edge_info, rel_dist, basis, global_feats=None, pos_emb=None, mask=None, residual=None):
        forward_only_guard('AttentionSE3', [self], list(features.values()))
        idx, nmask, _ = edge_info
        queries = self.to_q(features)
        k_idx = None
        geom = basis[2] if isinstance(basis, tuple) and len(basis) > 2 else None
        fuse = geom is not None and not os.environ.get('SE3B200_NO_ATTN_ROTATE')    # rotate-back fused into the attention kernel
        if self.linear_proj_keys:
            values = conv_forward([self.to_v], features, edge_info, rel_dist, basis, keep_aligned=fuse)[0]
            keys = self.to_k(features)            # node level; the attention kernel gathers through idx
            k_idx = idx
        elif self.to_k is None:
            values = conv_forward([self.to_v], features, edge_info, rel_dist, basis, keep_aligned=fuse)[0]
            keys = values
        else:
            keys, values = conv_forward([self.to_k, self.to_v], features, edge_info, rel_dist, basis, keep_aligned=fuse)
        if self.attend_self:
            self_keys, self_values = self.to_self_k(features), self.to_self_v(features)
        if exists(global_feats):
            global_keys, global_values = self.to_global_k(global_feats), self.to_global_v(global_feats)
        if exists(pos_emb):
            # rotary embeddings on the type-0 queries / keys / values (reference S:488-494, 623-629; rotary.py:15-24): cheap
            # elementwise glue in torch around the attention kernel.  The key embedding has 1 + k positions, self first.
            assert self.attend_self, 'rotary embeddings need attend_self = True (the key positions include the node itself, as in the reference)'
            q_emb, k_emb = pos_emb                                     # [b, n, rot], [b, n, 1 + k, rot]
            b_, n_ = q_emb.shape[:2]
            Dh, hk = self.dim_head, (1 if self.one_headed else self.heads)
            queries = dict(queries)
            queries['0'] = apply_rotary_pos_emb(queries['0'].view(b_, n_, self.heads, Dh, 1), q_emb[:, :, None, :, None]).reshape(b_, n_, -1, 1)
            if k_idx is not None:                                      # linear_proj_keys: keys live on the nodes; rotary is per edge
                keys = dict(keys)
                keys['0'] = keys['0'][torch.arange(b_, device=idx.device)[:, None, None], idx]
            nb_emb, self_emb = k_emb[:, :, 1:, None, :, None], k_emb[:, :, 0, None, :, None]
            kk = idx.shape[-1]
            new_k = apply_rotary_pos_emb(keys['0'].view(b_, n_, kk, hk, Dh, 1), nb_emb).reshape(b_, n_, kk, -1, 1)
            new_v = new_k if values is keys else apply_rotary_pos_emb(values['0'].view(b_, n_, kk, hk, Dh, 1), nb_emb).reshape(b_, n_, kk, -1, 1)
            keys, values = dict(keys), dict(values)
            keys['0'], values['0'] = new_k, new_v
            self_keys, self_values = dict(self_keys), dict(self_values)
            self_keys['0'] = apply_rotary_pos_emb(self_keys['0'].view(b_, n_, hk, Dh, 1), self_emb).reshape(b_, n_, -1, 1)
            self_values['0'] = apply_rotary_pos_emb(self_values['0'].view(b_, n_, hk, Dh, 1), self_emb).reshape(b_, n_, -1, 1)
        outputs = {}
        for degree in features.keys():
            kw = {}
            if self.attend_self:
                kw.update(self_k=self_keys[degree], self_v=self_values[degree])
            if self.use_null_kv:
                kw.update(null_k=self.null_keys[degree].reshape(-1, to_order(int(degree))),
                          null_v=self.null_values[degree].reshape(-1, to_order(int(degree))))
            if exists(global_feats) and degree == '0':
                kw.update(global_k=global_keys[degree], global_v=global_values[degree])
            kd, vd = keys[degree], values[degree]
            if isinstance(vd, AlignedKV) or isinstance(kd, AlignedKV):
                if isinstance(kd, AlignedKV) and not isinstance(vd, AlignedKV):
                    kd = geom.to_global(kd)           # (keys and values come from the same dispatch: not reached in practice)
                if isinstance(vd, AlignedKV):
                    k_al = isinstance(kd, AlignedKV)
                    kw.update(D=geom.frames().D[int(degree)], k_aligned=k_al)
                    kd, vd = (kd.t if k_al else kd), vd.t
            outputs[degree] = ops.attention(queries[degree], kd, vd, heads=self.heads, dim_head=self.dim_head,
                                            scale=self.scale, nmask=nmask, k_idx=(None if exists(pos_emb) and degree == '0' else k_idx),
                                            kv_heads=1 if self.one_headed else self.heads, **kw)
        if isinstance(self.to_out, LinearSE3):
            return self.to_out(outputs, residual=residual)             # residual added in the epilogue of to_out
        return outputs if residual is None else residual_add(outputs, residual)


class SinusoidalEmbeddings(nn.Module):
    """reference rotary.py:5-13"""

    def __init__(self, dim):
        super().__init__()
        self.register_buffer('inv_freq', 1. / (10000 ** (torch.arange(0, dim, 2).float() / dim)))

    def forward(self, t):
        freqs = t[..., None].float() * self.inv_freq
        return freqs.repeat_interleave(2, dim=-1)                      # '... d -> ... (d r)', r = 2


def rotate_half(x):
    """reference rotary.py:15-18 on [..., d, m]: pairs (x1, x2) of consecutive channels -> cat(-x2, x1) along d (NOT re-interleaved)."""
    return torch.cat((-x[..., 1::2, :], x[..., 0::2, :]), dim=-2)


def apply_rotary_pos_emb(t, freqs):
    """reference rotary.py:20-24: t [..., d, m], freqs [..., rot, 1] (rot <= d leading channels are rotated)."""
    rot = freqs.shape[-2]
    tr, tp = t[..., :rot, :], t[..., rot:, :]
    return torch.cat((tr * freqs.cos() + rotate_half(tr) * freqs.sin(), tp), dim=-2)


class OneHeadedKVAttentionSE3(AttentionSE3):
    def __init__(self, fiber, **kwargs):
        super().__init__(fiber, one_headed=True, **kwargs)


class AttentionBlockSE3(nn.Module):
    """reference S:656-683"""

    def __init__(self, fiber, dim_head=24, heads=8, attend_self=False, edge_dim=None, use_null_kv=False, fourier_encode_dist=False,
                 rel_dist_num_fourier_features=4, splits=4, global_feats_dim=False, linear_proj_keys=False, tie_key_values=False,
                 attention_klass=AttentionSE3, norm_gated_scale=False):
        super().__init__()
        self.attn = attention_klass(fiber, heads=heads, dim_head=dim_head, attend_self=attend_self, edge_dim=edge_dim,
                                    use_null_kv=use_null_kv, rel_dist_num_fourier_features=rel_dist_num_fourier_features,
                                    fourier_encode_dist=fourier_encode_dist, splits=splits, global_feats_dim=global_feats_dim,
                                    linear_proj_keys=linear_proj_keys, tie_key_values=tie_key_values)
        self.prenorm = NormSE3(fiber, gated_scale=norm_gated_scale)

    def forward(self, features, edge_info, rel_dist, basis, global_feats=None, pos_emb=None, mask=None):
        return self.attn(self.prenorm(features), edge_info, rel_dist, basis, global_feats, pos_emb, mask, residual=features)


class SequentialSequence(nn.Module):
    """reference reversible.py:189-198"""

    def __init__(self, blocks):
        super().__init__()
        self.blocks = blocks

    def forward(self, x, **kwargs):
        for attn, ff in self.blocks:
            x = attn(x, **kwargs)
            x = ff(x)
        return x


def masked_mean_nodes(t, mask):
    """reference utils.py:72-80 over the node axis (return_pooled, S:1365-1367)."""
    m = mask[(..., *((None,) * (t.dim() - mask.dim())))]
    tot = mask.sum(dim=1)
    tot = tot[(..., *((None,) * (t.dim() - 1 - tot.dim())))]
    mean = t.masked_fill(~m, 0.).sum(dim=1) / tot.clamp(min=1.)
    return mean.masked_fill(tot == 0, 0.)


class SE3Transformer(nn.Module):
    """Drop-in for se3_transformer_pytorch.SE3Transformer (reference S:936-1375), inference on B200.

    Not carried over (raise NotImplementedError): reversible, use_egnn -- they are outside the hot path named by BASELINE.json
    (SURVEY.md section 2, "OUT OF SCOPE")."""

    def __init__(self, *, dim, heads=8, dim_head=24, depth=2, input_degrees=1, num_degrees=None, output_degrees=1,
                 valid_radius=1e5, reduce_dim_out=False, num_tokens=None, num_positions=None, num_edge_tokens=None, edge_dim=None,
                 reversible=False, attend_self=True, use_null_kv=False, differentiable_coors=False, fourier_encode_dist=False,
                 rel_dist_num_fourier_features=4, num_neighbors=float('inf'), attend_sparse_neighbors=False, num_adj_degrees=None,
                 adj_dim=0, max_sparse_neighbors=float('inf'), dim_in=None, dim_out=None, norm_out=False, num_conv_layers=0,
                 causal=False, splits=4, global_feats_dim=None, linear_proj_keys=False, one_headed_key_values=False,
                 tie_key_values=False, rotary_position=False, rotary_rel_dist=False, norm_gated_scale=False, use_egnn=False,
                 egnn_hidden_dim=32, egnn_weights_clamp_value=None, egnn_feedforward=False, hidden_fiber_dict=None,
                 out_fiber_dict=None):
        super().__init__()
        for flag, name in ((reversible, 'reversible'), (use_egnn, 'use_egnn')):
            if flag:
                raise NotImplementedError(f'{name}=True is outside the B200 hot path of this package')
        if differentiable_coors:
            raise NotImplementedError('differentiable_coors=True needs the backward pass; this package is forward only (SURVEY.md 8f row 4)')
        dim_in = default(dim_in, dim)
        self.dim_in = dim_in if isinstance(dim_in, tuple) else (dim_in,) * input_degrees
        self.dim = dim
        self.token_emb = nn.Embedding(num_tokens, dim) if exists(num_tokens) else None
        self.rotary_rel_dist, self.rotary_position = rotary_rel_dist, rotary_position      # reference S:998-1004
        self.rotary_pos_emb = None
        if rotary_position or rotary_rel_dist:
            self.rotary_pos_emb = SinusoidalEmbeddings(dim_head // (int(rotary_position) + int(rotary_rel_dist)))
        self.num_positions = num_positions
        self.pos_emb = nn.Embedding(num_positions, dim) if exists(num_positions) else None
        assert not (exists(num_edge_tokens) and not exists(edge_dim)), 'edge dimension (edge_dim) must be supplied if SE3 transformer is to have edge tokens'
        self.edge_emb = nn.Embedding(num_edge_tokens, edge_dim) if exists(num_edge_tokens) else None
        self.has_edges = exists(edge_dim) and edge_dim > 0
        self.input_degrees = input_degrees
        assert not (exists(num_adj_degrees) and num_adj_degrees < 1), 'make sure adjacent degrees is greater than 1'
        assert exists(num_degrees) or exists(hidden_fiber_dict), 'either num_degrees or hidden_fiber_dict must be specified'
        self.num_degrees = num_degrees if exists(num_degrees) else (max(hidden_fiber_dict.keys()) + 1)
        self.output_degrees = output_degrees
        self.differentiable_coors = differentiable_coors
        self.valid_radius = valid_radius
        self.num_neighbors = num_neighbors
        self.attend_sparse_neighbors = attend_sparse_neighbors
        self.max_sparse_neighbors = max_sparse_neighbors
        self.num_adj_degrees = num_adj_degrees
        self.adj_emb = nn.Embedding(num_adj_degrees + 1, adj_dim) if exists(num_adj_degrees) and adj_dim > 0 else None
        edge_dim = (edge_dim if self.has_edges else 0) + (adj_dim if exists(self.adj_emb) else 0)
        dim_out = default(dim_out, dim)
        fiber_in = Fiber.create(input_degrees, dim_in)
        fiber_hidden = Fiber(hidden_fiber_dict) if exists(hidden_fiber_dict) else Fiber.create(num_degrees, dim)
        if exists(out_fiber_dict):
            fiber_out = Fiber(out_fiber_dict)
            self.output_degrees = max(out_fiber_dict.keys()) + 1
        elif exists(output_degrees):
            fiber_out = Fiber.create(output_degrees, dim_out)
        else:
            fiber_out = None
        conv_kwargs = dict(edge_dim=edge_dim, fourier_encode_dist=fourier_encode_dist, num_fourier_features=rel_dist_num_fourier_features,
                           splits=splits)
        assert not (causal and not attend_self), 'attending to self must be turned on if in autoregressive mode (for the first token)'
        self.causal = causal
        self.conv_in = ConvSE3(fiber_in, fiber_hidden, **conv_kwargs)
        self.convs = nn.ModuleList([])
        for _ in range(num_conv_layers):
            self.convs.append(nn.ModuleList([ConvSE3(fiber_hidden, fiber_hidden, **conv_kwargs),
                                             NormSE3(fiber_hidden, gated_scale=norm_gated_scale)]))
        self.accept_global_feats = exists(global_feats_dim)
        self.attend_self = attend_self
        klass = OneHeadedKVAttentionSE3 if one_headed_key_values else AttentionSE3
        layers = nn.ModuleList([])
        for _ in range(depth):
            layers.append(nn.ModuleList([
                AttentionBlockSE3(fiber_hidden, heads=heads, dim_head=dim_head, attend_self=attend_self, edge_dim=edge_dim,
                                  fourier_encode_dist=fourier_encode_dist, rel_dist_num_fourier_features=rel_dist_num_fourier_features,
                                  use_null_kv=use_null_kv, splits=splits, global_feats_dim=global_feats_dim,
                                  linear_proj_keys=linear_proj_keys, attention_klass=klass, tie_key_values=tie_key_values,
                                  norm_gated_scale=norm_gated_scale),
                FeedForwardBlockSE3(fiber_hidden, norm_gated_scale=norm_gated_scale)]))
        self.net = SequentialSequence(layers)
        self.conv_out = ConvSE3(fiber_hidden, fiber_out, **conv_kwargs) if exists(fiber_out) else None
        self.norm = NormSE3(fiber_out, gated_scale=norm_gated_scale, nonlin=nn.Identity()) if norm_out and exists(fiber_out) else nn.Identity()
        final_fiber = default(fiber_out, fiber_hidden)
        self.linear_out = LinearSE3(final_fiber, Fiber([(d, 1) for d, _ in final_fiber])) if reduce_dim_out else None

    # ---- weights ----------------------------------------------------------------------------------------
    def conv_modules(self):
        return [m for m in self.modules() if isinstance(m, ConvSE3)]

    def pack_weights(self, free_master=False, max_distance=None):
        """Pre-build the tensor-core weight images of every ConvSE3 (otherwise done lazily on the first forward); see
        ConvSE3.pack_weights."""
        for m in self.conv_modules():
            m.pack_weights(free_master=free_master, max_distance=max_distance)
        return self

    def graphed(self, feats, coors, mask=None, **fwd_kwargs):
        """Capture one forward for these (static) input shapes in a CUDA graph and return a replayable callable
        (see GraphedForward).  Small point clouds are launch bound (~100 kernels of a few microseconds each); replaying a
        graph removes the per-launch host cost.  Not available with attend_sparse_neighbors / neighbor_mask (their
        host-side `.item()` synchronisations, reference S:1208, 1253, cannot be captured)."""
        return GraphedForward(self, feats, coors, mask, **fwd_kwargs)

    # ---- forward ----------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, feats, coors, mask=None, adj_mat=None, edges=None, return_type=None, return_pooled=False,
                neighbor_mask=None, global_feats=None):
        kw = dict(mask=mask, adj_mat=adj_mat, edges=edges, return_type=return_type, return_pooled=return_pooled,
                  neighbor_mask=neighbor_mask, global_feats=global_feats)
        out, checks = self._forward_once(feats, coors, **kw)
        if torch.cuda.is_current_stream_capturing():
            self._graph_checks = checks               # static tensors of the graph: GraphedForward reads them after each replay
            return out
        bad = check_lowrank_stats(checks)             # the one host synchronisation of the low-rank plans, once per forward
        if bad:
            self.handle_plan_miss(bad)
            out, checks = self._forward_once(feats, coors, **kw)
            assert not check_lowrank_stats(checks)
        return out

    @staticmethod
    def handle_plan_miss(bad):
        """The radial trunk outputs of a forward left the cached low-rank subspace of these ConvSE3 (distances beyond the plan's
        range): with released masters there is nothing to fall back to; otherwise they run on the direct kernels from now on."""
        if any(conv.free_master for conv in bad):
            raise LowRankPlanMiss('low-rank radial plan does not cover this input; pack_weights(max_distance=...) was given too small a distance')
        import warnings
        warnings.warn(f'{len(bad)} ConvSE3 left their low-rank radial plan (residual above {ConvSE3.LR_RUNTIME_TOL:g}): evaluating them with '
                      'the direct K = 128 kernels')
        for conv in bad:
            conv._lr_blocked = True

    def _forward_once(self, feats, coors, mask=None, adj_mat=None, edges=None, return_type=None, return_pooled=False,
                      neighbor_mask=None, global_feats=None):
        assert not (self.accept_global_feats ^ exists(global_feats)), 'you cannot pass in global features unless you init the class correctly'
        _mask = mask
        # float64 models / inputs (reference tests/test_equivariance.py:228-258 runs under a float64 default dtype): the kernels
        # compute in float32; parameters are converted once, inputs are cast, results are returned in the caller's dtype
        out_dtype = coors.dtype if coors.dtype == torch.float64 else None
        if any(p.dtype == torch.float64 for p in self.parameters()):
            import warnings
            warnings.warn('se3_transformer_pytorch_b200 computes in float32: converting the float64 parameters of this model to float32')
            self.float()
        if self.output_degrees == 1:
            return_type = 0
        if exists(self.token_emb):
            feats = self.token_emb(feats)
        if exists(self.pos_emb):
            assert feats.shape[1] <= self.num_positions, 'feature sequence length must be less than the number of positions given at init'
            feats = feats + self.pos_emb(torch.arange(feats.shape[1], device=feats.device)).unsqueeze(0)
        assert not (self.attend_sparse_neighbors and not exists(adj_mat)), 'adjacency matrix (adjacency_mat) or edges (edges) must be passed in'
        assert not (self.has_edges and not exists(edges)), 'edge embedding (num_edge_tokens & edge_dim) must be supplied if one were to train on edge types'
        if torch.is_tensor(feats):
            feats = {'0': feats[..., None]}
        if torch.is_tensor(global_feats):
            global_feats = {'0': global_feats[..., None]}
        if exists(global_feats):
            global_feats = {k: v.float() for k, v in global_feats.items()}
        if exists(edges) and edges.is_floating_point():
            edges = edges.float()
        b, n, d = feats['0'].shape[:3]
        device = feats['0'].device
        if not coors.is_cuda:
            raise RuntimeError('se3_transformer_pytorch_b200 runs on CUDA (sm_100a) only; move the model and inputs to the GPU')
        assert d == self.dim_in[0], f'feature dimension {d} must be equal to dimension given at init {self.dim_in[0]}'
        assert set(map(int, feats.keys())) == set(range(self.input_degrees)), f'input must have {self.input_degrees} degree'
        feats = {k: v.float().contiguous() for k, v in feats.items()}
        neighbors, max_sparse, valid_radius = self.num_neighbors, self.max_sparse_neighbors, self.valid_radius
        assert self.attend_sparse_neighbors or neighbors > 0, 'you must either attend to sparsely bonded neighbors, or set number of locally attended neighbors to be greater than 0'

        eye = torch.eye(n, dtype=torch.bool, device=device)
        adj_indices = None
        if exists(self.num_adj_degrees):                       # N-hop adjacency, reference S:1177-1191
            if adj_mat.dim() == 2:
                adj_mat = adj_mat.unsqueeze(0).expand(b, -1, -1).clone()
            adj_indices = adj_mat.clone().long()
            for ind in range(self.num_adj_degrees - 1):
                degree = ind + 2
                nxt = (adj_mat.float() @ adj_mat.float()) > 0
                nxt_mask = (nxt.float() - adj_mat.float()).bool()
                adj_indices = adj_indices.masked_fill(nxt_mask, degree)
                adj_mat = nxt.clone()

        sparse_mask = None
        num_sparse = 0
        if self.attend_sparse_neighbors:                       # reference S:1198-1217
            assert exists(adj_mat), 'adjacency matrix must be passed in (keyword argument adj_mat)'
            if adj_mat.dim() == 2:
                adj_mat = adj_mat.unsqueeze(0).expand(b, -1, -1)
            adj_vals = adj_mat.float().masked_fill(eye.unsqueeze(0), 0.)
            adj_max = int(adj_vals.sum(dim=-1).max().item())
            if max_sparse < adj_max:
                adj_vals = adj_vals + torch.empty_like(adj_vals).uniform_(-0.01, 0.01).masked_fill(eye.unsqueeze(0), 0.)
                adj_vals = adj_vals.masked_fill(eye.unsqueeze(0), -1.)
            num_sparse = int(min(max_sparse, adj_max))
            if num_sparse > 0:
                vals, inds = adj_vals.topk(num_sparse, dim=-1)
                sparse_mask = torch.zeros_like(adj_vals).scatter_(-1, inds, vals) > 0.5
            else:
                sparse_mask = torch.zeros_like(adj_vals, dtype=torch.bool)

        if neighbors == 0:
            valid_radius = 0
        k_local = int(min(neighbors, n - 1))
        total = int(k_local + num_sparse)
        assert total > 0, 'you must be fetching at least 1 neighbor'
        total = int(min(total, n - 1))
        if exists(neighbor_mask):
            max_nb = int(neighbor_mask.masked_fill(eye.unsqueeze(0), False).sum(dim=-1).max().item())
            if max_nb > neighbors:
                print(f'neighbor_mask shows maximum number of neighbors as {max_nb} but specified number of neighbors is {neighbors}')

        idx, nmask, rel_pos, rel_dist = ops.knn(coors.float(), total, valid_radius, node_mask=mask, neighbor_mask=neighbor_mask,
                                                sparse_adj=sparse_mask, causal=self.causal)

        # edge features on the neighbour list (reference S:1231-1239, 1293-1294); gather first, embed after
        e = None
        if exists(edges):
            if exists(self.edge_emb):
                if edges.dim() == 2:                            # [b, n] tokens: the reference broadcasts them over rows (b == 1)
                    assert b == 1, 'edges of shape [b, n] only broadcast for batch size 1 (as in the reference)'
                    edges = edges.unsqueeze(1).expand(b, n, n)
                e = self.edge_emb(edges.gather(2, idx))
            else:
                e = ops.gather_pairs(edges.float(), idx)
        if exists(self.adj_emb):
            a = self.adj_emb(adj_indices.gather(2, idx))
            e = torch.cat((e, a), dim=-1) if exists(e) else a

        geom = Geometry(rel_pos, self.num_degrees - 1)
        geom.deferred = []
        basis = ops.basis_flat(rel_pos, self.num_degrees - 1) + (geom,)
        edge_info = (idx, nmask, e)
        x = self.conv_in(feats, edge_info, rel_dist=rel_dist, basis=basis)
        for conv, nonlin in self.convs:
            x = nonlin(x)
            x = conv(x, edge_info, rel_dist=rel_dist, basis=basis)
        pos_emb = None
        if exists(self.rotary_pos_emb):                         # reference S:1298-1325
            q_parts, k_parts = [], []
            if self.rotary_position:
                seq_emb = self.rotary_pos_emb(torch.arange(n, device=device))                       # [n, d]
                with_self = torch.cat((torch.arange(n, device=device).view(1, n, 1).expand(b, n, 1), idx), dim=2)
                k_parts.append(seq_emb[with_self])                                                   # [b, n, 1 + k, d]
                q_parts.append(seq_emb.unsqueeze(0).expand(b, n, -1))
            if self.rotary_rel_dist:
                k_parts.append(self.rotary_pos_emb(F.pad(rel_dist, (1, 0), value=0.) * 1e2))
                q_parts.append(self.rotary_pos_emb(torch.zeros(n, device=device)).unsqueeze(0).expand(b, n, -1))
            pos_emb = (torch.cat(q_parts, dim=-1), torch.cat(k_parts, dim=-1))
        x = self.net(x, edge_info=edge_info, rel_dist=rel_dist, basis=basis, global_feats=global_feats, pos_emb=pos_emb, mask=_mask)
        if exists(self.conv_out):
            x = self.conv_out(x, edge_info, rel_dist=rel_dist, basis=basis)
        x = self.norm(x)
        if exists(self.linear_out):
            x = self.linear_out(x)
            x = {k: v.squeeze(dim=2) for k, v in x.items()}
        if return_pooled:
            x = {k: (masked_mean_nodes(v, _mask) if exists(_mask) else v.mean(dim=1)) for k, v in x.items()}
        if '0' in x:
            x['0'] = x['0'].squeeze(dim=-1)
        if exists(out_dtype):
            x = {k: v.to(out_dtype) for k, v in x.items()}
        if exists(return_type):
            return x[str(return_type)], geom.deferred
        return x, geom.deferred


class GraphedForward:
    """CUDA-graph replay of SE3Transformer.forward for fixed shapes.  Inputs are copied into static device buffers
    (host tensors are accepted: the copy is then the H2D transfer); the returned tensors are the graph's static outputs
    and are overwritten by the next call."""

    def __init__(self, model, feats, coors, mask=None, warmup=2, **fwd_kwargs):
        assert not model.attend_sparse_neighbors and fwd_kwargs.get('neighbor_mask') is None, \
            'graph capture needs a synchronisation-free forward'
        dev = next(model.parameters()).device
        self.model, self.kw = model, fwd_kwargs
        clone = lambda t: t.to(dev).clone()
        self.feats = {k: clone(v) for k, v in feats.items()} if isinstance(feats, dict) else clone(feats)
        self.coors = clone(coors)
        self.mask = None if mask is None else clone(mask)
        self.static_kw = {k: (clone(v) if torch.is_tensor(v) else v) for k, v in fwd_kwargs.items()}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):                    # builds weight images / tables outside the capture
                model(self.feats, self.coors, self.mask, **self.static_kw)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = model(self.feats, self.coors, self.mask, **self.static_kw)
        self.checks = model._graph_checks

    def __call__(self, feats, coors, mask=None, **tensor_kwargs):
        if isinstance(feats, dict):
            for k, v in feats.items():
                self.feats[k].copy_(v, non_blocking=True)
        else:
            self.feats.copy_(feats, non_blocking=True)
        self.coors.copy_(coors, non_blocking=True)
        if (mask is None) != (self.mask is None):
            raise ValueError('GraphedForward: `mask` must be given exactly when the graph was captured with one')
        if mask is not None:
            self.mask.copy_(mask, non_blocking=True)
        for k, v in tensor_kwargs.items():                # edges / adj_mat / global_feats captured as static buffers
            if not torch.is_tensor(self.static_kw.get(k)):
                raise ValueError(f'GraphedForward: {k} was not a tensor argument of the captured forward')
            self.static_kw[k].copy_(v, non_blocking=True)
        self.graph.replay()
        # the run-time check of the low-rank plans, read once per replay (the tensors are static outputs of the graph)
        bad = check_lowrank_stats(self.checks)
        if bad:
            raise LowRankPlanMiss('captured forward: the low-rank radial plan does not cover this input (distances beyond the range '
                                  'seen when the graph was captured); build a new graph or pack_weights(max_distance=...) for a larger range')
        return self.out
