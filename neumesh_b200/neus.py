"""``NeuS`` - drop-in for the distillation teacher ``models/frameworks/neus/neus.py`` (``ImplicitSurface`` /
``RadianceNet`` of ``models/base.py:139-311,363-440``): same constructor arguments, same ``state_dict`` keys, same
method protocol (``forward``, ``forward_radiance``, ``forward_density_only``, ``forward_with_nablas``, ``forward_s``).

The trainer evaluates the teacher under ``torch.no_grad()`` at the 127 mid-points of every training ray
(``models/trainer.py:211-219``) - an 8 x 256 skip-MLP whose normals the reference obtains with ``autograd.grad``.  On CUDA
with grad mode off that evaluation runs on this library's kernels:

* every ``Linear`` is one ``nmb_tr_gemm`` (hand-written SGEMM, ``csrc/train.cu``) over FOUR stacked row blocks - the
  value rows and the three forward-mode tangent rows d/dx, d/dy, d/dz (same weights, no bias) - so the normals come out
  of the same pass, with no autograd graph;
* ``nmb_tr_softplus_fwd`` applies softplus(beta = 100) to the value rows and softplus' * (W t) to each tangent block;
* the radiance net runs with the fused ReLU epilogue.

Grad-enabled calls (not used by the reference's trainer for the teacher) follow the torch-op path, which is also the
specification of the fused one."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
from torch import autograd

from .neumesh import get_embedder


class DenseLayer(nn.Linear):
    def __init__(self, input_dim, out_dim, *args, activation=None, **kwargs):
        super().__init__(input_dim, out_dim, *args, **kwargs)
        self.activation = nn.ReLU(inplace=True) if activation is None else activation

    def forward(self, x):
        return self.activation(super().forward(x))


def _eff_weight(layer):
    """Effective weight of a (possibly weight-normed) Linear."""
    if hasattr(layer, "weight_g"):
        return torch._weight_norm(layer.weight_v, layer.weight_g, 0)
    return layer.weight


class ImplicitSurface(nn.Module):
    def __init__(self, W=256, D=8, skips=(4,), W_geo_feat=256, input_ch=3, radius_init=1.0, obj_bounding_size=2.0,
                 geometric_init=True, embed_multires=6, weight_norm=True, use_siren=False):
        super().__init__()
        if use_siren:
            raise NotImplementedError("SIREN surfaces are outside the teacher configurations of the reference's configs")
        self.radius_init = radius_init
        self.register_buffer("obj_bounding_size", torch.tensor([obj_bounding_size]).float())
        self.geometric_init, self.D, self.W, self.W_geo_feat = geometric_init, D, W, W_geo_feat
        self.skips, self.use_siren = list(skips), use_siren
        self.embed_fn, input_ch = get_embedder(embed_multires)
        self.embed_multires = embed_multires
        self.input_ch = input_ch
        layers = []
        for l in range(D + 1):
            if l == D:
                out_dim = 1 + W_geo_feat if W_geo_feat > 0 else 1
            elif (l + 1) in self.skips:
                out_dim = W - input_ch
            else:
                out_dim = W
            in_dim = input_ch if l == 0 else W
            layer = DenseLayer(in_dim, out_dim, activation=nn.Softplus(beta=100)) if l != D else nn.Linear(in_dim, out_dim)
            if geometric_init:   # sphere initialisation as in SAL / IDR (models/base.py:222-250)
                if l == D:
                    nn.init.normal_(layer.weight, mean=np.sqrt(np.pi) / np.sqrt(in_dim), std=0.0001)
                    nn.init.constant_(layer.bias, -radius_init)
                elif embed_multires > 0 and l == 0:
                    nn.init.constant_(layer.bias, 0.0)
                    nn.init.constant_(layer.weight[:, 3:], 0.0)
                    nn.init.normal_(layer.weight[:, :3], 0.0, np.sqrt(2) / np.sqrt(out_dim))
                elif embed_multires > 0 and l in self.skips:
                    nn.init.constant_(layer.bias, 0.0)
                    nn.init.normal_(layer.weight, 0.0, np.sqrt(2) / np.sqrt(out_dim))
                    nn.init.constant_(layer.weight[:, -(input_ch - 3):], 0.0)
                else:
                    nn.init.constant_(layer.bias, 0.0)
                    nn.init.normal_(layer.weight, 0.0, np.sqrt(2) / np.sqrt(out_dim))
            if weight_norm:
                layer = nn.utils.weight_norm(layer)
            layers.append(layer)
        self.surface_fc_layers = nn.ModuleList(layers)

    def forward(self, x, return_h=False):
        x = self.embed_fn(x)
        h = x
        for i in range(self.D):
            if i in self.skips:
                h = torch.cat([h, x], dim=-1) / np.sqrt(2)
            h = self.surface_fc_layers[i](h)
        out = self.surface_fc_layers[-1](h)
        if self.W_geo_feat > 0:
            h = out[..., 1:]
            out = out[..., :1].squeeze(-1)
        else:
            out = out.squeeze(-1)
        return (out, h) if return_h else out

    def forward_with_nablas(self, x, has_grad_bypass=None):
        has_grad = torch.is_grad_enabled() if has_grad_bypass is None else has_grad_bypass
        if not has_grad and x.is_cuda and _fused_ok(self):
            return _fused_surface(self, x)
        with torch.enable_grad():
            x = x.requires_grad_(True)
            val, h = self.forward(x, return_h=True)
            nabla = autograd.grad(val, x, torch.ones_like(val), create_graph=has_grad, retain_graph=has_grad,
                                  only_inputs=True)[0]
        if not has_grad:
            val, nabla, h = val.detach(), nabla.detach(), h.detach()
        return val, nabla, h


class RadianceNet(nn.Module):
    def __init__(self, D=4, W=256, skips=(), W_geo_feat=256, embed_multires=6, embed_multires_view=4, use_view_dirs=True,
                 weight_norm=True, use_siren=False):
        super().__init__()
        if use_siren:
            raise NotImplementedError("SIREN radiance nets are outside the teacher configurations of the reference")
        self.skips, self.D, self.W, self.use_view_dirs = list(skips), D, W, use_view_dirs
        self.embed_fn, ch_pts = get_embedder(embed_multires)
        if use_view_dirs:
            self.embed_fn_view, ch_views = get_embedder(embed_multires_view)
            in0 = ch_pts + ch_views + 3 + W_geo_feat
        else:
            in0 = ch_pts + W_geo_feat
        self.in_dim_0 = in0
        layers = []
        for l in range(D + 1):
            out_dim = 3 if l == D else W
            in_dim = in0 if l == 0 else (in0 + W if l in self.skips else W)
            layer = DenseLayer(in_dim, out_dim, activation=nn.ReLU(inplace=True)) if l != D else \
                DenseLayer(in_dim, out_dim, activation=nn.Sigmoid())
            if weight_norm:
                layer = nn.utils.weight_norm(layer)
            layers.append(layer)
        self.layers = nn.ModuleList(layers)

    def _input(self, x, view_dirs, normals, geometry_feature):
        x = self.embed_fn(x)
        if self.use_view_dirs:
            return torch.cat([x, self.embed_fn_view(view_dirs), normals, geometry_feature], dim=-1)
        return torch.cat([x, geometry_feature], dim=-1)

    def forward(self, x, view_dirs, normals, geometry_feature):
        inp = self._input(x, view_dirs, normals, geometry_feature)
        if not torch.is_grad_enabled() and inp.is_cuda and not self.skips:
            return _fused_radiance(self, inp)
        h = inp
        for i in range(self.D + 1):
            if i in self.skips:
                h = torch.cat([h, inp], dim=-1)
            h = self.layers[i](h)
        return h


class NeuS(nn.Module):
    def __init__(self, variance_init=0.05, speed_factor=1.0, input_ch=3, W_geo_feat=-1, use_outside_nerf=False,
                 obj_bounding_radius=1.0, surface_cfg=None, radiance_cfg=None):
        super().__init__()
        if use_outside_nerf:
            raise NotImplementedError("the NeRF++ background of the mask-free NeuS setting is out of scope (DESIGN.md)")
        self.ln_s = nn.Parameter(torch.Tensor([-np.log(variance_init) / speed_factor]), requires_grad=True)
        self.speed_factor = speed_factor
        self.implicit_surface = ImplicitSurface(W_geo_feat=W_geo_feat, input_ch=input_ch,
                                                obj_bounding_size=obj_bounding_radius, **(surface_cfg or {}))
        if W_geo_feat < 0:
            W_geo_feat = self.implicit_surface.W
        self.radiance_net = RadianceNet(W_geo_feat=W_geo_feat, **(radiance_cfg or {}))

    def forward_radiance(self, x, view_dirs):
        _, nablas, feat = self.implicit_surface.forward_with_nablas(x)
        return self.radiance_net.forward(x, view_dirs, nablas, feat)

    def forward_s(self):
        return torch.exp(self.ln_s * self.speed_factor)

    def forward(self, x, view_dirs):
        sdf, nablas, feat = self.implicit_surface.forward_with_nablas(x)
        return sdf, self.radiance_net.forward(x, view_dirs, nablas, feat)

    def forward_density_only(self, x):
        return self.implicit_surface.forward(x)

    def forward_with_nablas(self, x, has_grad_bypass=None):
        return self.implicit_surface.forward_with_nablas(x, has_grad_bypass)[:2]


# ------------------------------------------------------------------------------------------------------------------
# fused no-grad evaluation on the library's kernels
# ------------------------------------------------------------------------------------------------------------------
def _fused_ok(surface: ImplicitSurface) -> bool:
    return surface.W_geo_feat > 0 and surface.embed_multires >= 0 and all(
        isinstance(l, nn.Linear) for l in surface.surface_fc_layers)


def _embed_with_jacobian(x, L):
    """PE(x) [M, 3(1+2L)] and its three directional derivatives d/dx_j [3, M, 3(1+2L)] (base.py:52-70 ordering)."""
    M = x.shape[0]
    cols, jac = [x], [torch.eye(3, device=x.device).expand(M, 3, 3)]           # jac[..., j, c] = d col c / d x_j
    for k in range(L):
        f = 2.0 ** k
        s, c = torch.sin(x * f), torch.cos(x * f)
        cols += [s, c]
        jac += [torch.diag_embed(f * c), torch.diag_embed(-f * s)]
    return torch.cat(cols, -1), torch.cat(jac, -1).permute(1, 0, 2).contiguous()


def _fused_surface(surf: ImplicitSurface, x):
    """-> (sdf [...], nabla [...,3], feature [...,W_geo]) by value + 3 tangent row blocks through the library's GEMMs."""
    from . import train_ops
    lead = x.shape[:-1]
    flat = x.detach().reshape(-1, 3).float().contiguous()
    M, dev = flat.shape[0], flat.device
    P = train_ops.CudaPrims(dev)
    L = max(surf.embed_multires, 0)
    emb, jac = _embed_with_jacobian(flat, L)                   # [M, C], [3, M, C]
    # rows [0, M): values; [M, 2M), [2M, 3M), [3M, 4M): tangents w.r.t. x, y, z
    X0 = torch.cat([emb[None], jac], 0).reshape(4 * M, -1).contiguous()
    H = X0
    inv_sqrt2 = 1.0 / np.sqrt(2)
    for i in range(surf.D):
        if i in surf.skips:
            H = (torch.cat([H, X0], dim=-1) * inv_sqrt2).contiguous()
        lin = surf.surface_fc_layers[i]
        Wt = _eff_weight(lin).detach().float().contiguous()
        N, K = Wt.shape
        Z = torch.empty(4 * M, N, device=dev)
        # one GEMM for the four row blocks; the bias belongs to the value rows only
        P.gemm(H, H.shape[1], True, Wt, K, True, Z, N, 4 * M, N, K)
        Z[:M] += lin.bias.detach().float()
        Hn = torch.empty(4 * M, N, device=dev)
        scratch = torch.empty(M, N, device=dev)
        for j in range(3):     # value rows are (re)written by each call with identical values
            P.softplus_fwd(Z[:M], Z[(j + 1) * M:(j + 2) * M], Hn[:M] if j == 0 else scratch, Hn[(j + 1) * M:(j + 2) * M])
        H = Hn
    lin = surf.surface_fc_layers[-1]
    Wt = lin.weight.detach().float().contiguous() if not hasattr(lin, "weight_g") else _eff_weight(lin).detach().float().contiguous()
    N, K = Wt.shape
    Z = torch.empty(4 * M, N, device=dev)
    P.gemm(H, H.shape[1], True, Wt, K, True, Z, N, 4 * M, N, K)
    Z[:M] += lin.bias.detach().float()
    sdf = Z[:M, 0]
    nabla = torch.stack([Z[M:2 * M, 0], Z[2 * M:3 * M, 0], Z[3 * M:, 0]], dim=-1)
    feat = Z[:M, 1:]
    return sdf.reshape(lead), nabla.reshape(*lead, 3), feat.reshape(*lead, N - 1)


def _fused_surface_value(surf: ImplicitSurface, x):
    """-> sdf [M] of flat points x [M,3]: the value row block of ``_fused_surface`` alone (no tangent rows, no feature
    columns), for dense grids where only the sdf is kept.  Each hidden layer is one ``nmb_tr_gemm`` with the bias +
    softplus(beta = 100) epilogue, which computes the same fp32 operations as ``_fused_surface``'s value rows, so the
    two agree bit for bit; every row is independent, so the result does not depend on how the caller chunks x."""
    from . import train_ops
    flat = x.detach().reshape(-1, 3).float().contiguous()
    M, dev = flat.shape[0], flat.device
    P = train_ops.CudaPrims(dev)
    cols = [flat]
    for k in range(max(surf.embed_multires, 0)):        # the value columns of _embed_with_jacobian, same operations
        f = 2.0 ** k
        cols += [torch.sin(flat * f), torch.cos(flat * f)]
    X0 = torch.cat(cols, -1).contiguous()
    H = X0
    inv_sqrt2 = 1.0 / np.sqrt(2)
    for i in range(surf.D):
        if i in surf.skips:
            H = (torch.cat([H, X0], dim=-1) * inv_sqrt2).contiguous()
        lin = surf.surface_fc_layers[i]
        Wt = _eff_weight(lin).detach().float().contiguous()
        N, K = Wt.shape
        Z = torch.empty(M, N, device=dev)
        P.gemm(H, H.shape[1], True, Wt, K, True, Z, N, M, N, K, bias=lin.bias.detach().float().contiguous(), epilogue=3)
        H = Z
    lin = surf.surface_fc_layers[-1]
    Wt = _eff_weight(lin).detach().float()[:1].contiguous()     # row 0 is the sdf; the rest is the geometry feature
    K = Wt.shape[1]
    sdf = torch.empty(M, 1, device=dev)
    P.gemm(H, H.shape[1], True, Wt, K, True, sdf, 1, M, 1, K, bias=lin.bias.detach().float()[:1].contiguous())
    return sdf.reshape(M)


def _fused_radiance(net: RadianceNet, inp):
    from . import train_ops
    lead = inp.shape[:-1]
    H = inp.detach().reshape(-1, inp.shape[-1]).float().contiguous()
    M, dev = H.shape[0], H.device
    P = train_ops.CudaPrims(dev)
    for i in range(net.D + 1):
        lin = net.layers[i]
        Wt = _eff_weight(lin).detach().float().contiguous()
        N, K = Wt.shape
        Z = torch.empty(M, N, device=dev)
        P.gemm(H, H.shape[1], True, Wt, K, True, Z, N, M, N, K, bias=lin.bias.detach().float().contiguous(),
               epilogue=1 if i < net.D else 0)
        H = Z
    return torch.sigmoid(H).reshape(*lead, 3)
