"""Generalised linear model shards with a low-precision, HBM-resident design matrix.

Workloads from ``/root/repo/BASELINE.json`` (not present in the reference, whose only model is
the 10-point linear regression): *federated logistic GLM, 10M rows x 256 features per shard,
bf16 design matrix* and *hierarchical GLM, 8 partial-pooling groups, fp8 block-scaled design
matrix*.  ``theta = [intercept[G], beta[P]]`` (float32) per chain; a segment (shard) uses
``intercept[group]``, so G = 1 is the pooled GLM and G = #shards the partial-pooling one.
Result per chain: ``[LL, dLL/dintercept[G], dLL/dbeta[P]]`` (float64).

The families with fitted parameters (``normal``, ``student_t``, ``negative_binomial``) append their D
parameters phi: ``theta = [intercept[G], beta[P], phi[D]]`` and ``[LL, d intercept[G], d beta[P], d phi[D]]``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from .base import ShardModel

FAMILIES = {"logistic": 0, "poisson": 1, "gaussian": 2, "normal": 3, "student_t": 4, "negative_binomial": 5}

#: Families whose parameters phi are inferred along with the coefficients (tensor-core kernel only).  They are
#: fully normalised: the log-likelihood equals the scipy log density summed over the rows —
#: ``norm.logpdf(y, eta, sigma)``, ``t.logpdf(y, nu, eta, sigma)`` and, with ``mu = exp(eta)``,
#: ``nbinom.logpmf(y, alpha, alpha / (alpha + mu))`` (NB2, ``var = mu + mu^2 / alpha``, PyMC's
#: ``NegativeBinomial(mu, alpha)``).  ``gaussian`` keeps its unit variance.
FAMILY_PARAMS = {"normal": ("sigma",), "student_t": ("sigma", "nu"), "negative_binomial": ("alpha",)}

_TC_SHAPES = "bf16 design matrix, P % 8 == 0, 8 <= P <= 384, K <= 16 chains, 16-byte aligned rows"


def _family_code(family) -> int:
    return family.code_id if hasattr(family, "code_id") else FAMILIES[family]


class GlmShards(ShardModel):
    """The GLM segments that live on ONE GPU.

    Parameters
    ----------
    Xs, ys
        Per-segment design matrices ``[n_rows, P]`` (bf16, row-major) and responses ``[n_rows]``
        (float32).
    groups
        Intercept index of every segment.
    n_groups
        Total number of intercepts G in the federation.
    n_chains
        Parameter vectors evaluated per call (K).  ``K > 1`` needs the tensor-core kernel.
    family
        ``"logistic"``, ``"poisson"``, ``"gaussian"`` (unit variance), or one of the families with fitted
        parameters (:data:`FAMILY_PARAMS`): ``"normal"`` (sigma), ``"student_t"`` (sigma, nu) and
        ``"negative_binomial"`` (alpha).  These take a third input ``phi`` and return ``d_phi``; they run on the
        tensor-core kernel only.  A :class:`~pytensor_federated_b200.models.custom.CustomFamily` is accepted too.
    kernel
        ``"simt"`` (one chain, any P % 8 == 0 up to 512), ``"tc"`` (tcgen05 + TMA: bf16, any P % 8 == 0 up to
        384 — the tile is padded to whole 128-feature blocks by TMA's zero fill —, up to 16 chains) or ``"auto"``.
    node_ids, n_nodes
        Keep the result PER NODE instead of summed: segment ``s`` is (part of) node ``node_ids[s]`` of
        an ``n_nodes`` federation and the reduced vector holds one ``[K][1 + G + P]`` block per node
        (every kernel: the tensor-core kernels route a chunk's sums to its node's block, the CUDA-core kernels flush
        at node boundaries into fixed-point accumulators).  ``evaluate`` still returns the sum; :meth:`per_node` and
        :class:`~pytensor_federated_b200.federation.NodeFederation` expose the blocks — the reference's
        one-Op-per-node pattern (``/root/reference/demo_model.py:28-36``) answered by one launch.
    """

    def __init__(
        self,
        Xs: Sequence,
        ys: Sequence,
        *,
        groups: Optional[Sequence[int]] = None,
        n_groups: int = 1,
        family: str = "logistic",
        n_chains: int = 1,
        kernel: str = "auto",
        scales: Optional[Sequence] = None,
        node_ids: Optional[Sequence[int]] = None,
        n_nodes: Optional[int] = None,
    ) -> None:
        import torch

        if len(Xs) != len(ys):
            raise ValueError("Xs and ys must have the same length")
        self.Xs = list(Xs)
        self.ys = [y.to(torch.float32).contiguous() for y in ys]
        self.scales = list(scales) if scales is not None else None
        self.groups = list(groups) if groups is not None else [0] * len(Xs)
        self.n_groups = int(n_groups)
        self.family = family
        self.n_chains = int(n_chains)
        self.kernel = kernel
        X0 = self.Xs[0]
        self.n_features = int(X0.shape[1])
        self.ld = int(X0.stride(0))
        for X in self.Xs:
            if X.dim() != 2 or X.shape[1] != self.n_features or X.stride(1) != 1 or X.stride(0) != self.ld:
                raise ValueError("all design matrices must be row-major [n, P] with one row stride")
        self.device = X0.device
        #: names of the fitted family parameters phi, e.g. ``("sigma", "nu")`` (empty for the other families)
        self.family_param_names = FAMILY_PARAMS.get(family, ()) if isinstance(family, str) else ()
        self.n_family_params = len(self.family_param_names)
        if family == "negative_binomial":
            for y in self.ys:
                if y.numel() and not bool(((y >= 0) & (y == torch.floor(y))).all()):
                    raise ValueError("negative_binomial needs non-negative integer counts y")
        self.n_inputs = 3 if self.n_family_params else 2
        self.n_params = self.n_groups + self.n_features + self.n_family_params
        self.n_theta_words = self.n_chains * self.n_params
        if (node_ids is None) != (n_nodes is None):
            raise ValueError("node_ids and n_nodes come together")
        self.node_ids = list(node_ids) if node_ids is not None else None
        self.n_nodes = int(n_nodes) if n_nodes is not None else 1
        if self.node_ids is not None and (len(self.node_ids) != len(self.Xs) or not all(0 <= i < self.n_nodes for i in self.node_ids)):
            raise ValueError("node_ids needs one node index in [0, n_nodes) per segment")
        self.n_vals = self.n_nodes * self.n_chains * (1 + self.n_params)

    @property
    def n_rows(self) -> int:
        return int(sum(X.shape[0] for X in self.Xs))

    # -- packing ---------------------------------------------------------------------------
    def call_context(self, inputs):
        """``(batched, intercept shape)`` of one call: a 2-D ``beta`` means one row per chain."""
        intercept, beta = inputs[0], inputs[1]
        return (np.ndim(beta) == 2, np.shape(intercept))

    def _split_inputs(self, inputs):
        """``(intercept, beta, phi or None)``, checking the number of inputs against the family."""
        if len(inputs) != self.n_inputs:
            want = "(intercept, beta, phi)" if self.n_family_params else "(intercept, beta)"
            raise ValueError(f"the {self.family!s} GLM takes {self.n_inputs} inputs {want}, got {len(inputs)}")
        return inputs[0], inputs[1], (inputs[2] if self.n_family_params else None)

    def _check_phi(self, phi) -> np.ndarray:
        ph = np.asarray(phi, dtype=np.float64).reshape(self.n_chains, self.n_family_params)
        if not np.all(np.isfinite(ph) & (ph > 0)):
            raise ValueError(f"family parameters {self.family_param_names} must be finite and > 0, got {ph.tolist()}")
        return ph

    _pack_views = None

    def pack_theta(self, inputs, out: np.ndarray):
        intercept, beta, phi = self._split_inputs(inputs)
        views = self._pack_views
        if views is None or views[0] is not out:
            # float32 windows into the staging buffer, built once per buffer (this runs on every evaluation)
            th = out.view(np.float32).reshape(self.n_chains, self.n_params)
            G, GP = self.n_groups, self.n_groups + self.n_features
            views = self._pack_views = (out, th[:, :G], th[:, G:GP], th[:, GP:])
        ic = intercept if type(intercept) is np.ndarray else np.asarray(intercept)
        bt = beta if type(beta) is np.ndarray else np.asarray(beta)
        batched = bt.ndim == 2
        ctx = (batched, ic.shape)
        if phi is not None:
            ph = self._check_phi(phi)   # before anything is written: a rejected call leaves the buffer alone
        self._batched, self._icpt_shape = ctx
        # the assignments convert to float32 while they copy
        views[1][...] = ic.reshape(self.n_chains, -1) if batched else ic.reshape(1, -1)
        views[2][...] = bt.reshape(self.n_chains, self.n_features)
        if phi is not None:
            views[3][...] = ph
        return ctx

    _batched = False
    _icpt_shape = ()

    def _note_shapes(self, inputs):
        # single-threaded convenience state (tests call reference_partial then unpack_result);
        # the engine passes the context explicitly instead
        ctx = self.call_context(inputs)
        self._batched, self._icpt_shape = ctx
        return ctx

    def per_node(self, vals: np.ndarray) -> np.ndarray:
        """The reduced vector as ``[n_nodes, n_chains, 1 + G + P + D]`` (``[LL, d intercepts, d beta, d phi]`` per block)."""
        return np.asarray(vals, dtype=np.float64).reshape(self.n_nodes, self.n_chains, 1 + self.n_params)

    def unpack_result(self, vals: np.ndarray, ctx=None) -> List[np.ndarray]:
        v = self.per_node(vals).sum(axis=0) if self.n_nodes > 1 else np.asarray(vals, dtype=np.float64).reshape(self.n_chains, 1 + self.n_params)
        G, GP = self.n_groups, self.n_groups + self.n_features
        batched, icpt_shape = ctx if ctx is not None else (self._batched, self._icpt_shape)
        if batched:
            out = [v[:, 0].copy(), v[:, 1 : 1 + G].reshape((self.n_chains,) + tuple(icpt_shape[1:])).copy(),
                   v[:, 1 + G : 1 + GP].copy()]
            return out + [v[:, 1 + GP :].copy()] if self.n_family_params else out
        out = [np.asarray(v[0, 0]), v[0, 1 : 1 + G].reshape(icpt_shape).copy(), v[0, 1 + G : 1 + GP].copy()]
        return out + [v[0, 1 + GP :].copy()] if self.n_family_params else out

    # -- native ----------------------------------------------------------------------------
    def use_tensor_cores(self):
        """Kernel selector passed to the runtime: 0 = SIMT, 1 = tcgen05 (bf16), 2 = block-scaled fp8,
        3 / 4 = general-shape fallback (bf16 / fp32 design matrix)."""
        import torch

        X0 = self.Xs[0]
        tc_ok = (X0.dtype == torch.bfloat16 and self.n_features % 8 == 0 and 8 <= self.n_features <= 384
                 and self.n_chains <= 16 and all(X.data_ptr() % 16 == 0 for X in self.Xs) and self.ld % 8 == 0)
        if self.n_family_params:
            # the families with fitted parameters exist on the tensor-core kernel only
            if self.kernel not in ("tc", "auto") or not tc_ok:
                raise ValueError(f"the {self.family} family runs on the tensor-core kernel only ({_TC_SHAPES}); "
                                 f"kernel={self.kernel!r}, dtype {X0.dtype}, P = {self.n_features}, K = {self.n_chains}")
            return 1
        if hasattr(self.family, "code_id"):  # user-compiled likelihood: general-shape kernel
            if X0.dtype not in (torch.bfloat16, torch.float32) or self.n_chains != 1 or self.n_features > 1024:
                raise ValueError("custom likelihoods need a bf16/fp32 design matrix, one chain and P <= 1024")
            return 3 if X0.dtype == torch.bfloat16 else 4
        if self.kernel == "fp8":
            return 2
        if self.kernel == "tc":
            return 1
        if self.kernel == "simt":
            return 0
        generic = 3 if X0.dtype == torch.bfloat16 else (4 if X0.dtype == torch.float32 else None)
        if self.kernel == "generic":
            if generic is None:
                raise ValueError("the general-shape kernel needs a bf16 or fp32 design matrix")
            return generic
        # auto: the tcgen05 kernel wherever its shape constraints hold (it is faster even for one chain:
        # TMA streaming + the X tile reused from smem for both GEMMs), then SIMT, then the general kernel
        bf16 = X0.dtype == torch.bfloat16
        if tc_ok:
            return 1
        if self.n_chains > 1:
            raise ValueError("multi-chain evaluation needs the tensor-core kernel (bf16, P % 8 == 0, P <= 384, K <= 16)")
        simt_ok = (bf16 and self.n_features % 8 == 0 and self.n_features <= 512 and self.ld % 8 == 0
                   and all(X.data_ptr() % 16 == 0 for X in self.Xs))
        if simt_ok:
            return 0
        if generic is not None and self.n_features <= 1024:
            return generic
        raise ValueError(f"no fused GLM kernel for dtype {X0.dtype} with {self.n_features} features; "
                         "serve this model through ArraysToArraysService instead")

    def attach(self, lib, handle) -> None:
        from ..ops import native

        n = len(self.Xs)
        Xp = native.void_p_array([X.data_ptr() for X in self.Xs])
        yp = native.void_p_array([y.data_ptr() for y in self.ys])
        kernel_scales = getattr(self, "_kernel_scales", None) or self.scales   # fp8: packed per tile
        sp = native.void_p_array([s.data_ptr() for s in kernel_scales]) if kernel_scales else None
        rows = (C.c_longlong * n)(*[X.shape[0] for X in self.Xs])
        grp = (C.c_int * n)(*self.groups)
        code = int(self.use_tensor_cores())
        #: which fused kernel serves this model ("tc" / "fp8" = tcgen05 tensor cores, else CUDA cores)
        self.selected_kernel = {0: "simt", 1: "tc", 2: "fp8", 3: "generic-bf16", 4: "generic-fp32"}[code]
        if self.kernel == "auto" and code not in (1, 2) and not hasattr(self.family, "code_id"):
            import logging

            logging.getLogger(__name__).warning(
                "GLM with %d features (%s, row stride %d) is outside the tensor-core kernel's shapes (bf16, P %% 8 == 0, "
                "P <= 384, 16-byte aligned rows): using the %s CUDA-core kernel — single pass, but slower",
                self.n_features, self.Xs[0].dtype, self.ld, self.selected_kernel)
        out_grp = (C.c_int * n)(*self.node_ids) if self.node_ids is not None else None
        native.check(
            lib.b200_engine_set_glm(
                handle, n, Xp, yp, sp, rows, grp, self.n_features, self.ld, self.n_groups,
                self.n_chains, _family_code(self.family), code, out_grp, self.n_nodes, self.n_family_params,
            ),
            "set_glm",
        )
        if hasattr(self.family, "code_id"):
            lib.b200_engine_set_custom_launcher(handle, C.c_void_p(self.family.launcher_address()))

    # -- eager oracle (also the compute step of the NCCL baseline) ---------------------------
    def reference_partial(self, inputs, *, dtype=None, chunk_rows: int = 1 << 20) -> np.ndarray:
        """This node's partial with stock PyTorch ops (oracle of the kernels, compute step of the CPU / gloo
        path).  Rows are processed ``chunk_rows`` at a time (a multiple of 128), so an fp64 oracle of a
        10M-row shard needs 2 GB of scratch, not 20."""
        import torch

        dtype = dtype or torch.float32
        intercept, beta, phi = self._split_inputs(inputs)
        self._note_shapes(inputs)
        ic = torch.as_tensor(np.asarray(intercept, dtype=np.float64)).reshape(self.n_chains, -1)
        bt = torch.as_tensor(np.asarray(beta, dtype=np.float64)).reshape(self.n_chains, self.n_features)
        full = torch.zeros(self.n_nodes, self.n_chains, 1 + self.n_params, dtype=torch.float64, device=self.device)
        B = bt.to(self.device, dtype)                              # [K, P]
        ph = torch.as_tensor(self._check_phi(phi)).to(self.device, dtype) if phi is not None else None   # [K, D]
        GP = self.n_groups + self.n_features
        for si, (X, y, g) in enumerate(zip(self.Xs, self.ys, self.groups)):
            out = full[self.node_ids[si] if self.node_ids is not None else 0]
            icg = ic[:, g].to(self.device, dtype)
            for r0 in range(0, X.shape[0], chunk_rows):
                r1 = min(X.shape[0], r0 + chunk_rows)
                Xf = self._dequant_rows(si, r0, r1).to(dtype)
                eta = Xf @ B.T + icg                                # [n, K]
                yy = y[r0:r1].to(dtype).unsqueeze(1)
                if hasattr(self.family, "code_id"):
                    if self.family.torch_fn is None:
                        raise ValueError("this CustomFamily has no torch_fn oracle")
                    ll, r = self.family.torch_fn(yy, eta)
                elif ph is not None:
                    ll, r, dphi = _phi_family_terms(self.family, yy, eta, ph)
                    for j, dj in enumerate(dphi):
                        out[:, 1 + GP + j] += dj.double().sum(0)
                elif self.family == "logistic":
                    ll = yy * eta - torch.nn.functional.softplus(eta)
                    r = yy - torch.sigmoid(eta)
                elif self.family == "poisson":
                    mu = torch.exp(eta)
                    ll = yy * eta - mu
                    r = yy - mu
                else:
                    d = yy - eta
                    ll = -0.5 * d * d - 0.918938533204672742
                    r = d
                out[:, 0] += ll.double().sum(0)
                out[:, 1 + g] += r.double().sum(0)
                out[:, 1 + self.n_groups : 1 + GP] += (r.T @ Xf).double()
        return full.reshape(-1).cpu().numpy()

    def _dequant_rows(self, seg: int, r0: int, r1: int):
        """Rows ``[r0, r1)`` of segment ``seg`` as stored values (dense kernels: the matrix itself)."""
        return self.Xs[seg][r0:r1]

    def _dequant(self, X):
        return X

    def eager_partial(self, inputs) -> np.ndarray:
        """Stock-PyTorch evaluation as a practitioner would write it: two bf16 GEMMs (X @ beta, then
        r @ X) plus elementwise ops — the compute step of the NCCL baseline ("baseline B").  Reads the
        design matrix twice; no custom kernels."""
        import torch

        if self.Xs[0].dtype != torch.bfloat16 or self.n_family_params:
            return self.reference_partial(inputs)
        intercept, beta = inputs
        self._note_shapes(inputs)
        ic = torch.as_tensor(np.asarray(intercept, dtype=np.float32)).reshape(self.n_chains, -1).to(self.device)
        bt = torch.as_tensor(np.asarray(beta, dtype=np.float32)).reshape(self.n_chains, self.n_features).to(self.device)
        out = torch.zeros(self.n_chains, 1 + self.n_params, dtype=torch.float64, device=self.device)
        for X, y, g in zip(self.Xs, self.ys, self.groups):
            eta = (X @ bt.T.to(torch.bfloat16)).float() + ic[:, g]          # [n, K]
            yy = y.unsqueeze(1)
            if self.family == "logistic":
                ll = yy * eta - torch.nn.functional.softplus(eta)
                r = yy - torch.sigmoid(eta)
            elif self.family == "poisson":
                mu = torch.exp(eta)
                ll = yy * eta - mu
                r = yy - mu
            else:
                d = yy - eta
                ll = -0.5 * d * d - 0.918938533204672742
                r = d
            out[:, 0] += ll.sum(0).double()
            out[:, 1 + g] += r.sum(0).double()
            out[:, 1 + self.n_groups :] += (r.T.to(torch.bfloat16) @ X).double()
        return out.reshape(-1).cpu().numpy()

    def bytes_per_eval(self) -> int:
        return int(sum(X.shape[0] * (self.n_features * X.element_size() + 4) for X in self.Xs))

    def flops_per_eval(self) -> int:
        return int(4 * self.n_rows * self.n_features * self.n_chains)


def _phi_family_terms(family: str, y, eta, phi):
    """Per-row ``(ll, dll/deta, [dll/dphi_j])`` of a family with fitted parameters (``phi`` ``[K, D]``)."""
    import math

    import torch

    if family == "normal":
        s = phi[:, 0]
        z = (y - eta) / s
        return -0.5 * z * z - torch.log(s) - 0.5 * math.log(2 * math.pi), z / s, [(z * z - 1) / s]
    if family == "student_t":
        s, nu = phi[:, 0], phi[:, 1]
        d = y - eta
        z2 = (d / s) ** 2
        l1p = torch.log1p(z2 / nu)
        ll = (torch.lgamma((nu + 1) / 2) - torch.lgamma(nu / 2) - 0.5 * torch.log(nu * math.pi) - torch.log(s)
              - (nu + 1) / 2 * l1p)
        r = (nu + 1) * d / (nu * s * s + d * d)
        d_s = ((nu + 1) * z2 / (nu + z2) - 1) / s
        d_nu = 0.5 * (torch.digamma((nu + 1) / 2) - torch.digamma(nu / 2) - 1 / nu - l1p + (nu + 1) * z2 / (nu * (nu + z2)))
        return ll, r, [d_s, d_nu]
    a = phi[:, 0]                                        # negative_binomial
    mu = torch.exp(eta)
    l1 = torch.log1p(mu / a)
    ll = torch.lgamma(y + a) - torch.lgamma(a) - torch.lgamma(y + 1) - a * l1 + y * (eta - torch.log(a + mu))
    r = a * (y - mu) / (a + mu)
    d_a = torch.digamma(y + a) - torch.digamma(a) - l1 + (mu - y) / (a + mu)
    return ll, r, [d_a]


def quantize_block_fp8(X, block: int = 32):
    """Block-scaled FP8 quantisation of a design matrix (MX-style, 32 x 32 blocks).

    Returns ``(Xq, scales)``: ``Xq`` e4m3 bytes ``[n, P]`` (``torch.float8_e4m3fn``) and UE8M0 scale
    bytes ``[4 * ceil(n / 128), P / 32]`` (rows padded to whole 128-row tiles with 2^0), with
    ``X[r, f] ~= float(Xq[r, f]) * 2 ** (scales[r // 32, f // 32] - 127)``.
    """
    import torch

    n, P = X.shape
    if P % block:
        raise ValueError("P must be a multiple of 32")
    n_rb = (n + block - 1) // block
    n_rb_pad = ((n + 127) // 128) * 4
    Xf = X.float()
    pad = n_rb * block - n
    if pad:
        Xf = torch.cat([Xf, torch.zeros(pad, P, device=X.device)], 0)
    blocks = Xf.view(n_rb, block, P // block, block)
    amax = blocks.abs().amax(dim=(1, 3))                                  # [n_rb, P/32]
    # power-of-two scale such that amax / scale <= 448 (e4m3 max)
    exp = torch.ceil(torch.log2(torch.clamp(amax, min=2.0**-100) / 448.0)).clamp(-127, 127)
    exp = torch.where(amax > 0, exp, torch.zeros_like(exp))
    scale = torch.exp2(exp)
    q = (blocks / scale[:, None, :, None]).reshape(n_rb * block, P)[:n].to(torch.float8_e4m3fn)
    scales = torch.full((n_rb_pad, P // block), 127, dtype=torch.uint8, device=X.device)
    scales[:n_rb] = (exp + 127).to(torch.uint8)
    return q.contiguous(), scales.contiguous()


def dequantize_block_fp8(Xq, scales, block: int = 32):
    """Inverse of :func:`quantize_block_fp8` (fp32 result); the oracle of the fp8 kernel tests."""
    import torch

    n, P = Xq.shape
    s = torch.exp2(scales.float() - 127.0)                                 # [n_rb_pad, P/32]
    s_full = s.repeat_interleave(block, 0)[:n].repeat_interleave(block, 1)
    return Xq.float() * s_full


def pack_tile_scales(scales, n_features: int):
    """Re-orders the UE8M0 block scales ``[4 * tiles, P / 32]`` into the 16 words per 128-row tile that
    ``csrc/glm_fp8.cu`` copies into the TMEM scale-factor columns: words 0-7 for ``eta = X . Theta^T``
    (word ``4g + q`` = row group ``q``, feature blocks ``4g..4g+3``), words 8-15 for ``G += X^T . R``
    (word ``4h + qq`` = row groups 0..3 of feature block ``4h + qq``).  Returns ``uint8 [tiles, 64]``."""
    import torch

    nfb = n_features // 32
    if nfb not in (4, 8) or scales.shape[0] % 4 or scales.shape[1] != nfb:
        raise ValueError("the fp8 kernel takes P in {128, 256} and scales padded to whole 128-row tiles")
    tiles, g2 = scales.shape[0] // 4, nfb // 4
    s4 = scales.contiguous().view(tiles, 4, g2, 4)                       # [tile, q, g, j]
    packed = torch.full((tiles, 2, 2, 4, 4), 127, dtype=torch.uint8, device=scales.device)
    packed[:, 0, :g2] = s4.permute(0, 2, 1, 3)                           # [tile, g, q, byte j]
    packed[:, 1, :g2] = s4.permute(0, 2, 3, 1)                           # [tile, h, qq, byte q]
    return packed.reshape(tiles, 64).contiguous()


class Fp8GlmShards(GlmShards):
    """GLM shards whose design matrices are block-scaled FP8 (``quantize_block_fp8``).

    The hierarchical-GLM configuration of BASELINE.json: one partial-pooling group (intercept) per
    shard/GPU, e4m3 design matrix with 32 x 32 UE8M0 block scales, evaluated by ``csrc/glm_fp8.cu``
    (``tcgen05.mma.kind::mxf8f6f4.block_scale``).  Up to 3 chains per launch.  The residuals of the
    Poisson and Gaussian families are unbounded, so the kernel block-scales them too (one UE8M0
    exponent per 32-row group, written to the MMA's scale-factor-B columns).
    """

    def __init__(self, Xqs, scales, ys, *, groups=None, n_groups: int = 1, n_chains: int = 1,
                 family: str = "logistic", node_ids=None, n_nodes=None) -> None:
        if not 1 <= n_chains <= 3:
            raise ValueError("the fp8 kernel batches at most 3 chains per launch")
        if family in FAMILY_PARAMS:
            raise ValueError(f"the fp8 kernel has no {family} family: families with fitted parameters run on the "
                             f"bf16 tensor-core kernel ({_TC_SHAPES})")
        super().__init__(Xqs, ys, groups=groups, n_groups=n_groups, family=family, n_chains=n_chains, kernel="fp8",
                         scales=scales, node_ids=node_ids, n_nodes=n_nodes)
        self._kernel_scales = [pack_tile_scales(s, self.n_features) for s in self.scales]

    @classmethod
    def from_dense(cls, Xs, ys, **kw):
        pairs = [quantize_block_fp8(X) for X in Xs]
        return cls([p[0] for p in pairs], [p[1] for p in pairs], ys, **kw)

    def _dequant(self, X):
        idx = next(i for i, Xi in enumerate(self.Xs) if Xi is X)
        return dequantize_block_fp8(X, self.scales[idx])

    def _dequant_rows(self, seg: int, r0: int, r1: int):
        if r0 % 32:
            raise ValueError("row chunks of block-scaled matrices start on a 32-row boundary")
        return dequantize_block_fp8(self.Xs[seg][r0:r1], self.scales[seg][r0 // 32 : (r1 + 31) // 32])

    def bytes_per_eval(self) -> int:
        return int(sum(X.shape[0] * (self.n_features + 4) + s.numel() for X, s in zip(self.Xs, self._kernel_scales)))


def synth_logistic_shard(n_rows: int, n_features: int, *, seed: int, device, chunk_rows: int = 1 << 20,
                         beta_scale: float = 0.05):
    """Synthetic logistic-regression shard generated on the device in chunks
    (bf16 ``X ~ N(0,1)``, ``y ~ Bernoulli(sigmoid(X beta* + 0.3))``)."""
    import torch

    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    beta_true = (torch.randn(n_features, generator=gen, device=device) * beta_scale).float()
    X = torch.empty(n_rows, n_features, dtype=torch.bfloat16, device=device)
    y = torch.empty(n_rows, dtype=torch.float32, device=device)
    for r0 in range(0, n_rows, chunk_rows):
        r1 = min(n_rows, r0 + chunk_rows)
        xb = torch.randn(r1 - r0, n_features, generator=gen, device=device, dtype=torch.float32).to(torch.bfloat16)
        X[r0:r1] = xb
        p = torch.sigmoid(xb.float() @ beta_true + 0.3)
        y[r0:r1] = (torch.rand(r1 - r0, generator=gen, device=device) < p).float()
    return X, y, beta_true


def synth_logistic_shard_fp8(n_rows: int, n_features: int, *, seed: int, device, chunk_rows: int = 1 << 20):
    """Like :func:`synth_logistic_shard` but quantised chunk-wise to block-scaled FP8 (never holds
    the fp32 matrix): returns ``(Xq e4m3 [n, P], scales uint8 [4*ceil(n/128), P/32], y)``."""
    import torch

    assert chunk_rows % 128 == 0
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    beta_true = (torch.randn(n_features, generator=gen, device=device) * 0.05).float()
    col_scale = torch.exp(torch.randn(n_features, generator=gen, device=device) * 0.5)  # heterogeneous feature scales
    Xq = torch.empty(n_rows, n_features, dtype=torch.float8_e4m3fn, device=device)
    scales = torch.full((((n_rows + 127) // 128) * 4, n_features // 32), 127, dtype=torch.uint8, device=device)
    y = torch.empty(n_rows, dtype=torch.float32, device=device)
    for r0 in range(0, n_rows, chunk_rows):
        r1 = min(n_rows, r0 + chunk_rows)
        xb = torch.randn(r1 - r0, n_features, generator=gen, device=device) * col_scale
        q, s = quantize_block_fp8(xb)
        Xq[r0:r1] = q
        scales[r0 // 32 : r0 // 32 + s.shape[0]] = s
        xd = dequantize_block_fp8(q, s)
        p = torch.sigmoid(xd @ (beta_true / col_scale) + 0.3)
        y[r0:r1] = (torch.rand(r1 - r0, generator=gen, device=device) < p).float()
    return Xq, scales, y


def synth_glm_shard(n_rows: int, n_features: int, *, family: str = "logistic", phi=(), seed: int, device,
                    chunk_rows: int = 1 << 20, beta_scale: float = 0.05, intercept: float = 0.3, beta_true=None):
    """Synthetic shard of any built-in family, generated on the device in chunks: bf16 ``X ~ N(0,1)``,
    ``eta = X beta* + intercept`` and ``y`` drawn from the family with parameters ``phi`` (``(sigma,)``,
    ``(sigma, nu)`` or ``(alpha,)``; the negative binomial as a gamma-Poisson mixture).  ``beta*`` is drawn
    (``N(0, beta_scale^2)``) unless ``beta_true`` is given — nodes of one federation share it.  Returns
    ``(X, y, beta_true)``.  Draws come from a seeded fork of torch's generator, so the global state is untouched."""
    import torch

    names = FAMILY_PARAMS.get(family, ())
    phi = tuple(float(v) for v in np.atleast_1d(np.asarray(phi, dtype=np.float64)))
    if family not in FAMILIES or len(phi) != len(names):
        raise ValueError(f"family {family!r} takes parameters {names}, got {phi}")
    device = torch.device(device)
    with torch.random.fork_rng(devices=[device] if device.type == "cuda" else []):
        torch.manual_seed(seed)
        drawn = torch.randn(n_features, device=device) * beta_scale
        beta_true = (drawn if beta_true is None else torch.as_tensor(beta_true, device=device)).float()
        X = torch.empty(n_rows, n_features, dtype=torch.bfloat16, device=device)
        y = torch.empty(n_rows, dtype=torch.float32, device=device)
        for r0 in range(0, n_rows, chunk_rows):
            r1 = min(n_rows, r0 + chunk_rows)
            xb = torch.randn(r1 - r0, n_features, device=device, dtype=torch.float32).to(torch.bfloat16)
            X[r0:r1] = xb
            eta = xb.float() @ beta_true + intercept
            n = r1 - r0
            if family == "logistic":
                yb = (torch.rand(n, device=device) < torch.sigmoid(eta)).float()
            elif family == "poisson":
                yb = torch.poisson(torch.exp(eta))
            elif family == "gaussian":
                yb = eta + torch.randn(n, device=device)
            elif family == "normal":
                yb = eta + phi[0] * torch.randn(n, device=device)
            elif family == "student_t":
                chi2 = 2.0 * torch._standard_gamma(torch.full((n,), phi[1] / 2, device=device))
                yb = eta + phi[0] * torch.randn(n, device=device) / torch.sqrt(chi2 / phi[1])
            else:                                                  # negative_binomial
                alpha = phi[0]
                rate = torch._standard_gamma(torch.full((n,), alpha, device=device)) * (torch.exp(eta) / alpha)
                yb = torch.poisson(rate)
            y[r0:r1] = yb.float()
    return X, y, beta_true
