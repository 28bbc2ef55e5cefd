"""torch.autograd.Function wrappers over the C-ABI kernels.

Every op here launches hand-written sm_100a kernels through ``_lib`` (ctypes) on the current
CUDA stream.  Nothing falls back to eager PyTorch arithmetic: CPU tensors raise.
"""
from __future__ import annotations

import os

import torch

from . import _lib, parallel, profiling
from ._lib import check, ptr, stream, workspace
from .graph import structure_of

ACT_NONE, ACT_RELU, ACT_RELU_GRAD = 0, 1, 2
LOSS_KINDS = {"AUC": 0, "HingeAUC": 1, "WeightedHingeAUC": 2, "WeightedAUC": 3, "AdaAUC": 4, "AdaHingeAUC": 5,
              "LogRank": 6, "CE": 7, "InfoNCE": 8}

# which scatter kernel backs the endpoint-gather backward: "sorted" (deterministic, default)
# or "atomic" (red.global.add, order non-deterministic)
SCATTER_MODE = "sorted"

# dense-layer backend: "tf32x3c2" = tcgen05 tensor cores, CTA pairs (cta_group::2), error-compensated
# 3xTF32 (fp32 parity, default); "tf32x3" = the same with one CTA per tile; "tf32c2" / "tf32" = plain TF32
# (fast path, ~1e-3 relative, stated separately); "ffma" = exact fp32 on the CUDA cores
GEMM_BACKEND = os.environ.get("PLNLP_GEMM", "tf32x3c2")

# 3xTF32: largest K one TMEM accumulator may take before the split-k reduction combines partials (the tensor
# core accumulates with round-toward-zero, see gemm_raw).  1088 = 17 x 64 keeps the whole parity suite inside
# 1e-5 and cuts K = 4267 (the ddi-shape dense aggregation) into 4 splits = 272 CTAs = one full wave of the
# 296 resident CTA slots instead of 5 splits = 1.15 waves (0.167 -> 0.127 ms per aggregation).
TF32X3_KCAP = int(os.environ.get("PLNLP_GEMM_KCAP", "1088"))

# TMA-fed persistent GEMM (csrc/gemm_tma.cu) for tall-skinny products A[M, K] @ W^T / A @ W with a huge M and
# N, K of a few hundred: "auto" = when M >= 16 384, N <= 256 and K <= 512 (the encoder's dense layers on the big
# graphs; the large-K predictor GEMMs of the ddi shape stay on the CTA-pair kernel), "1" = whenever legal, "0" = off
GEMM_TMA = os.environ.get("PLNLP_GEMM_TMA", "auto")
# ... and its counterpart for weight gradients C = A^T B over a huge K with M, N <= 256 (csrc/gemm_tma_tn.cu): "auto" =
# when every SM gets at least four 1088-row units (K >= 644 096: the layer-1 weight gradient of the citation2 shape;
# at K = 262 144 the 241 units leave the 148 persistent CTAs unevenly loaded and the CTA-pair kernel is as fast),
# "1" = whenever legal, "0" = off
GEMM_TMA_TN = os.environ.get("PLNLP_GEMM_TMA_TN", "auto")

# fused edge scoring for the MLP head (gather + Hadamard + layer 1 + out layer in one tcgen05 kernel)
FUSED_EDGE_MLP = os.environ.get("PLNLP_FUSED_EDGE", "1") != "0"
# ... and its backward (dZ1 formed in the loaders of both GEMMs, Hadamard product re-gathered in the weight-gradient
# GEMM): "auto" = when the embedding table fits the L2 budget below, "1" = whenever legal, "0" = off
FUSED_EDGE_BWD = os.environ.get("PLNLP_FUSED_EDGE_BWD", "0")
FUSED_EDGE_BWD_L2_BYTES = 48 << 20


def _f32c(t):
    if t.dtype != torch.float32:
        raise RuntimeError(f"plnlp_b200 kernels are fp32; got {t.dtype}")
    if not t.is_cuda:
        raise RuntimeError("plnlp_b200 kernels need CUDA tensors; there is no CPU path")
    return t


def _rowmajor(t):
    """2-D tensor usable as a row-major matrix with a leading dimension (no copy when the
    inner stride is 1, e.g. column slices of a weight)."""
    _f32c(t)
    if t.dim() != 2:
        raise RuntimeError("expected a 2-D tensor")
    if t.stride(1) != 1 and t.size(1) != 1:
        t = t.contiguous()
    if t.size(1) == 1 and t.stride(0) < 1:
        t = t.contiguous()
    return t


def _ld(t):
    return t.stride(0) if t.size(0) > 1 else max(t.size(1), t.stride(0))


# SpMM operands of <= 64 columns whose rows sit on a 16-byte aligned pitch run on the two-rows-per-warp kernel
# (csrc/spmm.cu, spmm_csr_narrow_kernel; the library picks it from the layout it is handed).  Measured on the
# citation2-shape graph (profiles/r02_spmm_narrow_ab.txt): F = 64 53 % -> 71 % of the HBM copy peak, F = 32
# 30 % -> 41 %.  A width that is not a multiple of 4 (the 50-wide embedding) is NOT re-pitched: at <= 256 B per
# gathered row the kernel is bound by the rate of random DRAM row fetches (~17 G rows/s whatever the width
# between 16 and 64 floats), the generic kernel already reaches it, and the copy would cost more than it gains.


def _rows_for_spmm(rows, F, device):
    """uninitialised fp32 [rows, F] for a GEMM output that an SpMM gathers next: for F <= 64 the rows sit on a
    64-float (256-byte) pitch -- the GEMM epilogue then writes whole 16-byte vectors and the gather runs on the
    two-rows-per-warp kernel with every row inside one 256-byte window (F = 50: 3.91 -> 3.75 ms)"""
    if F <= 64 and F % 4:
        return torch.empty(rows, 64, dtype=torch.float32, device=device)[:, :F]
    return torch.empty(rows, F, dtype=torch.float32, device=device)


def apply_spmm_defaults():
    """reset the SpMM tuning knobs to the library defaults + environment overrides (after an A/B run)"""
    _lib.load().plnlp_spmm_tune(SPMM_TUNE_DEFAULT[0], SPMM_TUNE_DEFAULT[1], SPMM_TUNE_DEFAULT[2], 0)
    _lib.apply_spmm_tuning()


# the library's built-in (prefetch_mode, staged_mode, staged_warps): see csrc/spmm.cu g_spmm_*
SPMM_TUNE_DEFAULT = (3, 12, 4)


def new_seed():
    """64-bit Philox seed drawn from torch's CPU generator (reproducible under manual_seed,
    never touches the device)."""
    return int(torch.randint(0, 2 ** 62, (1,)).item())


# ---------------------------------------------------------------------------
# raw launches
# ---------------------------------------------------------------------------
def spmm_raw(plan, x, use_val, div_rows, bias=None, relu=False, drop_p=0.0, seed=0, out=None, x_index=None,
             mask=None, mask_scale=1.0):
    """fp32 features, or bf16 features (bf16 storage in and out, fp32 accumulation -- the separately stated
    bf16 path; autograd and the models stay fp32)."""
    lib = _lib.load()
    bf16 = x.dtype == torch.bfloat16
    if bf16:
        if not x.is_cuda or x.dim() != 2:
            raise RuntimeError("bf16 SpMM needs a 2-D CUDA tensor")
        if x.stride(1) != 1:
            x = x.contiguous()
    else:
        x = _rowmajor(x)
    F = x.size(1)
    if x_index is None and x.size(0) != plan.n_cols:
        raise RuntimeError(f"SpMM shape mismatch: adjacency has {plan.n_cols} columns, x has {x.size(0)} rows")
    if out is None:
        out = torch.empty(plan.n_rows, F, dtype=x.dtype, device=x.device)
    elif out.dtype != x.dtype:
        raise RuntimeError("SpMM output dtype must match the feature dtype")
    partial = None
    if plan.n_fix:
        partial = workspace.get("spmm_partial", plan.n_partial * F * 4, x.device)
    val = plan.val if use_val else None
    alg = plan.alg_bytes(F, 2 if bf16 else 4) - (0 if use_val or plan.val is None else plan.nnz * 4)
    fn, name = (lib.plnlp_spmm_csr_bf16, "spmm_csr_bf16") if bf16 else (lib.plnlp_spmm_csr_f32, "spmm_csr_f32")
    if x_index is not None:
        if x_index.dtype != torch.int32 or x_index.numel() != plan.n_cols or not x_index.is_cuda:
            raise RuntimeError("x_index must be a CUDA int32 vector with one entry per column of the adjacency")
        name += " (row-sparse operand)"
        alg = 0        # the live share of the entries is data dependent and not known on the host: no GB/s claim
    if getattr(plan, "subset", False):
        name += " (row subset)"
    with profiling.span(f"{name} F={F}", alg, 0):
        check(fn(ptr(plan.item_ptr), ptr(plan.item_row), ptr(plan.item_slot), plan.n_items,
                 ptr(plan.item_end), ptr(x_index), ptr(plan.col), ptr(val), ptr(plan.row_cnt if div_rows else None), ptr(bias),
                 int(relu), float(drop_p), int(seed), ptr(x), _ld(x), x.size(0), ptr(out), _ld(out), F,
                 ptr(partial), ptr(plan.fix_ptr), ptr(plan.fix_row), plan.n_fix,
                 ptr(mask), _ld(mask) if mask is not None else 0, float(mask_scale), stream()),
              "plnlp_" + name.split(" ")[0])
    return out


def gemm_raw(A, B, transa=False, transb=False, C=None, beta=0.0, bias=None, act=ACT_NONE, aux=None,
             drop_p=0.0, seed=0, split_k=None, backend=None, fixed_backend=False):
    """C = act(op(A) @ op(B) + beta*C + bias); A, B row-major with leading dimensions.  ``fixed_backend``: run
    ``backend`` itself, whatever the shape (no switch to the CUDA-core kernel for a small product, no TMA-fed
    kernel): for a caller whose results must not depend on the row count of A.

    A plain-TF32 request ("tf32", "tf32c2") on the CTA kernels runs one pass only when both operands take 16-byte
    loads (16-byte aligned base, leading dimension and contiguous extent multiples of 4 floats); otherwise they run
    their scalar-load instantiation, which exists only as 3xTF32.  That result is the "tf32x3" / "tf32x3c2" one bit
    for bit under the same split_k -- but a plain request keeps its split, it is not raised to TF32X3_KCAP k-terms per
    accumulator, so with a longer K per split the three passes share one round-toward-zero accumulator.  The TMA-fed
    tall-skinny kernel (below; it needs only A aligned) splits B itself and runs one pass whatever B's layout."""
    lib = _lib.load()
    A, B = _rowmajor(A), _rowmajor(B)
    M, K = (A.size(1), A.size(0)) if transa else (A.size(0), A.size(1))
    K2, N = (B.size(1), B.size(0)) if transb else (B.size(0), B.size(1))
    if K != K2:
        raise RuntimeError(f"GEMM inner dimensions differ: {K} vs {K2}")
    if C is None:
        C = torch.empty(M, N, dtype=torch.float32, device=A.device)
        beta = 0.0
    backend = backend or GEMM_BACKEND
    if backend != "ffma" and not fixed_backend and (K < 32 or N < 16 or M * N * K < (1 << 20)):
        backend = "ffma"                      # too little work for a tensor-core tile (a small M x N with a
                                              # huge K -- weight gradients -- does go to the tensor cores)
    bn = 128 if backend == "ffma" or (N <= 128 and not backend.endswith("c2")) else 256
    if split_k is None:
        tiles = ((M + 127) // 128) * ((N + bn - 1) // bn)
        split_k = 1
        if tiles < 148 and K >= 2048:
            split_k = int(min(max(1, (2 * 148) // tiles), K // 512, 64))
    if backend in ("tf32x3", "tf32x3c2"):
        # the tensor core accumulates with round-toward-zero: keep K per accumulator <= 1024 and
        # let the split-k reduction (RN adds on the CUDA cores) combine the partials
        split_k = max(split_k, (K + TF32X3_KCAP - 1) // TF32X3_KCAP)
    ws = None
    ws_bytes = 0
    if split_k > 1:
        ws_bytes = split_k * M * N * 4
        ws = workspace.get("gemm_splitk", ws_bytes, A.device)
    if (backend in ("tf32x3c2", "tf32c2", "tf32x3", "tf32") and GEMM_TMA != "0" and not fixed_backend and not transa
            and split_k == 1
            and K >= 32 and N <= 512 and _ld(A) % 4 == 0 and A.data_ptr() % 16 == 0
            and (GEMM_TMA == "1" or (M >= 16384 and N <= 256 and K <= 512))):
        nbytes = lib.plnlp_gemm_tf32_tma_workspace_bytes(N, K)
        wsb = workspace.get("gemm_tma_b", nbytes, A.device)
        passes = 3 if backend.startswith("tf32x3") else 1
        with profiling.span(f"gemm_tf32x{passes}_tma {M}x{N}x{K}", 0, 2 * M * N * K):
            check(lib.plnlp_gemm_tf32_tma(passes, int(transb), M, N, K, ptr(A), _ld(A), ptr(B), _ld(B), ptr(C), _ld(C),
                                          float(beta), ptr(bias), int(act), ptr(aux), _ld(aux) if aux is not None else 0,
                                          float(drop_p), int(seed), ptr(wsb), nbytes, stream()), "plnlp_gemm_tf32_tma")
        return C
    if (backend in ("tf32x3c2", "tf32c2", "tf32x3", "tf32") and GEMM_TMA_TN != "0" and not fixed_backend
            and transa and not transb
            and M <= 256 and 8 <= N <= 256 and beta == 0.0 and bias is None and act == ACT_NONE
            and _ld(A) % 4 == 0 and _ld(B) % 4 == 0 and A.data_ptr() % 16 == 0 and B.data_ptr() % 16 == 0
            and (GEMM_TMA_TN == "1" or K >= 4 * 148 * TF32X3_KCAP)):
        # weight gradient over a huge row count: both operands MN-major, consumed as the TMA lands them
        nbytes = lib.plnlp_gemm_tf32_tma_tn_workspace_bytes()
        wsp = workspace.get("gemm_tma_tn", nbytes, A.device)
        passes = 3 if backend.startswith("tf32x3") else 1
        with profiling.span(f"gemm_tf32x{passes}_tma_tn {M}x{N}x{K}", 0, 2 * M * N * K):
            check(lib.plnlp_gemm_tf32_tma_tn(passes, M, N, K, ptr(A), _ld(A), ptr(B), _ld(B), ptr(C), _ld(C), ptr(wsp),
                                             nbytes, stream()), "plnlp_gemm_tf32_tma_tn")
        return C
    tail = (int(transa), int(transb), M, N, K, ptr(A), _ld(A), ptr(B), _ld(B), ptr(C), _ld(C),
            float(beta), ptr(bias), int(act), ptr(aux), _ld(aux) if aux is not None else 0,
            float(drop_p), int(seed), ptr(ws), ws_bytes, int(split_k), stream())
    name = {"ffma": "gemm_f32", "tf32x3": "gemm_tf32x3", "tf32": "gemm_tf32", "tf32x3c2": "gemm_tf32x3_2cta",
            "tf32c2": "gemm_tf32_2cta"}[backend]
    with profiling.span(f"{name} {M}x{N}x{K}{' splitk' if split_k > 1 else ''}", 0, 2 * M * N * K):
        if backend == "ffma":
            check(lib.plnlp_gemm_f32(*tail), "plnlp_gemm_f32")
        elif backend.endswith("c2"):
            check(lib.plnlp_gemm_tf32_2cta(3 if backend == "tf32x3c2" else 1, *tail), "plnlp_gemm_tf32_2cta")
        else:
            check(lib.plnlp_gemm_tf32(3 if backend == "tf32x3" else 1, *tail), "plnlp_gemm_tf32")
    return C


def row_nonzero_index_raw(x):
    """int32 [rows]: r where row r of x has a non-zero entry, else -1 (an ``x_index`` for spmm_raw)"""
    lib = _lib.load()
    x = _rowmajor(x)
    index = torch.empty(x.size(0), dtype=torch.int32, device=x.device)
    with profiling.span("row_nonzero_index_f32", x.numel() * 4 + x.size(0) * 4, 0):
        check(lib.plnlp_row_nonzero_index_f32(ptr(x), _ld(x), x.size(0), x.size(1), ptr(index), stream()),
              "plnlp_row_nonzero_index_f32")
    return index


def colsum_raw(x, scale=1.0):
    lib = _lib.load()
    x = _rowmajor(x)
    rows, cols = x.shape
    out = torch.empty(cols, dtype=torch.float32, device=x.device)
    nbytes = lib.plnlp_colsum_workspace_bytes(rows, cols)
    ws = workspace.get("colsum", nbytes, x.device)
    with profiling.span("colsum_f32", rows * cols * 4, 0):
        check(lib.plnlp_colsum_f32(ptr(x), _ld(x), rows, cols, float(scale), ptr(out), ptr(ws), nbytes, stream()),
              "plnlp_colsum_f32")
    return out


def relu_drop_bwd_raw(y, dy, scale):
    lib = _lib.load()
    y, dy = _rowmajor(y), _rowmajor(dy)
    dx = torch.empty(y.shape, dtype=torch.float32, device=y.device)
    with profiling.span("relu_drop_bwd_f32", y.numel() * 12, 0):
        check(lib.plnlp_relu_drop_bwd_f32(ptr(y), _ld(y), ptr(dy), _ld(dy), float(scale), y.size(0), y.size(1),
                                          ptr(dx), _ld(dx), stream()), "plnlp_relu_drop_bwd_f32")
    return dx


def _edges_i64(edges):
    if edges.dtype != torch.int64 or not edges.is_cuda:
        raise RuntimeError("edges must be a CUDA int64 [P, 2] tensor")
    if edges.dim() != 2 or edges.size(1) != 2:
        raise RuntimeError("edges must have shape [P, 2]")
    return edges.contiguous()


def gather_hadamard_raw(h, edges):
    lib = _lib.load()
    h, edges = _rowmajor(h), _edges_i64(edges)
    P, H = edges.size(0), h.size(1)
    out = torch.empty(P, H, dtype=torch.float32, device=h.device)
    with profiling.span("gather_hadamard_f32", P * (3 * H * 4 + 16), 0):
        check(lib.plnlp_gather_hadamard_f32(ptr(h), _ld(h), h.size(0), ptr(edges), P, H, ptr(out), H, stream()),
              "plnlp_gather_hadamard_f32")
    return out


def gather_rows_raw(h, edges, side):
    """h[edges[:, side]] -> [P, H] (the column of the int64 [P, 2] edge tensor is read in place)"""
    lib = _lib.load()
    h, edges = _rowmajor(h), _edges_i64(edges)
    P, H = edges.size(0), h.size(1)
    out = torch.empty(P, H, dtype=torch.float32, device=h.device)
    with profiling.span("gather_rows_f32", P * (2 * H * 4 + 8), 0):
        check(lib.plnlp_gather_rows_f32(ptr(h), _ld(h), h.size(0), edges.data_ptr() + 8 * int(side), 2, P, H,
                                        ptr(out), H, stream()), "plnlp_gather_rows_f32")
    return out


def gather_rows_idx_raw(h, idx):
    """h[idx] for a 1-D int64 index vector -> [len(idx), H]"""
    lib = _lib.load()
    h = _rowmajor(h)
    if idx.dtype != torch.int64 or not idx.is_cuda or idx.dim() != 1:
        raise RuntimeError("idx must be a 1-D CUDA int64 tensor")
    idx = idx.contiguous()
    P, H = idx.numel(), h.size(1)
    out = torch.empty(P, H, dtype=torch.float32, device=h.device)
    with profiling.span("gather_rows_f32", P * (2 * H * 4 + 8), 0):
        check(lib.plnlp_gather_rows_f32(ptr(h), _ld(h), h.size(0), ptr(idx), 1, P, H, ptr(out), H, stream()),
              "plnlp_gather_rows_f32")
    return out


def row_scatter_raw(g, idx, n_rows):
    """grad_h [n_rows, H] with grad_h[n] = sum of g[p] over {p : idx[p] = n}, summed in increasing p (stable sort
    -> deterministic); the backward of ``gather_rows_raw``"""
    lib = _lib.load()
    g = _rowmajor(g)
    H = g.size(1)
    idx = torch.where(idx < 0, idx + n_rows, idx)
    key = idx.to(torch.int32) if n_rows < 2 ** 31 else idx
    skey, entry = torch.sort(key, stable=True)
    seg_ptr = torch.searchsorted(skey, _node_range(n_rows, key.dtype, g.device))
    grad_h = torch.empty(n_rows, H, dtype=torch.float32, device=g.device)
    with profiling.span("row_scatter_sorted_f32", g.numel() * 4 + grad_h.numel() * 4 + idx.numel() * 16, 0):
        check(lib.plnlp_row_scatter_sorted_f32(ptr(g), _ld(g), H, ptr(seg_ptr), n_rows, ptr(entry), ptr(grad_h), H,
                                               stream()), "plnlp_row_scatter_sorted_f32")
    return grad_h


def fused_edge_mlp_ok(h, params):
    """the fused forward covers the reference recipes' head: MLPPredictor with ONE hidden layer
    (mlp_num_layers = 2) on a tensor-core backend, embedding width H <= 1024 (the kernel keeps K = H in one
    accumulator and rejects more), any hidden width.  H < 32 is left to the unfused path on purpose: the kernel
    takes it, but gemm_raw runs a layer-1 GEMM with K < 32 on the CUDA cores."""
    if not FUSED_EDGE_MLP or GEMM_BACKEND not in ("tf32x3c2", "tf32c2") or len(params) != 4:
        return False
    W1, w2 = params[0], params[2]
    return (W1.dim() == 2 and W1.size(1) == h.size(1) and w2.numel() == W1.size(0) and h.size(1) <= 1024
            and h.size(1) >= 32 and W1.stride(1) == 1)


def edge_mlp_fwd_raw(h, edges, W1, b1, w2, b2, drop_p=0.0, seed=0, need_a1=True):
    """fused gather + Hadamard + Linear/relu/dropout + Linear(->1): -> (score [P], a1 [P, N1] or None).  With
    GEMM_BACKEND = "tf32c2" layer 1 runs one TF32 pass only when h and W1 take 16-byte loads (H, both leading
    dimensions multiples of 4 floats, 16-byte aligned bases); otherwise the scalar gather, which exists only as
    3xTF32, runs and the result is the "tf32x3c2" one bit for bit."""
    lib = _lib.load()
    h, edges, W1 = _rowmajor(h), _edges_i64(edges), _rowmajor(W1)
    w2 = _f32c(w2).reshape(-1).contiguous()
    P, H, N1 = edges.size(0), h.size(1), W1.size(0)
    nq = 2 * ((N1 + 255) // 256)
    part = torch.empty(nq, P, dtype=torch.float32, device=h.device)
    a1 = torch.empty(P, N1, dtype=torch.float32, device=h.device) if need_a1 else None
    passes = 3 if GEMM_BACKEND == "tf32x3c2" else 1
    with profiling.span(f"edge_mlp_fwd_fused {P}x{N1}x{H}", 0, 2 * P * N1 * H):
        check(lib.plnlp_edge_mlp_fwd_tf32(passes, ptr(h), _ld(h), h.size(0), ptr(edges), P, H, ptr(W1), _ld(W1),
                                          ptr(b1), N1, float(drop_p), int(seed), ptr(w2), ptr(a1),
                                          N1 if need_a1 else 0, ptr(part), P, stream()),
              "plnlp_edge_mlp_fwd_tf32")
    score = part[0].clone() if nq == 1 else part.sum(0)        # fixed order: partial 0 + 1 + 2 + ...
    if b2 is not None:
        score = score + b2.reshape(())
    return score, a1


def edge_dot_raw(h, edges):
    lib = _lib.load()
    h, edges = _rowmajor(h), _edges_i64(edges)
    P, H = edges.size(0), h.size(1)
    score = torch.empty(P, dtype=torch.float32, device=h.device)
    with profiling.span("edge_dot_fwd_f32", P * (2 * H * 4 + 20), 0):
        check(lib.plnlp_edge_dot_fwd_f32(ptr(h), _ld(h), h.size(0), ptr(edges), P, H, ptr(score), stream()),
              "plnlp_edge_dot_fwd_f32")
    return score


def mlp_out_fwd_raw(a, w, b):
    lib = _lib.load()
    a = _rowmajor(a)
    w = _f32c(w).reshape(-1).contiguous()
    P, H = a.shape
    score = torch.empty(P, dtype=torch.float32, device=a.device)
    with profiling.span("mlp_out_fwd_f32", P * (H * 4 + 4), 0):
        check(lib.plnlp_mlp_out_fwd_f32(ptr(a), _ld(a), ptr(w), ptr(b), P, H, ptr(score), stream()),
              "plnlp_mlp_out_fwd_f32")
    return score


def mlp_out_bwd_raw(a, w, dscore, mask_a, drop_scale, need_dz=True, need_dzsum=False):
    """-> dz [P,H] (None when need_dz is False), dw [H], db [1] (, dzsum [H] = column sums of dz when asked for)"""
    lib = _lib.load()
    a = _rowmajor(a)
    w = _f32c(w).reshape(-1).contiguous()
    dscore = _f32c(dscore).contiguous()
    P, H = a.shape
    dz = torch.empty(P, H, dtype=torch.float32, device=a.device) if need_dz else None
    dw = torch.empty(H, dtype=torch.float32, device=a.device)
    db = torch.empty(1, dtype=torch.float32, device=a.device)
    dzsum = torch.empty(H, dtype=torch.float32, device=a.device) if need_dzsum else None
    nbytes = lib.plnlp_mlp_out_bwd_workspace_bytes(P, H)
    ws = workspace.get("mlp_out_bwd", nbytes, a.device)
    with profiling.span("mlp_out_bwd_f32" if need_dz else "mlp_out_bwd_f32 (reductions only)",
                        P * ((2 if need_dz else 1) * H * 4 + 4), 0):
        check(lib.plnlp_mlp_out_bwd_f32(ptr(a), _ld(a), ptr(w), ptr(dscore), P, H, int(mask_a), float(drop_scale),
                                        ptr(dz), H, ptr(dw), ptr(db), ptr(dzsum), ptr(ws), nbytes, stream()),
              "plnlp_mlp_out_bwd_f32")
    if need_dzsum:
        return dz, dw, db, dzsum
    return dz, dw, db


def fused_edge_mlp_bwd_ok(h, a1, params):
    """the fused backward re-gathers the Hadamard product inside the weight-gradient GEMM: it pays while the embedding
    table the pairs index stays in the L2 (ddi shape: 8.7 MB; the 232 MB compact table of the citation2 shape would be
    gathered from DRAM inside a tensor-core loader with two slabs in flight)"""
    if FUSED_EDGE_BWD == "0":
        return False
    W1 = params[0]
    H, N1 = h.size(1), W1.size(0)
    ok = (H % 4 == 0 and N1 % 4 == 0 and N1 <= 1088 and _ld(h) % 4 == 0 and _ld(W1) % 4 == 0 and _ld(a1) % 4 == 0
          and h.data_ptr() % 16 == 0 and W1.data_ptr() % 16 == 0 and a1.data_ptr() % 16 == 0)
    if FUSED_EDGE_BWD == "1":
        return ok
    return ok and h.numel() * 4 <= FUSED_EDGE_BWD_L2_BYTES


def edge_mlp_bwd_raw(h, edges, W1, a1, dscore, w2, drop_scale):
    """fused backward of the 2-layer MLP head behind the Hadamard gather: -> dA0 [P, H], dW1 [N1, H]"""
    lib = _lib.load()
    h, edges, W1, a1 = _rowmajor(h), _edges_i64(edges), _rowmajor(W1), _rowmajor(a1)
    w2 = _f32c(w2).reshape(-1).contiguous()
    dscore = _f32c(dscore).contiguous()
    P, H, N1 = edges.size(0), h.size(1), W1.size(0)
    da0 = torch.empty(P, H, dtype=torch.float32, device=h.device)
    dw1 = torch.empty(N1, H, dtype=torch.float32, device=h.device)
    passes = 3 if GEMM_BACKEND == "tf32x3c2" else 1
    tiles = ((N1 + 127) // 128) * ((H + 255) // 256)           # the split-k rule of gemm_raw for dW1 [N1, H] over K = P
    split_k = 1
    if tiles < 148 and P >= 2048:
        split_k = int(min(max(1, (2 * 148) // tiles), P // 512, 64))
    if passes == 3:
        split_k = max(split_k, (P + TF32X3_KCAP - 1) // TF32X3_KCAP)
    nbytes = lib.plnlp_edge_mlp_bwd_workspace_bytes(P, H, N1, split_k)
    ws = workspace.get("gemm_splitk", nbytes, h.device)
    with profiling.span(f"edge_mlp_bwd_fused {P}x{N1}x{H}", 0, 4 * P * N1 * H):
        check(lib.plnlp_edge_mlp_bwd_tf32(passes, ptr(h), _ld(h), h.size(0), ptr(edges), P, H, ptr(W1), _ld(W1), N1,
                                          ptr(a1), _ld(a1), ptr(dscore), ptr(w2), float(drop_scale), ptr(da0), H,
                                          ptr(dw1), H, ptr(ws), nbytes, split_k, stream()),
              "plnlp_edge_mlp_bwd_tf32")
    return da0, dw1


_RANGE_CACHE = {}


def _node_range(n_rows, dtype, device):
    key = (n_rows, dtype, device)
    r = _RANGE_CACHE.get(key)
    if r is None:
        if len(_RANGE_CACHE) > 8:
            _RANGE_CACHE.clear()
        r = _RANGE_CACHE[key] = torch.arange(n_rows + 1, dtype=dtype, device=device)
    return r


def edge_scatter_raw(h, edges, da=None, dscore=None, mode=None):
    """grad_h [n_rows, H] of the endpoint gather; da [P,H] (MLP head) or dscore [P] (DOT)."""
    lib = _lib.load()
    mode = mode or SCATTER_MODE
    h, edges = _rowmajor(h), _edges_i64(edges)
    P, H, n_rows = edges.size(0), h.size(1), h.size(0)
    if da is not None:
        da = _rowmajor(da)
    if dscore is not None:
        dscore = _f32c(dscore).contiguous()
    ldda = _ld(da) if da is not None else 0
    if mode == "atomic":
        grad_h = torch.zeros(n_rows, H, dtype=torch.float32, device=h.device)
        with profiling.span("edge_scatter_atomic_f32", P * (5 * H * 4 + 16), 0):
            check(lib.plnlp_edge_scatter_atomic_f32(ptr(h), _ld(h), n_rows, ptr(edges), P, H, ptr(da), ldda,
                                                    ptr(dscore), ptr(grad_h), H, stream()),
                  "plnlp_edge_scatter_atomic_f32")
        return grad_h
    # node-sorted incidence list (a CSR over ALL nodes): a STABLE sort of the endpoint ids orders the
    # entries t = 2p + side by node and, inside a node, by t -> fixed summation order.  One segment per
    # node (empty ones included, they write their zero row), so there is no data-dependent size and no
    # host synchronisation, and grad_h needs no separate zero fill.
    _sp = profiling.span("torch: stable sort + searchsorted for sorted scatter")
    _sp.__enter__()
    flat = edges.reshape(-1)                          # entry id t = 2p + side  <->  flat[t]
    flat = torch.where(flat < 0, flat + n_rows, flat)
    key = flat.to(torch.int32) if n_rows < 2 ** 31 else flat
    skey, entry = torch.sort(key, stable=True)
    # seg_ptr[i] = first position whose node id is >= i (one binary search per node, no bincount / scan)
    seg_ptr = torch.searchsorted(skey, _node_range(n_rows, key.dtype, edges.device))
    _sp.__exit__()
    grad_h = torch.empty(n_rows, H, dtype=torch.float32, device=h.device)
    with profiling.span("edge_scatter_sorted_f32", P * (5 * H * 4 + 32), 0):
        check(lib.plnlp_edge_scatter_sorted_f32(ptr(h), _ld(h), n_rows, ptr(edges), P, H, ptr(da), ldda, ptr(dscore),
                                                ptr(seg_ptr), None, n_rows, ptr(entry),
                                                ptr(grad_h), H, stream()), "plnlp_edge_scatter_sorted_f32")
    return grad_h


def pair_loss_raw(kind, pos, neg, num_neg, weight=None):
    """-> loss [1], dpos [B], dneg [B*num_neg]"""
    lib = _lib.load()
    pos = _f32c(pos).reshape(-1).contiguous()
    neg = _f32c(neg).reshape(-1).contiguous()
    B = pos.numel()
    if neg.numel() != B * num_neg:
        raise RuntimeError(f"neg_out has {neg.numel()} scores, expected {B} x {num_neg}")
    if weight is not None:
        weight = _f32c(weight).reshape(-1).contiguous()
    loss = torch.empty(1, dtype=torch.float32, device=pos.device)
    dpos = torch.empty(B, dtype=torch.float32, device=pos.device)
    dneg = torch.empty(B * num_neg, dtype=torch.float32, device=pos.device)
    nbytes = lib.plnlp_pair_loss_workspace_bytes(B)
    ws = workspace.get("pair_loss", nbytes, pos.device)
    with profiling.span("pair_loss_f32", (B + B * num_neg) * 8, 0):
        check(lib.plnlp_pair_loss_f32(int(kind), ptr(pos), ptr(neg), ptr(weight), B, int(num_neg), ptr(loss), ptr(dpos),
                                      ptr(dneg), ptr(ws), nbytes, stream()), "plnlp_pair_loss_f32")
    return loss, dpos, dneg


# ---------------------------------------------------------------------------
# autograd Functions
# ---------------------------------------------------------------------------
class SpMM(torch.autograd.Function):
    """out = epi(A @ x) with A given by ``adj``; reduce 'sum' uses the stored values, 'mean'
    drops them (SAGEConv) and divides by max(row_nnz, 1).  Optional fused epilogue
    bias -> relu -> dropout (GCNConv + layer.py:21-22).  Backward runs the same kernel on the
    cached transposed structure."""

    @staticmethod
    def forward(ctx, x, bias, adj, reduce, relu, drop_p, seed, sparse_grad=False):
        st = structure_of(adj)
        mean = reduce == "mean"
        ctx.sparse_grad = bool(sparse_grad)
        ctx.dense = st.dense_ok and GEMM_BACKEND != "ffma" and x.size(1) >= 32
        if ctx.dense:
            # small, dense-ish adjacency (graph.Structure.dense_ok): multiply it as a dense matrix on the
            # tensor cores; same epilogue and the same Philox indexing (row * F + col) as the gather kernel
            out = gemm_raw(st.dense(mean), x, bias=bias, act=ACT_RELU if relu else ACT_NONE,
                           drop_p=drop_p if relu else 0.0, seed=seed)
        else:
            plan = st.fwd_noval if mean else st.fwd
            out = spmm_raw(plan, x, use_val=not mean, div_rows=mean, bias=bias, relu=relu, drop_p=drop_p,
                           seed=seed)
        ctx.st, ctx.mean, ctx.relu, ctx.drop_p = st, mean, relu, drop_p
        ctx.has_bias = bias is not None
        ctx.save_for_backward(out if (relu or drop_p > 0) else None)
        return out

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        g = _rowmajor(g)
        if out is not None:
            g = relu_drop_bwd_raw(out, g, 1.0 / (1.0 - ctx.drop_p))      # zero rows stay zero rows
        gb = colsum_raw(g) if (ctx.has_bias and ctx.needs_input_grad[1]) else None
        gx = None
        if ctx.needs_input_grad[0]:
            if ctx.dense:
                gx = gemm_raw(ctx.st.dense(ctx.mean), g, transa=True)          # A^T g on the tensor cores
            else:
                # sparse_grad (set by the layer in forward): the caller reads this conv's output only at the
                # endpoint rows of the edge batch, so most rows of g are exactly zero.  The index of the live
                # rows is measured HERE, on this node's own incoming gradient (one pass over g) -- never
                # handed between autograd nodes, whose gradient buffers autograd may accumulate into in place.
                x_index = row_nonzero_index_raw(g) if ctx.sparse_grad else None
                plan = ctx.st.bwd_mean if ctx.mean else ctx.st.bwd
                gx = spmm_raw(plan, g, use_val=True if ctx.mean else ctx.st.has_value, div_rows=False,
                              x_index=x_index)
        return gx, gb, None, None, None, None, None, None


def spmm(adj, x, reduce="sum", bias=None, relu=False, drop_p=0.0, seed=0, sparse_grad=False):
    """``sparse_grad``: the gradient arriving at the output will be non-zero only at a few rows (the endpoint
    rows of an edge batch); the backward then gathers only those (see SpMM.backward)."""
    if reduce == "add":
        reduce = "sum"
    if isinstance(adj, parallel.ShardedAdj):      # row-partitioned encoder (citation2-shape, SURVEY 8e)
        return parallel.pspmm(adj, x, reduce, bias=bias, relu=relu, drop_p=drop_p, seed=seed,
                              sparse_grad=sparse_grad)
    if reduce not in ("sum", "mean"):
        raise NotImplementedError(f"reduce={reduce!r}")
    return SpMM.apply(x, bias, adj, reduce, bool(relu), float(drop_p), int(seed), bool(sparse_grad))


class SpMMRows(torch.autograd.Function):
    """out[t, :] = epi( (A @ x)[rows[t], :] ): the SpMM for a SUBSET of the output rows, written compactly.

    The last conv's output is read only at the endpoint rows of the edge batch (model.py:152-156), so the other
    rows are never computed: ~10 % of citation2-shape's rows / ~25 % of the stored entries per batch.  The values
    at the selected rows are those of the full product, bit for bit (same per-row accumulation order).  Backward:
    A[rows, :]^T @ g with the compact gradient as a row-sparse operand of the transposed plan (x_index)."""

    @staticmethod
    def forward(ctx, x, bias, adj, rows, reduce, relu, drop_p, seed, premask=None):
        from .graph import build_subset_plan
        # premask (a float: the dropout scale of the layer that produced x): x is a relu(-dropout) OUTPUT with no other
        # consumer; the backward then returns the gradient w.r.t. that layer's PRE-activation (mask fused into the
        # SpMM epilogue) and the producing layer skips its own relu backward (``grad_premasked``)
        ctx.premask = premask
        st = structure_of(adj)
        mean = reduce == "mean"
        parent = st.fwd_noval if mean else st.fwd
        ready = getattr(rows, "_plnlp_prepared", {}).get(id(st)) if not mean else None
        if ready is not None:                                     # BaseModel.prepare_batch built them ahead of time
            plan, ctx.x_index = ready
        else:
            ctx.x_index = None
            with profiling.span("torch: row-subset plan (index ops, 3 host reads)"):
                plan = build_subset_plan(parent, st.rowptr, rows)
        out = spmm_raw(plan, x, use_val=not mean, div_rows=mean, bias=bias, relu=relu, drop_p=drop_p, seed=seed)
        ctx.st, ctx.mean, ctx.drop_p, ctx.has_bias = st, mean, drop_p, bias is not None
        ctx.save_for_backward(rows, out if (relu or drop_p > 0) else None, x if premask is not None else None)
        return out

    @staticmethod
    def backward(ctx, g):
        rows, out, xmask = ctx.saved_tensors
        st = ctx.st
        g = _rowmajor(g)
        if out is not None:
            g = relu_drop_bwd_raw(out, g, 1.0 / (1.0 - ctx.drop_p))
        gb = colsum_raw(g) if (ctx.has_bias and ctx.needs_input_grad[1]) else None
        gx = None
        if ctx.needs_input_grad[0]:
            x_index = ctx.x_index
            if x_index is None:
                with profiling.span("torch: x_index of the compact gradient"):
                    x_index = torch.full((st.n_rows,), -1, dtype=torch.int32, device=g.device)
                    x_index[rows] = torch.arange(rows.numel(), dtype=torch.int32, device=g.device)
            plan = st.bwd_mean if ctx.mean else st.bwd
            gx = spmm_raw(plan, g, use_val=True if ctx.mean else st.has_value, div_rows=False, x_index=x_index,
                          mask=xmask, mask_scale=ctx.premask if xmask is not None else 1.0)
        return gx, gb, None, None, None, None, None, None, None


def spmm_rows(adj, x, rows, reduce="sum", bias=None, relu=False, drop_p=0.0, seed=0, premask=None):
    if reduce == "add":
        reduce = "sum"
    if reduce not in ("sum", "mean"):
        raise NotImplementedError(f"reduce={reduce!r}")
    if rows.dtype != torch.int64 or rows.dim() != 1 or not rows.is_cuda:
        raise RuntimeError("rows must be a 1-D CUDA int64 tensor of distinct row ids")
    return SpMMRows.apply(x, bias, adj, rows, reduce, bool(relu), float(drop_p), int(seed),
                          None if premask is None else float(premask))


class FusedLinear(torch.autograd.Function):
    """Y = act( sum_i X_i @ W_i^T + bias ), act in {none, relu(+dropout)}.

    One or more (X_i, W_i) pairs accumulate into one output through the GEMM's beta=1 path, so
    SAGEConv's lin_l(agg) + lin_r(x) and the concat-free ``[emb | x] @ W^T`` never materialise an
    intermediate.  W_i may be a column slice of a larger weight (leading dimension respected)."""

    @staticmethod
    def forward(ctx, bias, addend, act, drop_p, seed, n, *xw):
        xs, ws = xw[:n], xw[n:]
        # ``addend`` (optional): accumulated in the first GEMM's epilogue (beta = 1) -- a conv's aggregate plus its
        # root / skip linear, as AddLinear does for a single input block
        Y = None if addend is None else addend.clone()
        for i, (x, w) in enumerate(zip(xs, ws)):
            last = i == n - 1
            Y = gemm_raw(x, w, transb=True, C=Y, beta=0.0 if Y is None else 1.0,
                         bias=bias if i == 0 else None,
                         act=act if last else ACT_NONE, drop_p=drop_p if last else 0.0, seed=seed)
        ctx.n, ctx.act, ctx.drop_p = n, act, drop_p
        ctx.has_bias = bias is not None
        ctx.save_for_backward(Y if act == ACT_RELU else None, *xs, *ws)
        return Y

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        Y, n = saved[0], ctx.n
        xs, ws = saved[1:1 + n], saved[1 + n:]
        g = _rowmajor(g)
        if Y is not None:
            g = relu_drop_bwd_raw(Y, g, 1.0 / (1.0 - ctx.drop_p))
        gb = colsum_raw(g) if (ctx.has_bias and ctx.needs_input_grad[0]) else None
        gxs, gws = [], []
        for i in range(n):
            gx = gemm_raw(g, ws[i]) if ctx.needs_input_grad[6 + i] else None          # dX = dY @ W
            gw = gemm_raw(g, xs[i], transa=True) if ctx.needs_input_grad[6 + n + i] else None  # dW = dY^T @ X
            gxs.append(gx)
            gws.append(gw)
        return (gb, g if ctx.needs_input_grad[1] else None, None, None, None, None, *gxs, *gws)


def fused_linear(xs, ws, bias=None, act=ACT_NONE, drop_p=0.0, seed=0, addend=None):
    xs, ws = list(xs), list(ws)
    return FusedLinear.apply(bias, addend, int(act), float(drop_p), int(seed), len(xs), *xs, *ws)


def aggregate_into(adj, x, out):
    """out = A @ x through the raw kernel (no autograd), ``out`` possibly a column slice of a wider buffer.
    Row-partitioned adjacency: x is this rank's row block, all-gathered first (parallel.ShardedAdj)."""
    if isinstance(adj, parallel.ShardedAdj):
        st = structure_of(adj.local)
        x = parallel.all_gather_rows(parallel.pad_rows(x, adj.blk), adj.group)
    else:
        st = structure_of(adj)
    return spmm_raw(st.fwd, x, use_val=st.has_value, div_rows=False, out=out)


# row-partitioned, symmetric adjacency: A^T g as all-gather(g) + row-block SpMM instead of transposed SpMM + reduce-scatter
AGG_T_BY_GATHER = os.environ.get("PLNLP_AGG_T", "gather") == "gather"


class _Deferred:
    """a result that is only computed when asked for (after communication that was started earlier has landed)"""

    def __init__(self, fn):
        self.fn = fn


def aggregate_t(adj, g, sparse_rows=False, async_op=False):
    """A^T @ g through the raw kernel; row-partitioned: the transposed product over all columns is
    reduce-scattered to the owners of the rows.  ``sparse_rows``: most rows of g are exactly zero -- measure
    which (one pass over g) and gather only the live ones.  ``async_op``: -> (result, wait); on a row-partitioned
    adjacency the reduce-scatter is then in flight until ``wait()`` is called."""
    if isinstance(adj, parallel.ShardedAdj) and adj.symmetric and AGG_T_BY_GATHER:
        # A == A^T: this rank's rows of A^T g are A[rows, :] @ g -- ALL-GATHER g (async: the caller's weight-gradient
        # GEMM runs meanwhile) and multiply with the row block the forward pass uses.  Same bytes on the wire as the
        # reduce-scatter of the transposed product, but a gather (pull over peer memory, no reduction), one CSR
        # structure for both directions, and every row accumulated in the single-GPU order.
        st = structure_of(adj.local)
        full, wait = parallel.all_gather_rows(parallel.pad_rows(g, adj.blk), adj.group, tag="grad rows", async_op=True,
                                              name="nccl all_gather (grad rows)")

        def finish():
            wait()
            xi = row_nonzero_index_raw(full) if sparse_rows else None
            return spmm_raw(st.fwd, full, use_val=st.has_value, div_rows=False, x_index=xi)
        return (_Deferred(finish), None) if async_op else finish()
    x_index = row_nonzero_index_raw(g) if sparse_rows else None
    if isinstance(adj, parallel.ShardedAdj):
        st = structure_of(adj.local)
        full = spmm_raw(st.bwd, g, use_val=st.has_value, div_rows=False, x_index=x_index)
        return parallel._reduce_scatter_rows(full, adj.blk, adj.group, async_op=async_op)
    st = structure_of(adj)
    out = spmm_raw(st.bwd, g, use_val=st.has_value, div_rows=False, x_index=x_index)
    return (out, (lambda: None)) if async_op else out


class AggLinear(torch.autograd.Function):
    """Y = act( [A x_0 | A x_1 | ...] W^T + bias ) for GCNConv's "aggregate first" order (layer.GCNConv).

    ``buf`` [N, K] is a persistent buffer whose CONSTANT column blocks (the aggregate of data.x) were filled once
    by the caller; the blocks of the inputs that change between steps (``xs``, at column offsets ``offs``) are
    written by the SpMM kernel straight into their slice of ``buf`` (leading dimension K), so the layer is one
    SpMM per live block and ONE GEMM over K instead of a GEMM per block, and its weight gradient is one GEMM too.
    ``holder['stamp']`` counts forwards: if another forward overwrote ``buf`` before this node's backward runs,
    the live blocks are recomputed first.  Works on a row-partitioned adjacency too (``aggregate_into``)."""

    @staticmethod
    def forward(ctx, W, bias, adj, buf, holder, offs, act, drop_p, seed, sparse_grad, grad_premasked, *xs):
        ctx.sparse_grad = bool(sparse_grad)
        ctx.grad_premasked = bool(grad_premasked)      # the consumer's backward already applied this layer's relu mask
        for off, x in zip(offs, xs):
            aggregate_into(adj, x, buf[:, off:off + x.size(1)])
        holder["stamp"] = holder.get("stamp", 0) + 1
        Y = gemm_raw(buf, W, transb=True, bias=bias, act=act, drop_p=drop_p, seed=seed)
        ctx.adj, ctx.buf, ctx.holder, ctx.stamp, ctx.offs = adj, buf, holder, holder["stamp"], offs
        ctx.act, ctx.drop_p, ctx.has_bias = act, drop_p, bias is not None
        ctx.save_for_backward(Y if act == ACT_RELU else None, W, *xs)
        return Y

    @staticmethod
    def backward(ctx, g):
        Y, W = ctx.saved_tensors[:2]
        xs = ctx.saved_tensors[2:]
        buf = ctx.buf
        g = _rowmajor(g)
        if Y is not None and not ctx.grad_premasked:
            g = relu_drop_bwd_raw(Y, g, 1.0 / (1.0 - ctx.drop_p))
        if ctx.holder["stamp"] != ctx.stamp:          # buf was reused by a later forward: restore our blocks
            for off, x in zip(ctx.offs, xs):
                aggregate_into(ctx.adj, x, buf[:, off:off + x.size(1)])
            ctx.holder["stamp"] += 1
        # input gradients first: on a row-partitioned adjacency their reduce-scatter then travels over NVLink while
        # the weight-gradient GEMM below runs
        gxs, waits = [], []
        for i, (off, x) in enumerate(zip(ctx.offs, xs)):
            if not ctx.needs_input_grad[11 + i]:
                gxs.append(None)
                continue
            gu = gemm_raw(g, W[:, off:off + x.size(1)], C=_rows_for_spmm(g.size(0), x.size(1), g.device))   # d(A x_i) = dY W_i
            gx, wait = aggregate_t(ctx.adj, gu, ctx.sparse_grad, async_op=True)                 # A^T .
            gxs.append(gx if isinstance(gx, _Deferred) else gx[: x.size(0)])
            waits.append(wait)
        gW = gb = None
        ext = ctx.holder.get("ext")
        want_b = ctx.has_bias and ctx.needs_input_grad[1]
        if ctx.needs_input_grad[0] and want_b and ext is not None:
            # dY^T [A x | 1]: the weight gradient and, in the last column, the bias gradient (column sums of dY)
            gWe = gemm_raw(g, ext, transa=True)
            gW, gb = gWe[:, :-1].contiguous(), gWe[:, -1].contiguous()
        else:
            gW = gemm_raw(g, buf, transa=True) if ctx.needs_input_grad[0] else None         # dW = dY^T [A x]
            gb = colsum_raw(g) if want_b else None
        for wait in waits:
            if wait is not None:
                wait()
        gxs = [gx.fn()[: x.size(0)] if isinstance(gx, _Deferred) else gx for gx, x in zip(gxs, xs)]
        return (gW, gb, None, None, None, None, None, None, None, None, None, *gxs)


def agg_linear(adj, buf, holder, offs, xs, W, bias, act=ACT_NONE, drop_p=0.0, seed=0, sparse_grad=False,
               grad_premasked=False):
    return AggLinear.apply(W, bias, adj, buf, holder, tuple(offs), int(act), float(drop_p), int(seed),
                           bool(sparse_grad), bool(grad_premasked), *xs)


class GatherHadamard(torch.autograd.Function):
    """h[edges[:,0]] * h[edges[:,1]] in one kernel (model.py:155-156 + layer.py:81)."""

    @staticmethod
    def forward(ctx, h, edges):
        ctx.save_for_backward(h, edges)
        return gather_hadamard_raw(h, edges)

    @staticmethod
    def backward(ctx, g):
        h, edges = ctx.saved_tensors
        return edge_scatter_raw(h, edges, da=g), None


class EdgeDot(torch.autograd.Function):
    """DotPredictor over gathered endpoints: score[p] = <h[src_p], h[dst_p]>."""

    @staticmethod
    def forward(ctx, h, edges):
        ctx.save_for_backward(h, edges)
        return edge_dot_raw(h, edges)

    @staticmethod
    def backward(ctx, g):
        h, edges = ctx.saved_tensors
        return edge_scatter_raw(h, edges, dscore=g), None


class GatherRows(torch.autograd.Function):
    """x = h[edges[:, side]] (model.py:155-156, one endpoint); backward = deterministic sorted segment sum."""

    @staticmethod
    def forward(ctx, h, edges, side):
        ctx.save_for_backward(edges)
        ctx.side, ctx.n_rows = side, h.size(0)
        return gather_rows_raw(h, edges, side)

    @staticmethod
    def backward(ctx, g):
        (edges,) = ctx.saved_tensors
        return row_scatter_raw(g, edges[:, ctx.side], ctx.n_rows), None, None


class PairMean(torch.autograd.Function):
    """(x[:P] + x[P:]) / 2 for a [2P] score vector (MLPCatPredictor averages the two concatenation orders,
    layer.py:115); the column-sum kernel on the [2, P] view."""

    @staticmethod
    def forward(ctx, x):
        P = x.numel() // 2
        return colsum_raw(x.reshape(2, P), 0.5)

    @staticmethod
    def backward(ctx, g):
        return (0.5 * g).repeat(2)


def row_dot(a, b):
    """sum(a * b, -1) for two [P, H] matrices with autograd, on the edge-dot kernels (rows p of a and b are the
    two endpoints of pair p in the stacked matrix)."""
    P = a.size(0)
    ar = torch.arange(P, device=a.device)
    return EdgeDot.apply(torch.cat([a, b], 0), torch.stack([ar, ar + P], 1))


class MLPOut(torch.autograd.Function):
    """last MLPPredictor layer (out_channels = 1): a @ w^T + b -> [P, 1]."""

    @staticmethod
    def forward(ctx, a, w, b):
        ctx.save_for_backward(a, w)
        ctx.has_b = b is not None
        return mlp_out_fwd_raw(a, w, b).reshape(-1, 1)

    @staticmethod
    def backward(ctx, g):
        a, w = ctx.saved_tensors
        dz, dw, db = mlp_out_bwd_raw(a, w, g.reshape(-1), mask_a=False, drop_scale=1.0)
        return dz, dw.reshape(w.shape), (db if ctx.has_b else None)


class PairLoss(torch.autograd.Function):
    """loss.py:5-14, 31-35: forward and d loss / d score from one kernel."""

    @staticmethod
    def forward(ctx, pos_out, neg_out, weight, kind, num_neg):
        loss, dpos, dneg = pair_loss_raw(kind, pos_out, neg_out, num_neg, weight)
        ctx.save_for_backward(dpos, dneg)
        ctx.shapes = (pos_out.shape, neg_out.shape)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        dpos, dneg = ctx.saved_tensors
        return (dpos * g).reshape(ctx.shapes[0]), (dneg * g).reshape(ctx.shapes[1]), None, None, None


def pair_loss(name, pos_out, neg_out, num_neg, weight=None):
    return PairLoss.apply(pos_out, neg_out, weight, LOSS_KINDS[name], int(num_neg))


class EdgeScoreLoss(torch.autograd.Function):
    """The fused scoring step of BaseModel.train (model.py:152-160): gather both endpoints of
    every positive and negative pair, Hadamard, predictor head, pairwise loss and d loss / d score,
    returning the scalar loss; backward produces grad_h and the predictor parameter gradients
    without autograd recording the per-pair intermediates.

    head = 'MLP': params = (W_0, b_0, ..., W_{L-1}, b_{L-1}) with the last layer [1, H];
    head = 'DOT': no params.
    """

    @staticmethod
    def forward(ctx, h, edges, weight, head, kind, num_neg, n_pos, drop_p, seed, *params):
        edges = _edges_i64(edges)
        fused = False
        if head == "DOT":
            score = edge_dot_raw(h, edges)
            acts = []
        else:
            L = len(params) // 2
            fused = fused_edge_mlp_ok(h, params)
            if fused:
                # ONE kernel: gather + Hadamard + layer 1 (tcgen05) + bias/relu/dropout + the out layer's dot;
                # the Hadamard product a0 is never written to HBM (backward re-gathers it)
                score, a1 = edge_mlp_fwd_raw(h, edges, params[0], params[1], params[2], params[3], drop_p,
                                             seed + 7919, need_a1=True)
                acts = [a1]
            else:
                a = gather_hadamard_raw(h, edges)
                acts = [a]
                for i in range(L - 1):
                    a = gemm_raw(a, params[2 * i], transb=True, bias=params[2 * i + 1], act=ACT_RELU,
                                 drop_p=drop_p, seed=seed + 7919 * (i + 1))
                    acts.append(a)
                score = mlp_out_fwd_raw(a, params[2 * (L - 1)], params[2 * (L - 1) + 1])
        loss, dpos, dneg = pair_loss_raw(kind, score[:n_pos], score[n_pos:], num_neg, weight)
        ctx.head, ctx.drop_p, ctx.n_params, ctx.fused = head, drop_p, len(params), fused
        ctx.save_for_backward(h, edges, dpos, dneg, *acts, *params)
        ctx.n_acts = len(acts)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        h, edges, dpos, dneg = saved[:4]
        acts = saved[4:4 + ctx.n_acts]
        params = saved[4 + ctx.n_acts:]
        dscore = torch.cat([dpos, dneg]) * g
        if ctx.head == "DOT":
            gh = edge_scatter_raw(h, edges, dscore=dscore)
            return (gh,) + (None,) * 8
        L = len(params) // 2
        scale = 1.0 / (1.0 - ctx.drop_p)
        grads = [None] * len(params)
        if ctx.fused and fused_edge_mlp_bwd_ok(h, acts[0], params):
            # one pass over a1 for the reductions (dw2, db2, db1), then the two GEMMs with dZ1 formed in their loaders
            # and the Hadamard product re-gathered inside the dW1 loader: no [P, H] intermediate but dA0
            a1 = acts[0]
            _, dw2, db2, db1 = mlp_out_bwd_raw(a1, params[2], dscore, mask_a=True, drop_scale=scale, need_dz=False,
                                               need_dzsum=True)
            da0, dw1 = edge_mlp_bwd_raw(h, edges, params[0], a1, dscore, params[2], scale)
            grads[0], grads[1] = dw1, db1.reshape(params[1].shape)
            grads[2], grads[3] = dw2.reshape(params[2].shape), db2.reshape(params[3].shape)
            gh = edge_scatter_raw(h, edges, da=da0)
            return (gh,) + (None,) * 8 + tuple(grads)
        if ctx.fused:        # the forward never stored the Hadamard product: re-gather it for dW_0
            acts = (gather_hadamard_raw(h, edges),) + tuple(acts)
        # last layer: dz w.r.t. the pre-activation of the previous hidden layer (mask fused)
        dz, dw, db = mlp_out_bwd_raw(acts[-1], params[2 * (L - 1)], dscore, mask_a=(L > 1), drop_scale=scale)
        grads[2 * (L - 1)] = dw.reshape(params[2 * (L - 1)].shape)
        grads[2 * (L - 1) + 1] = db.reshape(params[2 * (L - 1) + 1].shape)
        for i in range(L - 2, -1, -1):
            W = params[2 * i]
            grads[2 * i] = gemm_raw(dz, acts[i], transa=True)            # dW_i = dZ_i^T @ A_{i-1}
            grads[2 * i + 1] = colsum_raw(dz)
            if i > 0:   # dA_{i-1} = dZ_i @ W_i, masked by relu/dropout of layer i-1
                dz = gemm_raw(dz, W, act=ACT_RELU_GRAD, aux=acts[i], drop_p=ctx.drop_p)
            else:
                dz = gemm_raw(dz, W)                                      # d loss / d hadamard
        gh = edge_scatter_raw(h, edges, da=dz)
        return (gh,) + (None,) * 8 + tuple(grads)


def edge_score_loss(h, pos_edge, neg_edge, num_neg, loss_name, weight=None, head="MLP", params=(),
                    drop_p=0.0, seed=0):
    """pos_edge [B,2], neg_edge [B*num_neg,2] (negatives of positive i in rows i*k..i*k+k-1)."""
    edges = torch.cat([pos_edge, neg_edge], 0)
    return EdgeScoreLoss.apply(h, edges, weight, head, LOSS_KINDS[loss_name], int(num_neg), pos_edge.size(0),
                               float(drop_p), int(seed), *params)


# ---------------------------------------------------------------------------
# attention conv pieces (TransformerConv under the reference's Transformer encoder, layer.py:57-63)
# ---------------------------------------------------------------------------
class SegmentSoftmax(torch.autograd.Function):
    """alpha = softmax of scale * s over the stored entries of every CSR row (per destination node)"""

    @staticmethod
    def forward(ctx, s, rowptr, scale):
        lib = _lib.load()
        s = _f32c(s).contiguous()
        alpha = torch.empty_like(s)
        n_rows = rowptr.numel() - 1
        with profiling.span("segment_softmax_fwd_f32", s.numel() * 8, 0):
            check(lib.plnlp_segment_softmax_fwd_f32(ptr(rowptr), n_rows, ptr(s), float(scale), ptr(alpha), stream()),
                  "plnlp_segment_softmax_fwd_f32")
        ctx.scale = float(scale)
        ctx.save_for_backward(alpha, rowptr)
        return alpha

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        alpha, rowptr = ctx.saved_tensors
        g = _f32c(g).contiguous()
        ds = torch.empty_like(alpha)
        with profiling.span("segment_softmax_bwd_f32", alpha.numel() * 12, 0):
            check(lib.plnlp_segment_softmax_bwd_f32(ptr(rowptr), rowptr.numel() - 1, ptr(alpha), ptr(g), ctx.scale,
                                                    ptr(ds), stream()), "plnlp_segment_softmax_bwd_f32")
        return ds, None, None


class SpMMValues(torch.autograd.Function):
    """out = A(alpha) @ v where alpha holds one value per stored entry of ``adj`` (CSR order): the SpMM kernel
    with the attention weights as its values.  Backward: d v = A(alpha)^T g (the transposed plan with the
    permuted weights), d alpha[e] = <g[row_e], v[col_e]> (the edge-dot kernel over the entry list)."""

    @staticmethod
    def forward(ctx, alpha, v, adj):
        from .graph import _share_plan
        st = structure_of(adj)
        alpha = _f32c(alpha).contiguous()
        out = spmm_raw(_share_plan(st.fwd, alpha), v, use_val=True, div_rows=False)
        ctx.st = st
        ctx.save_for_backward(alpha, v)
        return out

    @staticmethod
    def backward(ctx, g):
        from .graph import _share_plan
        alpha, v = ctx.saved_tensors
        st = ctx.st
        g = _rowmajor(g)
        dalpha = dv = None
        if ctx.needs_input_grad[0]:
            dalpha = edge_dot_raw(torch.cat([g, v], 0), st.entry_pairs())
        if ctx.needs_input_grad[1]:
            dv = spmm_raw(_share_plan(st.bwd, alpha[st.t_perm].contiguous()), g, use_val=True, div_rows=False)
        return dalpha, dv, None


def attn_score_raw(plan, q, k):
    """score[e] = <q[row(e)], k[col(e)]> for every stored entry of the CSR block behind ``plan`` (an SpMM plan over
    the whole block, ``Structure.fwd`` / ``.bwd``), in CSR order; q [n_rows, F] and k [n_cols, F] may be column slices
    with a leading dimension"""
    lib = _lib.load()
    q, k = _rowmajor(q), _rowmajor(k)
    if getattr(plan, "subset", False):
        raise RuntimeError("attn_score_raw needs the plan of a whole block, not a row subset")
    if q.size(0) != plan.n_rows or k.size(0) != plan.n_cols or q.size(1) != k.size(1):
        raise RuntimeError(f"attention score shapes: block {plan.n_rows}x{plan.n_cols}, q {tuple(q.shape)}, "
                           f"k {tuple(k.shape)}")
    F = q.size(1)
    score = torch.empty(plan.nnz, dtype=torch.float32, device=q.device)
    with profiling.span(f"attn_score_csr_f32 F={F}", plan.nnz * (F * 4 + 8) + plan.n_rows * F * 4, 2 * plan.nnz * F):
        check(lib.plnlp_attn_score_csr_f32(ptr(plan.item_ptr), ptr(plan.item_row), plan.n_items, ptr(plan.col),
                                           ptr(q), _ld(q), ptr(k), _ld(k), F, ptr(score), stream()),
              "plnlp_attn_score_csr_f32")
    return score


def block_attention_fwd(q, k, v, st, scale):
    """the attention of a CSR row block with separate query and key / value tables -> (score [nnz], alpha [nnz],
    agg [n_rows, F]): per-entry scores (attn_score_raw), the per-row softmax, and the SpMM with the weights as values"""
    from .graph import _share_plan
    if st.fwd.nnz == 0:                       # an empty block (padding rows only): nothing to attend to
        s = torch.empty(0, dtype=torch.float32, device=q.device)
        return s, s, torch.zeros(st.n_rows, q.size(1), dtype=torch.float32, device=q.device)
    s = attn_score_raw(st.fwd, q, k)
    alpha = torch.empty_like(s)
    lib = _lib.load()
    with profiling.span("segment_softmax_fwd_f32", s.numel() * 8, 0):
        check(lib.plnlp_segment_softmax_fwd_f32(ptr(st.rowptr), st.n_rows, ptr(s), float(scale), ptr(alpha), stream()),
              "plnlp_segment_softmax_fwd_f32")
    agg = spmm_raw(_share_plan(st.fwd, alpha), v, use_val=True, div_rows=False)
    return s, alpha, agg


class BlockAttention(torch.autograd.Function):
    """agg = softmax_row(scale <q_i, k_j>) v_j over the stored entries of a row block ``adj`` [n_q, n_k] (the
    row-partitioned TransformerConv).  q [n_q, F] holds the block's own rows; kv [n_k, 2F] = [k | v] holds every
    gathered row.  Backward, on the plans the block's Structure already has (fixed order, deterministic):
    dalpha = score(g, v), ds = softmax backward, dq = A(ds) k, dk = A(ds)^T q, dv = A(alpha)^T g -- dk and dv
    written side by side into one [n_k, 2F] gradient of kv."""

    @staticmethod
    def forward(ctx, q, kv, adj, scale):
        st = structure_of(adj)
        F = q.size(1)
        _, alpha, agg = block_attention_fwd(q, kv[:, :F], kv[:, F:], st, scale)
        ctx.st, ctx.scale = st, float(scale)
        ctx.save_for_backward(q, kv, alpha)
        return agg

    @staticmethod
    def backward(ctx, g):
        from .graph import _share_plan
        q, kv, alpha = ctx.saved_tensors
        st, F = ctx.st, q.size(1)
        if st.fwd.nnz == 0:
            return torch.zeros_like(q), torch.zeros_like(kv), None, None
        g = _rowmajor(g)
        k, v = kv[:, :F], kv[:, F:]
        dalpha = attn_score_raw(st.fwd, g, v)
        ds = torch.empty_like(alpha)
        lib = _lib.load()
        with profiling.span("segment_softmax_bwd_f32", alpha.numel() * 12, 0):
            check(lib.plnlp_segment_softmax_bwd_f32(ptr(st.rowptr), st.n_rows, ptr(alpha), ptr(dalpha), ctx.scale,
                                                    ptr(ds), stream()), "plnlp_segment_softmax_bwd_f32")
        dq = spmm_raw(_share_plan(st.fwd, ds), k, use_val=True, div_rows=False) if ctx.needs_input_grad[0] else None
        dkv = None
        if ctx.needs_input_grad[1]:
            dkv = torch.empty(kv.size(0), 2 * F, dtype=torch.float32, device=kv.device)
            spmm_raw(_share_plan(st.bwd, ds[st.t_perm].contiguous()), q, use_val=True, div_rows=False, out=dkv[:, :F])
            spmm_raw(_share_plan(st.bwd, alpha[st.t_perm].contiguous()), g, use_val=True, div_rows=False,
                     out=dkv[:, F:])
        return dq, dkv, None, None


def block_attention(q, kv, adj, scale):
    return BlockAttention.apply(q, kv, adj, float(scale))


class AddLinear(torch.autograd.Function):
    """Y = act( x @ W^T + bias + addend ): the root / skip connection of a conv accumulated onto its aggregate in
    the GEMM epilogue (beta = 1), with the layer's relu + dropout fused"""

    @staticmethod
    def forward(ctx, x, W, bias, addend, act, drop_p, seed):
        Y = gemm_raw(x, W, transb=True, C=addend.clone(), beta=1.0, bias=bias, act=act, drop_p=drop_p, seed=seed)
        ctx.act, ctx.drop_p, ctx.has_bias = act, drop_p, bias is not None
        ctx.save_for_backward(Y if act == ACT_RELU else None, x, W)
        return Y

    @staticmethod
    def backward(ctx, g):
        Y, x, W = ctx.saved_tensors
        g = _rowmajor(g)
        if Y is not None:
            g = relu_drop_bwd_raw(Y, g, 1.0 / (1.0 - ctx.drop_p))
        gx = gemm_raw(g, W) if ctx.needs_input_grad[0] else None
        gW = gemm_raw(g, x, transa=True) if ctx.needs_input_grad[1] else None
        gb = colsum_raw(g) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return gx, gW, gb, (g if ctx.needs_input_grad[3] else None), None, None, None


# ---------------------------------------------------------------------------
# samplers and ranking (no autograd)
# ---------------------------------------------------------------------------
def local_neg_sample_raw(pos_edges, num_nodes, num_neg, seed):
    lib = _lib.load()
    pos_edges = _edges_i64(pos_edges)
    E = pos_edges.size(0)
    out = torch.empty(E, num_neg, 2, dtype=torch.int64, device=pos_edges.device)
    check(lib.plnlp_local_neg_sample(ptr(pos_edges), E, int(num_nodes), int(num_neg), int(seed), ptr(out),
                                     stream()), "plnlp_local_neg_sample")
    return out


def global_neg_candidates_raw(edge_ids_sorted, num_nodes, n_cand, seed):
    """-> (cand_ids [n_cand] int64, keep [n_cand] uint8)"""
    lib = _lib.load()
    dev = edge_ids_sorted.device
    table_size = 1
    while table_size < 2 * max(n_cand, 1):
        table_size *= 2
    keys = torch.full((table_size,), -1, dtype=torch.int64, device=dev)
    first = torch.full((table_size,), -1, dtype=torch.int32, device=dev)
    cand = torch.empty(n_cand, dtype=torch.int64, device=dev)
    keep = torch.empty(n_cand, dtype=torch.uint8, device=dev)
    check(lib.plnlp_global_neg_candidates(ptr(edge_ids_sorted), edge_ids_sorted.numel(), int(num_nodes), n_cand,
                                          int(seed), ptr(cand), ptr(keys), ptr(first), table_size, stream()),
          "plnlp_global_neg_candidates")
    check(lib.plnlp_global_neg_keep(ptr(cand), n_cand, ptr(keys), ptr(first), table_size, ptr(keep), stream()),
          "plnlp_global_neg_keep")
    return cand, keep


def kth_largest_raw(x, K):
    lib = _lib.load()
    x = _f32c(x).reshape(-1).contiguous()
    out = torch.empty(1, dtype=torch.float32, device=x.device)
    ws = workspace.get("kth", 8192, x.device)
    check(lib.plnlp_kth_largest_f32(ptr(x), x.numel(), int(K), ptr(out), ptr(ws), 8192, stream()),
          "plnlp_kth_largest_f32")
    return out


def count_greater_raw(x, thresh):
    lib = _lib.load()
    x = _f32c(x).reshape(-1).contiguous()
    cnt = torch.empty(1, dtype=torch.int64, device=x.device)
    check(lib.plnlp_count_greater_f32(ptr(x), x.numel(), ptr(thresh), ptr(cnt), stream()),
          "plnlp_count_greater_f32")
    return cnt


def mrr_counts_raw(pos, neg):
    lib = _lib.load()
    pos = _f32c(pos).reshape(-1).contiguous()
    neg = _rowmajor(neg)
    S, K = neg.shape
    gt = torch.empty(S, dtype=torch.int32, device=pos.device)
    ge = torch.empty(S, dtype=torch.int32, device=pos.device)
    check(lib.plnlp_mrr_counts_f32(ptr(pos), ptr(neg), _ld(neg), S, K, ptr(gt), ptr(ge), stream()),
          "plnlp_mrr_counts_f32")
    return gt, ge


def _cand_ids(cand, N):
    if cand.dtype != torch.int64 or cand.dim() != 1 or cand.numel() != N:
        raise RuntimeError("cand must be int64 with one entry per score column")
    return cand.contiguous()


def score_mask_raw(s, nodes, rowptr=None, col=None, exclude_self=True, col0=0, cand=None):
    """in place: s[q, j] = -inf for the known links j of nodes[q] (CSR rowptr int64 / col int32) and, with
    ``exclude_self``, for j = nodes[q].  The chunk covers the global candidate ids [col0, col0 + N): col and nodes
    are global ids.  ``cand`` (int64 [N], strictly ascending global ids): column j is the node cand[j] instead."""
    lib = _lib.load()
    if _f32c(s).dim() != 2 or s.stride(1) != 1:
        raise RuntimeError("the score chunk must be a 2-D fp32 matrix with unit column stride (masked in place)")
    nodes = nodes.contiguous()
    if nodes.dtype != torch.int64 or nodes.numel() != s.size(0):
        raise RuntimeError("nodes must be int64 with one entry per score row")
    if (rowptr is None) != (col is None):
        raise RuntimeError("rowptr and col come together")
    if col is not None and (rowptr.dtype != torch.int64 or col.dtype != torch.int32):
        raise RuntimeError("the known-link CSR is int64 rowptr + int32 col")
    Q, N = s.shape
    if cand is not None:
        cand = _cand_ids(cand, N)
        with profiling.span("score_mask_f32", 0, 0):
            check(lib.plnlp_score_mask_cand_f32(ptr(s), _ld(s), Q, N, ptr(cand), ptr(nodes), ptr(rowptr), ptr(col),
                                                int(bool(exclude_self)), stream()), "plnlp_score_mask_cand_f32")
        return s
    with profiling.span("score_mask_f32", 0, 0):
        check(lib.plnlp_score_mask_cols_f32(ptr(s), _ld(s), Q, N, int(col0), ptr(nodes), ptr(rowptr), ptr(col),
                                            int(bool(exclude_self)), stream()), "plnlp_score_mask_cols_f32")
    return s


def topk_rows_raw(s, k, target=None, target_score=None, col0=0, cand=None):
    """per row of s [Q, N]: the k largest finite entries (score descending, then column ascending; tail (-1, -inf))
    and, with ``target``, the filtered rank counts gt / ge against ``target_score``.  -> (ids int64 [Q, k] or None,
    scores [Q, k] or None, gt int32 [Q] or None, ge int32 [Q] or None).  One read of s.  The chunk covers the
    global candidate ids [col0, col0 + N): ids, ties and ``target`` are global ids.  ``cand`` (int64 [N], strictly
    ascending global ids, col0 = 0): column j is the node cand[j]; ids are cand[j], ``target`` stays a global id."""
    lib = _lib.load()
    s = _rowmajor(s)
    Q, N = s.shape
    dev = s.device
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev) if k > 0 else None
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev) if k > 0 else None
    gt = ge = None
    if target is not None:
        target = target.contiguous()
        target_score = _f32c(target_score).contiguous()
        if target.dtype != torch.int64 or target.numel() != Q or target_score.numel() != Q:
            raise RuntimeError("target (int64) and target_score need one entry per score row")
        gt = torch.empty(Q, dtype=torch.int32, device=dev)
        ge = torch.empty(Q, dtype=torch.int32, device=dev)
    nbytes = max(int(lib.plnlp_topk_rows_workspace_bytes(Q, N, max(int(k), 0))), 16)
    ws = workspace.get("topk_rows", nbytes, dev)
    if cand is not None:
        cand = _cand_ids(cand, N)
        with profiling.span(f"topk_rows_f32 k={k}", Q * N * 4, 0):
            check(lib.plnlp_topk_rows_cand_f32(ptr(s), _ld(s), Q, N, int(col0), int(k), ptr(target),
                                               ptr(target_score), ptr(ids), ptr(scores), ptr(gt), ptr(ge), ptr(ws),
                                               nbytes, ptr(cand), stream()), "plnlp_topk_rows_cand_f32")
        return ids, scores, gt, ge
    with profiling.span(f"topk_rows_f32 k={k}", Q * N * 4, 0):
        check(lib.plnlp_topk_rows_cols_f32(ptr(s), _ld(s), Q, N, int(col0), int(k), ptr(target), ptr(target_score),
                                           ptr(ids), ptr(scores), ptr(gt), ptr(ge), ptr(ws), nbytes, stream()),
              "plnlp_topk_rows_cols_f32")
    return ids, scores, gt, ge


def topk_merge_raw(ids_in, scores_in, k):
    """the k best entries per row of R sorted per-shard lists ids_in int64 / scores_in fp32 [R, Q, k_in] (dead
    entries: id -1) -> (ids int64 [Q, k], scores [Q, k]) under the tie rule of ``topk_rows_raw``"""
    lib = _lib.load()
    if ids_in.dim() != 3 or ids_in.shape != scores_in.shape or ids_in.dtype != torch.int64:
        raise RuntimeError("ids_in (int64) and scores_in must both be [R, Q, k_in]")
    ids_in, scores_in = ids_in.contiguous(), _f32c(scores_in).contiguous()
    R, Q, k_in = ids_in.shape
    ids = torch.empty(Q, k, dtype=torch.int64, device=ids_in.device)
    scores = torch.empty(Q, k, dtype=torch.float32, device=ids_in.device)
    with profiling.span(f"topk_merge_f32 R={R}", ids_in.numel() * 12, 0):
        check(lib.plnlp_topk_merge_f32(ptr(ids_in), ptr(scores_in), R, Q, k_in, int(k), ptr(ids), ptr(scores),
                                       stream()), "plnlp_topk_merge_f32")
    return ids, scores


def link_heuristic_raw(rowptr, col, weight, edges):
    """fp64 [P]: for every pair edges[p] = (u, v) (int64 [P, 2], ids in [-1, n); a pair with a negative id has no
    common neighbour and gives 0) the sum of ``weight[w]`` (fp64 [n]) over the common neighbours w of rows u and v of
    the cleaned CSR (rowptr int64 [n + 1], col int32), or their count when ``weight`` is None (heuristics.py)"""
    lib = _lib.load()
    if rowptr.dtype != torch.int64 or col.dtype != torch.int32 or edges.dtype != torch.int64:
        raise RuntimeError("link_heuristic_raw: rowptr and edges must be int64, col int32")
    if weight is not None and weight.dtype != torch.float64:
        raise RuntimeError("link_heuristic_raw: weight must be fp64")
    P = edges.size(0)
    out = torch.empty(P, dtype=torch.float64, device=edges.device)
    with profiling.span("link_heuristic_f64", P * 16, 0):
        check(lib.plnlp_link_heuristic_f64(ptr(rowptr.contiguous()), ptr(col.contiguous()), rowptr.numel() - 1,
                                           col.numel(), ptr(None if weight is None else weight.contiguous()),
                                           ptr(edges.contiguous()), P, ptr(out), stream()), "plnlp_link_heuristic_f64")
    return out


def common_neighbour_list_raw(rowptr, col, edges, out_ptr):
    """int32 [out_ptr[-1]]: the common neighbours of every pair edges[p] (int64 [P, 2], ids in [-1, n); a negative id
    has none) in rows of the cleaned CSR (rowptr int64 [n + 1], col int32), ascending, at [out_ptr[p], out_ptr[p + 1])
    -- ``out_ptr`` int64 [P + 1] the running sum of the ``link_heuristic_raw`` counts (heuristics.py)"""
    lib = _lib.load()
    if rowptr.dtype != torch.int64 or col.dtype != torch.int32 or edges.dtype != torch.int64 \
            or out_ptr.dtype != torch.int64:
        raise RuntimeError("common_neighbour_list_raw: rowptr, edges and out_ptr must be int64, col int32")
    P = edges.size(0)
    if out_ptr.numel() != P + 1:
        raise RuntimeError("common_neighbour_list_raw: out_ptr must have P + 1 entries")
    total = int(out_ptr[-1])
    out = torch.empty(total, dtype=torch.int32, device=edges.device)
    if total == 0:
        return out
    with profiling.span("common_neighbour_list", P * 16 + total * 4, 0):
        check(lib.plnlp_common_neighbour_list(ptr(rowptr.contiguous()), ptr(col.contiguous()), rowptr.numel() - 1,
                                              col.numel(), ptr(edges.contiguous()), P, ptr(out_ptr.contiguous()),
                                              ptr(out), stream()), "plnlp_common_neighbour_list")
    return out


CN_CHUNK = 256      # entries of a common-neighbour list per SpMM work item: fixes the order of every sum


def _cn_plan(rowptr, col, n_rows, n_cols):
    from .graph import build_plan
    return build_plan(rowptr, col, None, n_rows, n_cols, chunk=CN_CHUNK)


class CommonNeighbourSum(torch.autograd.Function):
    """c[p] = sum of h[w] over w in col[rowptr[p] .. rowptr[p + 1]) (the NCN predictor's common-neighbour term): the
    SpMM kernel with the P x N 0/1 matrix of the lists, planned per call at the fixed chunk ``CN_CHUNK`` so every bit
    of c depends on the list and h only (not on the batch).  Backward: C^T g on the transposed plan (entries sorted by
    (col, row)), built only when h needs a gradient -- deterministic, no atomics."""

    @staticmethod
    def forward(ctx, h, rowptr, col):
        P, n = rowptr.numel() - 1, h.size(0)
        ctx.save_for_backward(rowptr, col)
        ctx.n = n
        if col.numel() == 0:
            return torch.zeros(P, h.size(1), dtype=torch.float32, device=h.device)
        with profiling.span("torch: common-neighbour SpMM plan"):
            plan = _cn_plan(rowptr, col, P, n)
        with profiling.span("NCN: common-neighbour SpMM forward"):
            return spmm_raw(plan, h, use_val=False, div_rows=False)

    @staticmethod
    def backward(ctx, g):
        rowptr, col = ctx.saved_tensors
        P, n = rowptr.numel() - 1, ctx.n
        if not ctx.needs_input_grad[0]:
            return None, None, None
        if col.numel() == 0:
            return torch.zeros(n, g.size(1), dtype=torch.float32, device=g.device), None, None
        with profiling.span("torch: transposed common-neighbour SpMM plan"):
            c = col.to(torch.int64)
            row = torch.repeat_interleave(torch.arange(P, device=c.device), rowptr[1:] - rowptr[:-1],
                                          output_size=c.numel())
            perm = torch.argsort(c * P + row, stable=True)
            t_rowptr = torch.zeros(n + 1, dtype=torch.int64, device=c.device)
            t_rowptr[1:] = torch.cumsum(torch.bincount(c, minlength=n), 0)
            plan = _cn_plan(t_rowptr, row[perm], n, P)
        with profiling.span("NCN: common-neighbour SpMM backward (C^T g)"):
            return spmm_raw(plan, _rowmajor(g), use_val=False, div_rows=False), None, None


def common_neighbour_sum(h, cn):
    """``CommonNeighbourSum`` of h [N, H] over the lists ``cn = (rowptr int64 [P + 1], col)`` (col: rows of h)"""
    rowptr, col = cn
    if rowptr.dtype != torch.int64 or rowptr.dim() != 1 or col.dim() != 1:
        raise RuntimeError("common_neighbour_sum: cn must be (rowptr int64 [P + 1], col [nnz])")
    return CommonNeighbourSum.apply(_rowmajor(h), rowptr, col)


def _two_hop_args(rowptr, col, nodes, W, col0, cand):
    if rowptr.dtype != torch.int64 or col.dtype != torch.int32 or nodes.dtype != torch.int64:
        raise RuntimeError("two_hop: rowptr and nodes must be int64, col int32")
    if cand is not None:
        cand = _cand_ids(cand, W)
        if col0 != 0:
            raise RuntimeError("two_hop: a candidate chunk has col0 = 0")
    return rowptr.contiguous(), col.contiguous(), nodes.contiguous(), cand


def two_hop_mark_raw(rowptr, col, rrowptr, rcol, nodes, W, col0=0, cand=None):
    """int32 [Qc, ceil(W / 32)] bitmap (read as uint32): bit c of row q is set when column c's node -- col0 + c, or
    cand[c] -- shares a neighbour with nodes[q]: it lies in row w of the transposed table (rrowptr int64, rcol int32)
    for some w in row nodes[q] of the cleaned table (rowptr int64, col int32) (heuristics.py)"""
    lib = _lib.load()
    rowptr, col, nodes, cand = _two_hop_args(rowptr, col, nodes, W, col0, cand)
    if rrowptr.dtype != torch.int64 or rcol.dtype != torch.int32 or rrowptr.numel() != rowptr.numel():
        raise RuntimeError("two_hop_mark_raw: the transposed table is int64 rrowptr + int32 rcol over the same nodes")
    Qc = nodes.numel()
    bitmap = torch.zeros(Qc, (W + 31) // 32, dtype=torch.int32, device=nodes.device)
    if col.numel() == 0 or rcol.numel() == 0:         # a table without entries (an empty block) reaches nothing
        return bitmap
    item_ptr = torch.zeros(Qc + 1, dtype=torch.int64, device=nodes.device)
    item_ptr[1:] = torch.cumsum(rowptr[nodes + 1] - rowptr[nodes], 0)
    with profiling.span("two_hop_mark", 0, 0):
        check(lib.plnlp_two_hop_mark(ptr(rowptr), ptr(col), ptr(rrowptr.contiguous()), ptr(rcol.contiguous()),
                                     rowptr.numel() - 1, ptr(nodes), ptr(item_ptr), Qc, int(col0), int(W), ptr(cand),
                                     ptr(bitmap), stream()), "plnlp_two_hop_mark")
    return bitmap


def two_hop_score_raw(rowptr, col, weight, nodes, bitmap, W, col0=0, cand=None, dtype=torch.float32):
    """S [Qc, W] in ``dtype`` (fp32: each sum rounded once; fp64: kept): for every set bit of ``bitmap``
    (``two_hop_mark_raw``) the ``link_heuristic_raw`` value of the pair (nodes[q], column c's node), bit for bit; 0
    elsewhere"""
    lib = _lib.load()
    rowptr, col, nodes, cand = _two_hop_args(rowptr, col, nodes, W, col0, cand)
    if weight is not None and weight.dtype != torch.float64:
        raise RuntimeError("two_hop_score_raw: weight must be fp64")
    Qc = nodes.numel()
    if bitmap.dtype != torch.int32 or tuple(bitmap.shape) != (Qc, (W + 31) // 32):
        raise RuntimeError("two_hop_score_raw: bitmap must be the int32 [Qc, ceil(W / 32)] of two_hop_mark_raw")
    s = torch.zeros(Qc, W, dtype=dtype, device=nodes.device)
    f = {torch.float32: lib.plnlp_two_hop_score_f32, torch.float64: lib.plnlp_two_hop_score_f64}[dtype]
    with profiling.span(f"two_hop_score_{'f32' if dtype == torch.float32 else 'f64'}", 0, 0):
        check(f(ptr(rowptr), ptr(col), rowptr.numel() - 1, col.numel(),
                ptr(None if weight is None else weight.contiguous()), ptr(nodes), Qc, int(col0), int(W), ptr(cand),
                ptr(bitmap.contiguous()), ptr(s), W, stream()), "plnlp_two_hop_score")
    return s


def _f64_bits(v):
    import struct
    return struct.unpack("<Q", struct.pack("<d", float(v)))[0]


def propagate_raw(plan, weight, x, src, c, b, live_in=None, r0=0, y=None, live_out=None):
    """one hop of the path scores (paths.py): for every row j of [r0, r0 + plan.n_rows), y[j - r0, a] =
    fp32(c * sum over the row's entries w of weight[w] * x[w, a] + (b if src[a] == j else 0)) in fp64, summed in the
    order of ``plan`` (graph.build_plan over the rows).  x fp32 [n, B] node-major (B in 32, 64, 128, 256, row stride
    free), weight fp64 [n] or None (1), src int64 [B] (-1: padding column), live_in uint8 [n] or None (every row
    read).  -> (y fp32 [rows, B], live_out uint8 [rows]); ``y`` / ``live_out`` may be given (y's rows contiguous)."""
    lib = _lib.load()
    B = x.size(1)
    rows = plan.n_rows
    if x.dtype != torch.float32 or x.stride(1) != 1 or src.dtype != torch.int64 or src.numel() != B:
        raise RuntimeError("propagate_raw: x must be fp32 [n, B] with unit column stride and src int64 [B]")
    if weight is not None and weight.dtype != torch.float64:
        raise RuntimeError("propagate_raw: weight must be fp64")
    if live_in is not None and (live_in.dtype != torch.uint8 or live_in.numel() < x.size(0)):
        raise RuntimeError("propagate_raw: live_in must be uint8 [n]")
    if y is None:
        y = torch.empty(rows, B, dtype=torch.float32, device=x.device)
    if live_out is None:
        live_out = torch.empty(rows, dtype=torch.uint8, device=x.device)
    partial = None
    if plan.n_fix:
        partial = workspace.get("propagate", plan.n_partial * B * 8, x.device).view(torch.float64)
    with profiling.span(f"propagate_f32 B={B}", 0, 0):
        check(lib.plnlp_propagate_f32(ptr(plan.item_ptr), ptr(plan.item_row), ptr(plan.item_slot), plan.n_items,
                                      ptr(plan.col), ptr(plan.fix_ptr), ptr(plan.fix_row), plan.n_fix, ptr(partial),
                                      ptr(None if weight is None else weight.contiguous()), ptr(x), x.stride(0),
                                      ptr(src.contiguous()), B, _f64_bits(c), _f64_bits(b), ptr(live_in),
                                      ptr(live_out), int(r0), rows, ptr(y), y.stride(0), stream()),
              "plnlp_propagate_f32")
    return y, live_out
