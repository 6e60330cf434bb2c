"""torch.autograd bindings of the C ABI (include/gcgcn_b200.h).

PyTorch is plumbing here: it owns device memory, the current CUDA stream and the autograd
tape.  Every numerical operation of the hot path is one of this package's own CUDA kernels,
reached through ``_lib.call``.  CPU tensors are rejected -- there is no fallback.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch.autograd import Function

from . import _lib
from .batch import PairTables, PoolTable, RaggedBatch

D = 128

_WS: dict = {}


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Per-(device, stream) scratch arena handed to the library (it never allocates)."""
    key = (device.index, _stream(device))
    t = _WS.get(key)
    if t is None or t.numel() < nbytes:
        t = torch.empty(int(nbytes) + (1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = t
    return t


def _ws_for(batch: RaggedBatch, heads: int, device):
    n = _lib.load().gcgcn_workspace_bytes(batch.total_nodes, batch.total_pairs, heads)
    t = workspace(device, n)
    return t.data_ptr(), t.numel()


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.GcgcnError(f"{name} is a CPU tensor: gcgcn_b200 runs on CUDA only (no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def _edge(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _lib.GcgcnError(f"{name} is a CPU tensor: gcgcn_b200 runs on CUDA only (no CPU fallback)")
    if t.dtype == torch.float32:
        return t.contiguous(), _lib.F32
    if t.dtype == torch.bfloat16:
        return t.contiguous(), _lib.BF16
    raise _lib.GcgcnError(f"{name}: edge features must be float32 or bfloat16, got {t.dtype}")


# ------------------------------------------------------------------------------- a1 pooling
class PoolFn(Function):
    """x0 = node_pos @ ctx as a CSR gather (replaces G:297-298)."""

    @staticmethod
    def forward(ctx, context: torch.Tensor, table: PoolTable):
        context = _cuda(context, "context_output")
        if context.shape != (table.total_tokens, D):
            raise _lib.GcgcnError(f"context must be [{table.total_tokens}, {D}], got {tuple(context.shape)}")
        x0 = torch.empty(table.total_nodes, D, device=context.device, dtype=torch.float32)
        _lib.call("gcgcn_pool_fwd", _p(context), _p(table.ent_ptr), _p(table.tok_idx), _p(table.w),
                  table.total_nodes, _p(x0), _stream(context.device))
        ctx.table = table
        return x0

    @staticmethod
    def backward(ctx, dx0):
        t = ctx.table
        dx0 = _cuda(dx0, "dx0")
        dctx = torch.empty(t.total_tokens, D, device=dx0.device, dtype=torch.float32)
        _lib.call("gcgcn_pool_bwd", _p(dx0), _p(t.tok_ptr), _p(t.ent_idx), _p(t.w_t), t.total_tokens,
                  _p(dctx), _stream(dx0.device))
        return dctx, None


# ------------------------------------------------------------------------------- edge mean
class EdgeMeanFn(Function):
    """ebar_i = mean_j e_ij -- all GraphConv needs from the edge tensor (G:40-41 collapsed)."""

    @staticmethod
    def forward(ctx, e: torch.Tensor, batch: RaggedBatch):
        e, dt = _edge(e, "edge_feat")
        ebar = torch.empty(batch.total_nodes, D, device=e.device, dtype=torch.float32)
        _lib.call("gcgcn_edge_mean_fwd", batch.ref, _p(e), dt, _p(ebar), _stream(e.device))
        ctx.batch, ctx.dt, ctx.shape, ctx.edtype = batch, dt, e.shape, e.dtype
        return ebar

    @staticmethod
    def backward(ctx, debar):
        debar = _cuda(debar, "debar")
        de = torch.empty(ctx.shape, device=debar.device, dtype=ctx.edtype)
        _lib.call("gcgcn_edge_mean_bwd", ctx.batch.ref, _p(debar), ctx.dt, _p(de), _stream(debar.device))
        return de, None


# ------------------------------------------------------------------------------- a2 GAT
class GatFn(Function):
    """GATAttention.forward (G:154-168) + the edge mean of the same pass.  Returns (A, ebar)."""

    @staticmethod
    def forward(ctx, x, e, u, v, c, batch: RaggedBatch, mask_u8, apply_mask: bool, keep):
        x = _cuda(x, "node_feat")
        e, dt = _edge(e, "edge_feat")
        u, v, c = _cuda(u, "u"), _cuda(v, "v"), _cuda(c, "c")
        dev = x.device
        P = torch.empty(batch.total_pairs, device=dev, dtype=torch.float32)
        A = P if keep is None else torch.empty_like(P)
        ebar = torch.empty(batch.total_nodes, D, device=dev, dtype=torch.float32)
        if keep is not None:
            keep = _cuda(keep, "keep")
        if mask_u8 is not None:
            mask_u8 = _cuda(mask_u8, "mask", torch.uint8)
        ws, wsb = _ws_for(batch, 1, dev)
        _lib.call("gcgcn_gat_fwd", batch.ref, _p(x), _p(e), dt, _p(u), _p(v), _p(c), _p(mask_u8),
                  int(bool(apply_mask)), _p(keep), _p(P), _p(A), _p(ebar), ws, wsb, _stream(dev))
        ctx.save_for_backward(x, e, u, v, P, keep, mask_u8)
        ctx.batch, ctx.dt, ctx.apply_mask = batch, dt, bool(apply_mask)
        return A, ebar

    @staticmethod
    def backward(ctx, dA, debar):
        x, e, u, v, P, keep, mask_u8 = ctx.saved_tensors
        bt, dev = ctx.batch, x.device
        dA = torch.zeros_like(P) if dA is None else _cuda(dA, "dA")
        debar = None if debar is None else _cuda(debar, "debar")
        dx = torch.empty_like(x)
        de = torch.empty_like(e)
        duvc = torch.empty(2 * D + 1, device=dev)          # [du | dv | dc] contiguous: GatCollapseFn consumes it as is
        du, dv, dc = duvc[:D], duvc[D:2 * D], duvc[2 * D:]
        ws, wsb = _ws_for(bt, 1, dev)
        _lib.call("gcgcn_gat_bwd", bt.ref, _p(x), _p(e), ctx.dt, _p(u), _p(v), _p(mask_u8),
                  int(ctx.apply_mask), _p(keep), _p(P), _p(dA), _p(debar), _p(dx), _p(de), _p(du),
                  _p(dv), _p(dc), ws, wsb, _stream(dev))
        return dx, de, du, dv, dc.reshape(()), None, None, None, None


# ------------------------------------------------------------------------------- a5 MHA
class MhaFn(Function):
    """MultiHeadAttention.forward (G:133-142).  Returns A [H, total_pairs]."""

    @staticmethod
    def forward(ctx, x, Wq, bq, batch: RaggedBatch, heads: int, keep):
        x, Wq, bq = _cuda(x, "node_feat"), _cuda(Wq, "Wq"), _cuda(bq, "bq")
        dev = x.device
        q = torch.empty(batch.total_nodes, D, device=dev, dtype=torch.float32)
        P = torch.empty(heads, batch.total_pairs, device=dev, dtype=torch.float32)
        A = P if keep is None else torch.empty_like(P)
        if keep is not None:
            keep = _cuda(keep, "keep")
        ws, wsb = _ws_for(batch, heads, dev)
        _lib.call("gcgcn_mha_fwd", batch.ref, heads, _p(x), _p(Wq), _p(bq), _p(keep), _p(q), _p(P), _p(A),
                  ws, wsb, _stream(dev))
        ctx.save_for_backward(x, Wq, q, P, keep)
        ctx.batch, ctx.heads = batch, heads
        return A

    @staticmethod
    def backward(ctx, dA):
        x, Wq, q, P, keep = ctx.saved_tensors
        bt, dev = ctx.batch, x.device
        dA = _cuda(dA, "dA")
        dx = torch.empty_like(x)
        dWq = torch.empty_like(Wq)
        dbq = torch.empty(D, device=dev)
        ws, wsb = _ws_for(bt, ctx.heads, dev)
        _lib.call("gcgcn_mha_bwd", bt.ref, ctx.heads, _p(x), _p(Wq), _p(q), _p(keep), _p(P), _p(dA),
                  _p(dx), _p(dWq), _p(dbq), ws, wsb, _stream(dev))
        return dx, dWq, dbq, None, None, None


# ------------------------------------------------------------------------------- a3/a4/a6 stack
class StackFn(Function):
    """Dense-connected GraphConv stack + output linear (G:36-50, 63-80, 97-120)."""

    @staticmethod
    def forward(ctx, x, ebar, A, WnX, We, Winner, Wout, bout, batch: RaggedBatch, heads: int,
                layers: int, in_dim: int, slab: int, flags: int, keep):
        x, ebar, A = _cuda(x, "node_feat"), _cuda(ebar, "ebar"), _cuda(A, "adj_matrix")
        WnX, We = _cuda(WnX, "WnX"), _cuda(We, "We")
        Winner = None if Winner is None else _cuda(Winner, "Winner")
        linear = bool(flags & _lib.STACK_LINEAR)
        if linear:
            Wout, bout = _cuda(Wout, "Wout"), _cuda(bout, "bout")
        if keep is not None:
            keep = _cuda(keep, "keep")
        dev, M, HD = x.device, batch.total_nodes, heads * slab
        if A.numel() != heads * batch.total_pairs:
            raise _lib.GcgcnError(f"attention has {A.numel()} entries, expected {heads} x {batch.total_pairs}")
        Z = torch.empty(M, HD, device=dev)
        G = torch.empty(M, HD, device=dev)
        F = torch.empty(M, HD, device=dev) if linear else None
        y = torch.empty(M, D if linear else slab, device=dev)
        ws, wsb = _ws_for(batch, heads, dev)
        _lib.call("gcgcn_graphconv_stack_fwd", batch.ref, heads, layers, in_dim, slab, flags, _p(x), _p(ebar),
                  _p(A), _p(WnX), _p(We), _p(Winner), _p(Wout), _p(bout), _p(keep), _p(Z), _p(G), _p(F),
                  _p(y), ws, wsb, _stream(dev))
        ctx.save_for_backward(x, ebar, A, WnX, We, Winner, Wout, keep, Z, G, F)
        ctx.cfg = (batch, heads, layers, in_dim, slab, flags)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, ebar, A, WnX, We, Winner, Wout, keep, Z, G, F = ctx.saved_tensors
        batch, heads, layers, in_dim, slab, flags = ctx.cfg
        dev = x.device
        dy = _cuda(dy, "dy")
        linear = bool(flags & _lib.STACK_LINEAR)
        dx = torch.empty_like(x)
        debar = torch.empty_like(ebar)
        dA = torch.empty_like(A)
        dWnX, dWe = torch.empty_like(WnX), torch.empty_like(We)
        dWinner = None if Winner is None else torch.empty_like(Winner)
        dWout = torch.empty_like(Wout) if linear else None
        dbout = torch.empty(D, device=dev) if linear else None
        ws, wsb = _ws_for(batch, heads, dev)
        _lib.call("gcgcn_graphconv_stack_bwd", batch.ref, heads, layers, in_dim, slab, flags, _p(x), _p(ebar),
                  _p(A), _p(WnX), _p(We), _p(Winner), _p(Wout), _p(keep), _p(Z), _p(G), _p(F), _p(dy),
                  _p(dx), _p(debar), _p(dA), _p(dWnX), _p(dWe), _p(dWinner), _p(dWout), _p(dbout),
                  ws, wsb, _stream(dev))
        return (dx, debar, dA, dWnX, dWe, dWinner, dWout, dbout, None, None, None, None, None, None, None)


# ------------------------------------------------------------------------------- fused blocks
def block_supported(batch: RaggedBatch, heads: int, layers: int, mha: bool) -> bool:
    """True when the (document, head) block kernels cover this batch (gcgcn_block_supported)."""
    return bool(_lib.load().gcgcn_block_supported(batch.ref, heads, layers, int(mha)))


def _drop_ref(drop):
    """(seed, p_att, p_gcn) or None -> argument for a `const gcgcn_dropout*` parameter."""
    if drop is None:
        return None
    import ctypes
    seed, p_att, p_gcn = drop
    return ctypes.byref(_lib.Dropout(int(seed) & 0xFFFFFFFFFFFFFFFF, float(p_att), float(p_gcn)))


def dropout_mask(seed: int, stream_id: int, p: float, count: int, device) -> torch.Tensor:
    """The keep-scale factors (0 or 1/(1-p)) the block kernels regenerate for one dropout stream."""
    out = torch.empty(int(count), device=device, dtype=torch.float32)
    _lib.call("gcgcn_dropout_mask", int(seed) & 0xFFFFFFFFFFFFFFFF, int(stream_id), float(p), int(count), _p(out),
              _stream(out.device))
    return out


class CaggcFn(Function):
    """CAGGC block without dropout masks: GATAttention + GraphConvolution on one pass over e
    (G:330-333) through gcgcn_caggc_fwd / gcgcn_caggc_bwd.  Returns (y, A) -- A is the GAT map."""

    @staticmethod
    def forward(ctx, x, e, u, v, c, WnX, We, Winner, Wout, bout, batch: RaggedBatch, layers: int, drop=None):
        x = _cuda(x, "node_feat")
        e, dt = _edge(e, "edge_feat")
        u, v, c = _cuda(u, "u"), _cuda(v, "v"), _cuda(c, "c")
        WnX, We, Wout, bout = _cuda(WnX, "WnX"), _cuda(We, "We"), _cuda(Wout, "Wout"), _cuda(bout, "bout")
        Winner = None if Winner is None else _cuda(Winner, "Winner")
        dev = x.device
        nb = _lib.load().gcgcn_block_saved_bytes(batch.total_nodes, batch.total_pairs, 1)
        saved = torch.empty(int(nb), dtype=torch.uint8, device=dev)
        y = torch.empty(batch.total_nodes, D, device=dev)
        ws, wsb = _ws_for(batch, 1, dev)
        _lib.call("gcgcn_caggc_fwd", batch.ref, layers, _p(x), _p(e), dt, _p(u), _p(v), _p(c), _p(WnX), _p(We),
                  _p(Winner), _p(Wout), _p(bout), _p(y), _p(saved), _drop_ref(drop), ws, wsb, _stream(dev))
        ctx.save_for_backward(x, e, u, v, WnX, We, Winner, Wout, saved)
        ctx.cfg = (batch, layers, dt, drop)
        att = saved[: batch.total_pairs * 4].view(torch.float32)      # P is the first slab of the arena
        ctx.mark_non_differentiable(att)
        return y, att

    @staticmethod
    def backward(ctx, dy, _datt):
        x, e, u, v, WnX, We, Winner, Wout, saved = ctx.saved_tensors
        batch, layers, dt, drop = ctx.cfg
        dev = x.device
        dy = _cuda(dy, "dy")
        dx, de = torch.empty_like(x), torch.empty_like(e)
        duvc = torch.empty(2 * D + 1, device=dev)          # [du | dv | dc] contiguous: GatCollapseFn consumes it as is
        du, dv, dc = duvc[:D], duvc[D:2 * D], duvc[2 * D:]
        dWnX, dWe, dWout = torch.empty_like(WnX), torch.empty_like(We), torch.empty_like(Wout)
        dWinner = None if Winner is None else torch.empty_like(Winner)
        dbout = torch.empty(D, device=dev)
        ws, wsb = _ws_for(batch, 1, dev)
        _lib.call("gcgcn_caggc_bwd", batch.ref, layers, _p(x), _p(e), dt, _p(u), _p(v), _p(WnX), _p(We), _p(Winner),
                  _p(Wout), _p(dy), _p(saved), _p(dx), _p(de), _p(du), _p(dv), _p(dc), _p(dWnX), _p(dWe),
                  _p(dWinner), _p(dWout), _p(dbout), _drop_ref(drop), ws, wsb, _stream(dev))
        return dx, de, du, dv, dc.reshape(()), dWnX, dWe, dWinner, dWout, dbout, None, None, None


class MhaStackFn(Function):
    """MultiHeadAttention + MultiGraphConvolution without dropout masks (G:336-337) with the attention
    softmax, its backward and dq inside the block kernels.  Returns (y, P [H, total_pairs])."""

    @staticmethod
    def forward(ctx, x, ebar, Wq, bq, WnX, We, Winner, Wout, bout, batch: RaggedBatch, heads: int, layers: int,
                drop=None):
        x, ebar = _cuda(x, "node_feat"), _cuda(ebar, "ebar")
        Wq, bq = _cuda(Wq, "Wq"), _cuda(bq, "bq")
        WnX, We, Wout, bout = _cuda(WnX, "WnX"), _cuda(We, "We"), _cuda(Wout, "Wout"), _cuda(bout, "bout")
        Winner = None if Winner is None else _cuda(Winner, "Winner")
        dev, M, HD = x.device, batch.total_nodes, heads * D
        q = torch.empty(M, D, device=dev)
        P = torch.empty(heads, batch.total_pairs, device=dev)
        Z, G, F = (torch.empty(M, HD, device=dev) for _ in range(3))
        y = torch.empty(M, D, device=dev)
        ws, wsb = _ws_for(batch, heads, dev)
        _lib.call("gcgcn_mha_stack_fwd", batch.ref, heads, layers, _p(x), _p(ebar), _p(Wq), _p(bq), _p(WnX), _p(We),
                  _p(Winner), _p(Wout), _p(bout), _p(q), _p(P), _p(Z), _p(G), _p(F), _p(y), _drop_ref(drop), ws, wsb,
                  _stream(dev))
        ctx.save_for_backward(x, ebar, Wq, WnX, We, Winner, Wout, q, P, Z, G, F)
        ctx.cfg = (batch, heads, layers, drop)
        ctx.mark_non_differentiable(P)
        return y, P

    @staticmethod
    def backward(ctx, dy, _dP):
        x, ebar, Wq, WnX, We, Winner, Wout, q, P, Z, G, F = ctx.saved_tensors
        batch, heads, layers, drop = ctx.cfg
        dev = x.device
        dy = _cuda(dy, "dy")
        dx, debar = torch.empty_like(x), torch.empty_like(ebar)
        dWq, dbq = torch.empty_like(Wq), torch.empty(D, device=dev)
        dWnX, dWe, dWout = torch.empty_like(WnX), torch.empty_like(We), torch.empty_like(Wout)
        dWinner = None if Winner is None else torch.empty_like(Winner)
        dbout = torch.empty(D, device=dev)
        ws, wsb = _ws_for(batch, heads, dev)
        _lib.call("gcgcn_mha_stack_bwd", batch.ref, heads, layers, _p(x), _p(ebar), _p(Wq), _p(WnX), _p(We),
                  _p(Winner), _p(Wout), _p(q), _p(P), _p(Z), _p(G), _p(F), _p(dy), _p(dx), _p(debar), _p(dWq),
                  _p(dbq), _p(dWnX), _p(dWe), _p(dWinner), _p(dWout), _p(dbout), _drop_ref(drop), ws, wsb, _stream(dev))
        return dx, debar, dWq, dbq, dWnX, dWe, dWinner, dWout, dbout, None, None, None, None


# ------------------------------------------------------------------------------- parameter packing
_PTR_TABLES: dict = {}


def _ptr_table(tensors, device) -> torch.Tensor:
    key = tuple(t.data_ptr() for t in tensors)
    tab = _PTR_TABLES.get(key)
    if tab is None:
        if len(_PTR_TABLES) > 64:
            _PTR_TABLES.clear()
        tab = _PTR_TABLES[key] = torch.tensor(key, dtype=torch.int64, device=device)
    return tab


class PackStackFn(Function):
    """(weights_node_k, weights_edge_k for k = h*L + l) -> WnX, We, Winner in one launch; the backward
    scatters the packed gradients into per-parameter views of two flat buffers in one launch."""

    @staticmethod
    def forward(ctx, heads: int, layers: int, *params):
        wn = [_cuda(p, "weights_node") for p in params[0::2]]
        we = [_cuda(p, "weights_edge") for p in params[1::2]]
        dev = wn[0].device
        slab = layers * we[0].shape[1]
        g = slab // layers
        WnX = torch.empty(D, heads * slab, device=dev)
        We = torch.empty(D, heads * slab, device=dev)
        Winner = torch.empty(heads, layers, slab, g, device=dev) if layers > 1 else None
        _lib.call("gcgcn_pack_stack_weights", _p(_ptr_table(wn, dev)), _p(_ptr_table(we, dev)), heads, layers, slab,
                  _p(WnX), _p(We), _p(Winner), _stream(dev))
        ctx.cfg = (heads, layers, slab, [tuple(t.shape) for t in wn], [tuple(t.shape) for t in we])
        ctx._keepalive = (wn, we)
        if Winner is None:
            ctx.mark_non_differentiable()
            return WnX, We
        return WnX, We, Winner

    @staticmethod
    def backward(ctx, dWnX, dWe, dWinner=None):
        heads, layers, slab, wn_shapes, we_shapes = ctx.cfg
        dev = dWnX.device
        dWnX, dWe = _cuda(dWnX, "dWnX"), _cuda(dWe, "dWe")
        if layers > 1:
            dWinner = torch.zeros(heads, layers, slab, slab // layers, device=dev) if dWinner is None \
                else _cuda(dWinner, "dWinner")
        dwn_flat = torch.empty(sum(a * b for a, b in wn_shapes), device=dev)
        dwe_flat = torch.empty(sum(a * b for a, b in we_shapes), device=dev)
        _lib.call("gcgcn_unpack_stack_grads", _p(dWnX), _p(dWe), _p(dWinner), heads, layers, slab, _p(dwn_flat),
                  _p(dwe_flat), _stream(dev))
        gn = [v.view(s) for v, s in zip(torch.split(dwn_flat, [a * b for a, b in wn_shapes]), wn_shapes)]
        ge = [v.view(s) for v, s in zip(torch.split(dwe_flat, [a * b for a, b in we_shapes]), we_shapes)]
        out = [None, None]
        for a, b in zip(gn, ge):
            out += [a, b]
        return tuple(out)


class GatCollapseFn(Function):
    """(linear_node_h, linear_node_t, linear_edge_r, wt) -> u [128], v [128], c []: the exact collapse of G:156-162
    (energy_ij = u.x_j + v.e_ij + c) in one launch; the backward fills the eight parameter gradients in one launch."""

    @staticmethod
    def forward(ctx, Wh, bh, Wt, bt, Wr, br, w, b):
        ts = [_cuda(t, "GAT parameter") for t in (Wh, bh, Wt, bt, Wr, br, w, b)]
        hid = ts[0].shape[0]
        if ts[0].shape[1] != D or ts[6].numel() != 3 * hid:
            raise _lib.GcgcnError(f"GATAttention collapse: weights must be [hidden, {D}] and wt [1, 3*hidden]")
        out = torch.empty(2 * D + 1, device=ts[0].device)
        _lib.call("gcgcn_gat_collapse_fwd", *[_p(t) for t in ts], hid, _p(out), _stream(out.device))
        ctx.save_for_backward(*ts[:7])
        return out[:D], out[D:2 * D], out[2 * D]

    @staticmethod
    def backward(ctx, du, dv, dc):
        Wh, bh, Wt, bt, Wr, br, w = ctx.saved_tensors
        dev, hid = Wh.device, Wh.shape[0]
        if (du is not None and dv is not None and dc is not None and du.is_contiguous() and dv.is_contiguous()
                and dv.data_ptr() == du.data_ptr() + 4 * D and dc.data_ptr() == du.data_ptr() + 8 * D):
            dout = du                                       # the consumer wrote [du | dv | dc] into one buffer
        else:
            dout = torch.zeros(2 * D + 1, device=dev)
            if du is not None:
                dout[:D] = du
            if dv is not None:
                dout[D:2 * D] = dv
            if dc is not None:
                dout[2 * D] = dc
        g = [torch.empty_like(t) for t in (Wh, bh, Wt, bt, Wr, br, w)] + [torch.empty(1, device=dev)]
        _lib.call("gcgcn_gat_collapse_bwd", _p(Wh), _p(bh), _p(Wt), _p(bt), _p(Wr), _p(br), _p(w), _p(dout), hid,
                  *[_p(t) for t in g], _stream(dev))
        return tuple(g)


class PackRowsFn(Function):
    """Concatenate equally shaped parameters along dim 0 through a device pointer table (one launch); the backward
    hands out views of the incoming gradient."""

    @staticmethod
    def forward(ctx, *params):
        ps = [_cuda(p, "parameter") for p in params]
        dev = ps[0].device
        elems = ps[0].numel()
        out = torch.empty((len(ps) * ps[0].shape[0],) + tuple(ps[0].shape[1:]), device=dev)
        _lib.call("gcgcn_pack_rows", _p(_ptr_table(ps, dev)), len(ps), elems, _p(out), _stream(dev))
        ctx.rows, ctx.count = ps[0].shape[0], len(ps)
        ctx._keepalive = ps
        return out

    @staticmethod
    def backward(ctx, dout):
        return tuple(dout[i * ctx.rows:(i + 1) * ctx.rows] for i in range(ctx.count))


# ------------------------------------------------------------------------------- a8 pair gathers
class PairGatherFn(Function):
    """P_h[p] = cat(feat[h_idx[p]], dis[dis_h[p]]), P_t likewise (G:306-307, 351-352)."""

    @staticmethod
    def forward(ctx, feat, dis, tables: PairTables, batch: RaggedBatch):
        feat = _cuda(feat, "node_feats")
        fw = feat.shape[1]
        dw = 0
        if dis is not None:
            dis = _cuda(dis, "dis_embed")
            dw = dis.shape[1]
            if not tables.has_dis:
                raise _lib.GcgcnError("PairTables were built without node_relative_pos")
            tables.check_dis_rows(dis.shape[0])
        dev = feat.device
        out_h = torch.empty(batch.total_pairs, fw + dw, device=dev)
        out_t = torch.empty(batch.total_pairs, fw + dw, device=dev)
        _lib.call("gcgcn_pair_gather_fwd", batch.ref, _p(feat), fw, _p(dis), dw, _p(tables.h_idx),
                  _p(tables.t_idx), _p(tables.dis_h) if dw else None, _p(tables.dis_t) if dw else None,
                  _p(out_h), _p(out_t), _stream(dev))
        ctx.cfg = (tables, batch, fw, dw, 0 if dis is None else dis.shape[0], feat.shape[0])
        return out_h, out_t

    @staticmethod
    def backward(ctx, dh, dt):
        tables, batch, fw, dw, rows, nrows = ctx.cfg
        dev = dh.device if dh is not None else dt.device
        shape = (batch.total_pairs, fw + dw)
        dh = torch.zeros(shape, device=dev) if dh is None else _cuda(dh, "dout_h")
        dt = torch.zeros(shape, device=dev) if dt is None else _cuda(dt, "dout_t")
        dfeat = torch.empty(nrows, fw, device=dev)
        ddis = torch.empty(rows, dw, device=dev) if dw else None
        ws, wsb = _ws_for(batch, 1, dev)
        _lib.call("gcgcn_pair_gather_bwd", batch.ref, _p(dh), _p(dt), fw, dw, rows,
                  _p(tables.dis_h) if dw else None, _p(tables.dis_t) if dw else None, _p(dfeat), _p(ddis),
                  ws, wsb, _stream(dev))
        return dfeat, ddis, None, None


class PairDenseFn(Function):
    """entity_feature_h/t = tanh(U[h_idx] + Vd[dis_h]), tanh(U[t_idx] + Vd[dis_t])  (G:351-355 with dense_layer split by
    input columns; U = F W_F^T, Vd = dis_embed W_d^T + b are node-level and come from the caller)."""

    @staticmethod
    def forward(ctx, U, Vd, tables: PairTables, batch: RaggedBatch):
        U, Vd = _cuda(U, "U"), _cuda(Vd, "Vd")
        if U.shape != (batch.total_nodes, D) or Vd.shape[1] != D:
            raise _lib.GcgcnError(f"pair_dense: U must be [{batch.total_nodes}, {D}] and Vd [rows, {D}]")
        if not tables.has_dis:
            raise _lib.GcgcnError("PairTables were built without node_relative_pos")
        tables.check_dis_rows(Vd.shape[0])
        dev = U.device
        out_h = torch.empty(batch.total_pairs, D, device=dev)
        out_t = torch.empty(batch.total_pairs, D, device=dev)
        _lib.call("gcgcn_pair_dense_fwd", batch.ref, _p(U), _p(Vd), _p(tables.h_idx), _p(tables.t_idx),
                  _p(tables.dis_h), _p(tables.dis_t), _p(out_h), _p(out_t), _stream(dev))
        ctx.save_for_backward(out_h, out_t)
        ctx.cfg = (tables, batch, Vd.shape[0])
        return out_h, out_t

    @staticmethod
    def backward(ctx, dh, dt):
        out_h, out_t = ctx.saved_tensors
        tables, batch, rows = ctx.cfg
        dev = out_h.device
        dh = torch.zeros_like(out_h) if dh is None else _cuda(dh, "dout_h")
        dt = torch.zeros_like(out_t) if dt is None else _cuda(dt, "dout_t")
        dU = torch.empty(batch.total_nodes, D, device=dev)
        dVd = torch.empty(rows, D, device=dev)
        dpre = torch.empty(2 * batch.total_pairs, D, device=dev)
        wsb = int(_lib.load().gcgcn_pair_dense_ws_bytes(rows))
        ws = workspace(dev, wsb)
        _lib.call("gcgcn_pair_dense_bwd", batch.ref, _p(dh), _p(dt), _p(out_h), _p(out_t), rows, _p(tables.dis_h),
                  _p(tables.dis_t), _p(dU), _p(dVd), _p(dpre), ws.data_ptr(), ws.numel(), _stream(dev))
        return dU, dVd, None, None


def gemm(a: torch.Tensor, b: torch.Tensor, trans_a=False, trans_b=False, bias=None,
         out: Optional[torch.Tensor] = None, alpha=1.0, beta=0.0) -> torch.Tensor:
    """Thin test hook over gcgcn_gemm (row-major fp32).  ``out`` may be a row-strided view (e.g. a column slice of a
    wider buffer): it is written in place with its own row stride; its elements must be contiguous within a row."""
    a, b = _cuda(a, "A"), _cuda(b, "B")
    M = a.shape[1] if trans_a else a.shape[0]
    K = a.shape[0] if trans_a else a.shape[1]
    N = b.shape[0] if trans_b else b.shape[1]
    if out is None:      # beta == 0 overwrites every element: no fill needed
        out = torch.empty(M, N, device=a.device) if (beta == 0.0 and K > 0) else torch.zeros(M, N, device=a.device)
    if out.stride(1) != 1:
        raise _lib.GcgcnError(f"gemm: out needs unit column stride (strides {tuple(out.stride())})")
    ws = workspace(a.device, (24 << 20) + 4096)     # split-K partials / pre-split weight blobs
    _lib.call("gcgcn_gemm", int(trans_a), int(trans_b), M, N, K, float(alpha), _p(a), a.shape[1], _p(b),
              b.shape[1], float(beta), _p(out), out.stride(0), _p(bias), ws.data_ptr(), ws.numel(),
              _stream(a.device))
    return out


# ------------------------------------------------------------------------------- linear layers on gcgcn_gemm
class LinearFn(Function):
    """y = x W^T + b on gcgcn_gemm (3xTF32 tcgen05 tiles, or the CUDA-core kernel for tiny / unaligned shapes);
    backward = two more products and a column sum.  ``b`` may be None."""

    @staticmethod
    def forward(ctx, x, W, b):
        x, W = _cuda(x, "x"), _cuda(W, "weight")
        b = None if b is None else _cuda(b, "bias")
        ctx.save_for_backward(x, W)
        ctx.has_bias = b is not None
        if x.shape[0] == 0:
            return x.new_zeros(0, W.shape[0])
        return gemm(x, W, trans_b=True, bias=b)

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        dy = _cuda(dy, "dy")
        M = x.shape[0]
        dev = x.device
        if M == 0:
            return x.new_zeros(x.shape), torch.zeros_like(W), (torch.zeros(W.shape[0], device=dev) if ctx.has_bias else None)
        dx = gemm(dy, W) if ctx.needs_input_grad[0] else None
        dW = gemm(dy, x, trans_a=True) if ctx.needs_input_grad[1] else None
        db = None
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(W.shape[0], device=dev)
            ws = workspace(dev, 8 << 20)
            _lib.call("gcgcn_colsum", _p(dy), M, W.shape[0], dy.shape[1], _p(db), ws.data_ptr(), ws.numel(), _stream(dev))
        return dx, dW, db


def linear(x, layer):
    return LinearFn.apply(x, layer.weight, layer.bias)


