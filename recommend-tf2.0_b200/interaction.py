"""Host side of the feature-interaction kernels (K3 FM cross, K4 DLRM pairwise dot).

`dot_interact` / `embed_dot` implement the interaction the reference's DLRM leaves out
(src/ctr/dlrm/model.py:48 concatenates; the paper it cites at :7 defines the op, SURVEY §8 a5).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib as L
from .embedding import EmbeddingTables, _ptr_array


def dot_out_cols(F1: int, D: int, pad_to: int = 1) -> int:
    n = D + F1 * (F1 - 1) // 2
    return (n + pad_to - 1) // pad_to * pad_to


class _DotFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, pad_to):
        L.require_cuda(x, "dot_interact(x)")
        x = x.contiguous()
        B, F1, D = x.shape
        cols = dot_out_cols(F1, D, pad_to)
        out = torch.empty((B, cols), dtype=torch.float32, device=x.device)
        L.check(L.lib().rtf_dot_interact_fwd(x.data_ptr(), B, F1, D, out.data_ptr(), cols, cols,
                                             L.current_stream_ptr()), "rtf_dot_interact_fwd")
        ctx.save_for_backward(x)
        return out

    @staticmethod
    def backward(ctx, gout):
        (x,) = ctx.saved_tensors
        gout = gout.contiguous()
        B, F1, D = x.shape
        gx = torch.empty_like(x)
        L.check(L.lib().rtf_dot_interact_bwd(x.data_ptr(), gout.data_ptr(), gout.stride(0), B, F1,
                                             D, gx.data_ptr(), L.current_stream_ptr()),
                "rtf_dot_interact_bwd")
        return gx, None


def dot_interact(x: torch.Tensor, pad_to: int = 1) -> torch.Tensor:
    """(B, F1, D) -> (B, D + F1(F1-1)/2 [rounded up to pad_to, zero filled])."""
    return _DotFn.apply(x, pad_to)


class _EmbedDotFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tset: EmbeddingTables, ids, field_table, pad_to, prepare, dense, *weights):
        L.require_cuda(ids, "embed_dot(ids)")
        dense = dense.contiguous()
        B, F = ids.shape
        D = dense.shape[1]
        tables = [weights[t] for t in field_table]
        for t in tables:
            if t.shape[1] != D:
                raise ValueError("embed_dot: every table and the dense row must have the same dim")
        cols = dot_out_cols(F + 1, D, pad_to)
        out = torch.empty((B, cols), dtype=torch.float32, device=ids.device)
        rows = L.host_array(C.c_int64, [int(t.shape[0]) for t in tables])
        rc = L.lib().rtf_embed_dot_fwd(_ptr_array(tables), rows, F, D, ids.data_ptr(),
                                       int(ids.dtype == torch.int64), B, ids.stride(0),
                                       ids.stride(1), dense.data_ptr(), dense.stride(0),
                                       out.data_ptr(), cols, cols, tset.err.data_ptr(),
                                       L.current_stream_ptr())
        L.check(rc, "rtf_embed_dot_fwd")
        ctx.tset, ctx.ids, ctx.field_table = tset, ids, field_table
        # the id-only half of K2 (keys, sort, segments) starts now on a side stream and hides
        # behind the top MLP; the backward then only runs the gradient-dependent half
        ctx.prepared = tset.prepare_backward(ids, field_table) if prepare else None
        ctx.save_for_backward(dense)
        return out

    @staticmethod
    def backward(ctx, gout):
        (dense,) = ctx.saved_tensors
        tset, ids, field_table = ctx.tset, ctx.ids, ctx.field_table
        gout = gout.contiguous()
        B, F = ids.shape
        D = dense.shape[1]
        wl = tset.wlist()
        tables = [wl[t] for t in field_table]
        rows = L.host_array(C.c_int64, [int(t.shape[0]) for t in tables])
        gdense = torch.empty_like(dense)
        gemb = torch.empty((B, F * D), dtype=torch.float32, device=ids.device)
        rc = L.lib().rtf_embed_dot_bwd(_ptr_array(tables), rows, F, D, ids.data_ptr(),
                                       int(ids.dtype == torch.int64), B, ids.stride(0),
                                       ids.stride(1), dense.data_ptr(), dense.stride(0),
                                       gout.data_ptr(), gout.stride(0), gdense.data_ptr(),
                                       gdense.stride(0), gemb.data_ptr(), gemb.stride(0),
                                       L.current_stream_ptr())
        L.check(rc, "rtf_embed_dot_bwd")
        if ctx.prepared is not None:
            # with a trainer that opts in (async_update), the gradient half of K2 goes to the side
            # stream and overlaps the bottom MLP's backward GEMMs; wait_pending() orders the
            # tables again before anything else touches them
            if getattr(tset, "async_update", False):   # a trainer that calls wait_pending()
                tset.apply_prepared_async(ctx.prepared, gemb)
            else:
                tset.apply_prepared(ctx.prepared, gemb)
            return (None, None, None, None, None, gdense) + (None,) * len(wl)
        wgrads = tset.grads_from_lookup_grad(ids, field_table, gemb, "BF", None)
        return (None, None, None, None, None, gdense) + wgrads


def embed_dot(tset: EmbeddingTables, ids: torch.Tensor, dense: torch.Tensor,
              field_table: Optional[Sequence[int]] = None, pad_to: int = 1) -> torch.Tensor:
    """Fused K1+K4: out = dot_interact(stack([dense, lookup(ids)...])) without materialising the
    gathered rows in HBM.  ids (B, F) int32/int64, dense (B, D)."""
    if ids.dtype not in (torch.int32, torch.int64):
        raise TypeError("ids must be int32 or int64")
    wl = tset.wlist()
    if field_table is None:
        field_table = tuple(range(len(wl)))
    tset.wait_pending()
    # K2's id-only half is prepared only when a backward can follow.  ctx.needs_input_grad cannot
    # decide this: it stays True for the table Parameters inside torch.no_grad(), and
    # torch.is_grad_enabled() is always False inside Function.forward.  Under grad mode this is
    # exactly `any(ctx.needs_input_grad)` (ids are integers, never differentiable).
    prepare = (tset.optimizer is not None and torch.is_grad_enabled()
               and (dense.requires_grad or any(w.requires_grad for w in wl)))
    return _EmbedDotFn.apply(tset, ids, tuple(field_table), pad_to, prepare, dense, *wl)
