"""Autograd wrappers over the C ABI (include/nbody_b200.h).

One `torch.autograd.Function` per model: the whole EGNO / SEGNO forward is one C call that enqueues the
kernel sequence on the current CUDA stream, and the whole backward is another.  PyTorch only owns the
memory (inputs, outputs, the saved-for-backward buffer, scratch) and the stream.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence

import torch

from . import _cabi
from ._lib import check, load_library


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream_ptr(device: torch.device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda_f32(name: str, t: torch.Tensor, shape: Sequence[int]) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise ValueError(f"{name} must live on a CUDA device (this implementation has no CPU path); got {t.device}")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {t.dtype}")
    if tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")
    return t.contiguous()


class _ParamPack:
    """Keeps a module's parameters as views of ONE flat fp32 buffer (the layout of the C ABI, which is
    the order of named_parameters()).  The views survive optimizer steps and load_state_dict (both
    in-place); `.to()` / `.cuda()` replace parameter storage, which is detected and re-flattened."""

    def __init__(self, module: torch.nn.Module, skip_prefix: Optional[str] = None):
        self.module = module
        self.skip_prefix = skip_prefix      # parameters outside the C layout (kept as ordinary torch parameters)
        self.flat: Optional[torch.Tensor] = None
        self.offsets: List[int] = []

    def params(self) -> List[torch.nn.Parameter]:
        return [p for k, p in self.module.named_parameters() if not (self.skip_prefix and k.startswith(self.skip_prefix))]

    def _views_ok(self, ps) -> bool:
        f = self.flat
        if f is None or len(ps) != len(self.offsets):
            return False
        base = f.data_ptr()
        for p, off in zip(ps, self.offsets):
            if p.data_ptr() != base + 4 * off or p.device != f.device or p.dtype != torch.float32:
                return False
        return True

    def flat_params(self, expected: int, device: torch.device):
        ps = self.params()
        if not self._views_ok(ps) or self.flat.device != device:
            for p in ps:
                if p.dtype != torch.float32:
                    raise ValueError("parameters must be float32")
                if p.device != device:
                    raise ValueError(f"parameters live on {p.device} but inputs on {device}; call model.to(device)")
            with torch.no_grad():
                flat = torch.cat([p.detach().reshape(-1) for p in ps]).contiguous()
                offs, o = [], 0
                for p in ps:
                    offs.append(o)
                    p.data = flat[o:o + p.numel()].view(p.shape)
                    o += p.numel()
            self.flat, self.offsets = flat, offs
        if self.flat.numel() != expected:
            raise RuntimeError(f"parameter count {self.flat.numel()} != C layout {expected}")
        return self.flat, ps


def _maybe_allreduce(grad_flat: torch.Tensor, dp) -> None:
    """Data parallel: ONE all-reduce of the flat gradient bucket (NCCL over NVLink).  `dp` = (group, average): with
    average the bucket is divided by the world size here (any optimizer sees the mean gradient); without, the SUM is left
    in place and the 1 / world factor rides inside the fused optimizer kernel (FlatAdam(grad_scale=1 / world))."""
    if dp is None or dp_bucket(dp) is not None:   # peer-memory mode: FlatAdam reduces inside its update kernel
        return
    import torch.distributed as dist

    group, average = dp[0], dp[1]
    dist.all_reduce(grad_flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        grad_flat.div_(dist.get_world_size(group))


def dp_bucket(dp):
    """dp = (group, average[, PeerGradBucket]) -> the bucket or None"""
    return dp[2] if dp is not None and len(dp) > 2 else None


def _grad_buffer(flat: torch.Tensor, dp) -> torch.Tensor:
    """Where the backward writes the flat parameter gradient: a fresh buffer, or — peer-memory data parallel — the model's
    symmetric-memory bucket (its address is what the other ranks read)."""
    b = dp_bucket(dp)
    if b is None:
        return torch.empty_like(flat)
    if b.numel != flat.numel() or b.buf.device != flat.device:
        raise RuntimeError("peer gradient bucket does not match the model's flat parameter buffer")
    return b.buf


class _AllReduceGrad(torch.autograd.Function):
    """Identity whose backward all-reduces the incoming gradient over the data-parallel group: for the few parameters that
    are multiplied on the torch side (multi-input SEGNO: embedding and temporal attention, SEGNO/models/model.py:65-90,
    127-139) and therefore do not pass through the flat gradient bucket of the C call."""

    @staticmethod
    def forward(ctx, dp, t):
        ctx.dp = dp
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        import torch.distributed as dist

        group, average = ctx.dp[0], ctx.dp[1]
        g = g.contiguous().clone()
        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
        if average:
            g.div_(dist.get_world_size(group))
        return None, g


def dp_param(t: torch.Tensor, dp):
    """`t` itself without data parallelism, else a view whose gradient is reduced over the group before it reaches `t`."""
    return t if dp is None else _AllReduceGrad.apply(dp, t)


class EgnoFunction(torch.autograd.Function):
    """x, v, h = EGNO.forward(...)   (reference: EGNO/model/egno.py:37-111)."""

    @staticmethod
    def forward(ctx, cfg_tuple, dp_group, flat, x, nodes, edge_fea, v, loc_mean, tsteps, tsteps_in, *params):
        lib = load_library()
        cfg = _cabi.NbEgnoConfig(*cfg_tuple)
        dev = x.device
        Nn = cfg.T * cfg.B * cfg.N
        need_grad = any(ctx.needs_input_grad)   # False under torch.no_grad(): nothing is kept for backward
        x_out = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        v_out = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        h_out = torch.empty((Nn, 64), device=dev, dtype=torch.float32)
        saved = torch.empty(lib.nb_egno_saved_floats(ctypes.byref(cfg)), device=dev, dtype=torch.float32) if need_grad else None
        ws = torch.empty(lib.nb_egno_workspace_floats(ctypes.byref(cfg), 2 if need_grad else 0), device=dev, dtype=torch.float32)
        # int64 frame indices, or fp32 times (any real value) through the _ft entry points
        fwd = "nb_egno_forward_ft" if tsteps.is_floating_point() else "nb_egno_forward"
        check(getattr(lib, fwd)(ctypes.byref(cfg), _ptr(flat), _ptr(x), _ptr(nodes), _ptr(edge_fea), _ptr(v),
                                _ptr(loc_mean), _ptr(tsteps), _ptr(tsteps_in), _ptr(x_out), _ptr(v_out), _ptr(h_out),
                                _ptr(saved), _ptr(ws), _stream_ptr(dev)), fwd)
        ctx.cfg_tuple = cfg_tuple
        ctx.dp_group = dp_group
        ctx.param_shapes = [p.shape for p in params]
        ctx.save_for_backward(flat, nodes, edge_fea, loc_mean, tsteps, tsteps_in, saved)
        return x_out, v_out, h_out

    @staticmethod
    def backward(ctx, gx_out, gv_out, gh_out):
        lib = load_library()
        flat, nodes, edge_fea, loc_mean, tsteps, tsteps_in, saved = ctx.saved_tensors
        if saved is None:
            raise RuntimeError("EGNO forward ran without autograd state; cannot run backward")
        cfg = _cabi.NbEgnoConfig(*ctx.cfg_tuple)
        dev = flat.device
        n0 = cfg.B * cfg.N
        gx_out = None if gx_out is None else gx_out.contiguous()
        gv_out = None if gv_out is None else gv_out.contiguous()
        gh_out = None if gh_out is None else gh_out.contiguous()
        grad_flat = _grad_buffer(flat, ctx.dp_group)
        in_shape = (cfg.num_inputs, n0, 3) if cfg.num_inputs > 1 else (n0, 3)
        gx_in = torch.empty(in_shape, device=dev, dtype=torch.float32)
        gv_in = torch.empty(in_shape, device=dev, dtype=torch.float32)
        ws = torch.empty(lib.nb_egno_workspace_floats(ctypes.byref(cfg), 1), device=dev, dtype=torch.float32)
        # per-shard input gradients: under data parallelism nothing beyond the parameter bucket is reduced
        want = ctx.needs_input_grad
        g_nodes = torch.empty_like(nodes) if want[4] else None
        g_ef = torch.empty_like(edge_fea) if want[5] else None
        g_lm = torch.empty_like(loc_mean) if want[7] else None
        iws = None
        if want[4] or want[5]:
            iws = torch.empty(lib.nb_egno_input_grad_workspace_floats(ctypes.byref(cfg)), device=dev, dtype=torch.float32)
        args = [ctypes.byref(cfg), _ptr(flat), _ptr(nodes), _ptr(edge_fea), _ptr(loc_mean), _ptr(tsteps), _ptr(tsteps_in),
                _ptr(saved), _ptr(gx_out), _ptr(gv_out), _ptr(gh_out), _ptr(grad_flat), _ptr(gx_in), _ptr(gv_in),
                _ptr(g_nodes), _ptr(g_ef), _ptr(g_lm)]
        g_t = g_t_in = None
        if tsteps.is_floating_point():   # fp32 times: the _ft entry point, which also returns dL/dtimes when asked
            g_t = torch.empty_like(tsteps) if want[8] else None
            g_t_in = torch.empty_like(tsteps_in) if want[9] else None
            bwd, args = "nb_egno_backward_ft", args + [_ptr(g_t), _ptr(g_t_in)]
        else:
            bwd = "nb_egno_backward_ex"
        check(getattr(lib, bwd)(*args, _ptr(ws), _ptr(iws), _stream_ptr(dev)), bwd)
        _maybe_allreduce(grad_flat, ctx.dp_group)
        grads, o = [], 0
        for shp in ctx.param_shapes:
            n = shp.numel()
            grads.append(grad_flat[o:o + n].view(shp))
            o += n
        return (None, None, None, gx_in, g_nodes, g_ef, gv_in, g_lm, g_t, g_t_in, *grads)


class SegnoFunction(torch.autograd.Function):
    """x, h, v = SEGNO.forward_step(embedding(his), ...)   (reference: SEGNO/models/model.py:73,95-102)."""

    @staticmethod
    def forward(ctx, cfg_tuple, dp_group, flat, his, x, v, edge_attr, *params):
        lib = load_library()
        cfg = _cabi.NbSegnoConfig(*cfg_tuple)
        dev = x.device
        Nn = cfg.B * cfg.N
        need_grad = any(ctx.needs_input_grad)   # False under torch.no_grad(): nothing is kept for backward
        x_out = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        v_out = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        h_out = torch.empty((Nn, 64), device=dev, dtype=torch.float32)
        saved = torch.empty(lib.nb_segno_saved_floats(ctypes.byref(cfg)), device=dev, dtype=torch.float32) if need_grad else None
        ws = torch.empty(lib.nb_segno_workspace_floats(ctypes.byref(cfg), 2 if need_grad else 0), device=dev, dtype=torch.float32)
        check(lib.nb_segno_forward(ctypes.byref(cfg), _ptr(flat), _ptr(his), _ptr(x), _ptr(v), _ptr(edge_attr),
                                   _ptr(x_out), _ptr(h_out), _ptr(v_out), _ptr(saved), _ptr(ws), _stream_ptr(dev)),
              "nb_segno_forward")
        ctx.cfg_tuple = cfg_tuple
        ctx.dp_group = dp_group
        ctx.param_shapes = [p.shape for p in params]
        ctx.save_for_backward(flat, his, edge_attr, saved)
        return x_out, h_out, v_out

    @staticmethod
    def backward(ctx, gx_out, gh_out, gv_out):
        lib = load_library()
        flat, his, edge_attr, saved = ctx.saved_tensors
        if saved is None:
            raise RuntimeError("SEGNO forward ran without autograd state; cannot run backward")
        cfg = _cabi.NbSegnoConfig(*ctx.cfg_tuple)
        dev = flat.device
        Nn = cfg.B * cfg.N
        gx_out = None if gx_out is None else gx_out.contiguous()
        gv_out = None if gv_out is None else gv_out.contiguous()
        gh_out = None if gh_out is None else gh_out.contiguous()
        grad_flat = _grad_buffer(flat, ctx.dp_group)
        gx_in = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        gv_in = torch.empty((Nn, 3), device=dev, dtype=torch.float32)
        ws = torch.empty(lib.nb_segno_workspace_floats(ctypes.byref(cfg), 1), device=dev, dtype=torch.float32)
        gh_in = torch.empty((Nn, 64), device=dev, dtype=torch.float32) if cfg.h_given else None
        want_his = ctx.needs_input_grad[3] and not cfg.h_given
        g_his = torch.empty_like(his) if want_his else None
        g_ea = torch.empty_like(edge_attr) if ctx.needs_input_grad[6] else None
        iws = None
        if g_ea is not None:
            iws = torch.empty(lib.nb_segno_input_grad_workspace_floats(ctypes.byref(cfg)), device=dev, dtype=torch.float32)
        check(lib.nb_segno_backward_ex(ctypes.byref(cfg), _ptr(flat), _ptr(his), _ptr(edge_attr), _ptr(saved),
                                       _ptr(gx_out), _ptr(gh_out), _ptr(gv_out), _ptr(grad_flat), _ptr(gx_in),
                                       _ptr(gv_in), _ptr(gh_in), _ptr(g_his), _ptr(g_ea), _ptr(ws), _ptr(iws),
                                       _stream_ptr(dev)), "nb_segno_backward_ex")
        if want_his:
            gh_in = g_his
        _maybe_allreduce(grad_flat, ctx.dp_group)
        grads, o = [], 0
        for shp in ctx.param_shapes:
            n = shp.numel()
            grads.append(grad_flat[o:o + n].view(shp))
            o += n
        # coord_mlp_vel (the last four tensors) never enters the computation: its gradients are None in the reference
        # (gcl.py:64-67 builds it, forward never calls it), so optimizers leave it untouched
        grads[-4:] = [None] * 4
        if cfg.h_given:   # a segment of the multi-input forward: `his` is the hidden state, the embedding is outside
            grads[0] = grads[1] = None
        return (None, None, None, gh_in, gx_in, gv_in, g_ea, *grads)


class SegnoMultiFunction(torch.autograd.Function):
    """x, h, v = SEGNO.forward(his[BN, L, F], x[BN, L, 3], ..., in_steps)   (reference: SEGNO/models/model.py:65-90).

    ONE autograd node for the whole multi-input forward: the embedding of every observed frame, the integration segments
    (nb_segno_forward with h_given) and the 'sum' / attention merges between them (model.py:82-90, 105-139) are C calls
    enqueued back to back; the backward walks them in reverse, sums the segments' gradients of the shared parameters on
    the device and reduces the flat bucket once.  PyTorch only allocates.

    meta = (B, N, steps, in_node_nf, in_edge_nf, recurrent, coords_weight, mode) with mode 1 = 'sum', 2 = 'attn';
    `attn_flat` is the flat view of enc_attn_net's four tensors (None for 'sum')."""

    @staticmethod
    def forward(ctx, meta, dp_group, flat, attn_flat, his, x, v, edge_attr, n_params, *params):
        lib = load_library()
        B, N, steps, in_nf, in_ef, recurrent, cw, mode = meta
        dev = x.device
        n, L = B * N, x.shape[1]
        st = _stream_ptr(dev)
        need_grad = any(ctx.needs_input_grad)
        f32 = dict(device=dev, dtype=torch.float32)
        cfgs = [_cabi.NbSegnoConfig(B, N, int(T), in_nf, in_ef, recurrent, cw, 1) for T in steps]
        h_all = torch.empty((n, L, 64), **f32)
        check(lib.nb_segno_embed_forward(ctypes.byref(cfgs[0]), _ptr(flat), n * L, _ptr(his), _ptr(h_all), st),
              "nb_segno_embed_forward")
        cur = [torch.empty((n, 64), **f32), torch.empty((n, 3), **f32), torch.empty((n, 3), **f32)]   # h_, x_, v_
        check(lib.nb_segno_merge_forward(0, n, L, 0, _ptr(h_all), _ptr(x), _ptr(v), None, None, None, None,
                                         _ptr(cur[0]), _ptr(cur[1]), _ptr(cur[2]), None, st), "nb_segno_merge_forward")
        seg_in, seg_saved, seg_out, alphas = [], [], [], []
        out = None
        for i, cfg in enumerate(cfgs):
            xo, ho, vo = (torch.empty((n, 3), **f32), torch.empty((n, 64), **f32), torch.empty((n, 3), **f32))
            saved = torch.empty(lib.nb_segno_saved_floats(ctypes.byref(cfg)), **f32) if need_grad else None
            ws = torch.empty(lib.nb_segno_workspace_floats(ctypes.byref(cfg), 2 if need_grad else 0), **f32)
            check(lib.nb_segno_forward(ctypes.byref(cfg), _ptr(flat), _ptr(cur[0]), _ptr(cur[1]), _ptr(cur[2]), _ptr(edge_attr),
                                       _ptr(xo), _ptr(ho), _ptr(vo), _ptr(saved), _ptr(ws), st), "nb_segno_forward")
            seg_in.append(cur[0])          # the segment's input hidden state (its `his` in the backward)
            seg_saved.append(saved)
            seg_out.append((ho, xo, vo))
            out = (xo, ho, vo)
            if i < len(cfgs) - 1:
                nxt = [torch.empty((n, 64), **f32), torch.empty((n, 3), **f32), torch.empty((n, 3), **f32)]
                alpha = torch.empty((n, 2), **f32) if mode == 2 else None
                check(lib.nb_segno_merge_forward(mode, n, L, i + 1, _ptr(h_all), _ptr(x), _ptr(v), _ptr(ho), _ptr(xo), _ptr(vo),
                                                 _ptr(attn_flat), _ptr(nxt[0]), _ptr(nxt[1]), _ptr(nxt[2]), _ptr(alpha), st),
                      "nb_segno_merge_forward")
                alphas.append(alpha)
                cur = nxt
        ctx.meta, ctx.dp_group, ctx.n_params = meta, dp_group, n_params
        ctx.param_shapes = [p.shape for p in params]
        ctx.has_saved = need_grad
        if need_grad:
            ctx.save_for_backward(flat, attn_flat, his, x, v, edge_attr, h_all, *seg_in, *seg_saved,
                                  *[t for o in seg_out[:-1] for t in o], *alphas)
        return out

    @staticmethod
    def backward(ctx, gx_out, gh_out, gv_out):
        if not ctx.has_saved:
            raise RuntimeError("SEGNO forward ran without autograd state; cannot run backward")
        lib = load_library()
        B, N, steps, in_nf, in_ef, recurrent, cw, mode = ctx.meta
        S = len(steps)
        t = list(ctx.saved_tensors)
        flat, attn_flat, his, x, v, edge_attr, h_all = t[:7]
        seg_in, seg_saved = t[7:7 + S], t[7 + S:7 + 2 * S]
        rest = t[7 + 2 * S:]
        seg_out = [tuple(rest[3 * i:3 * i + 3]) for i in range(S - 1)]
        alphas = rest[3 * (S - 1):] if mode == 2 else [None] * (S - 1)
        dev = flat.device
        n, L = B * N, x.shape[1]
        st = _stream_ptr(dev)
        f32 = dict(device=dev, dtype=torch.float32)
        cfgs = [_cabi.NbSegnoConfig(B, N, int(T), in_nf, in_ef, recurrent, cw, 1) for T in steps]
        grad_flat = _grad_buffer(flat, ctx.dp_group)
        tmp = torch.empty_like(flat) if S > 1 else None
        g_h_all, g_x_all, g_v_all = torch.empty((n, L, 64), **f32), torch.empty((n, L, 3), **f32), torch.empty((n, L, 3), **f32)
        g_attn = torch.empty_like(attn_flat) if mode == 2 else None
        gh = None if gh_out is None else gh_out.contiguous()
        gx = None if gx_out is None else gx_out.contiguous()
        gv = None if gv_out is None else gv_out.contiguous()
        for i in range(S - 1, -1, -1):
            cfg = cfgs[i]
            target = grad_flat if i == S - 1 else tmp
            gx_in, gv_in, gh_in = torch.empty((n, 3), **f32), torch.empty((n, 3), **f32), torch.empty((n, 64), **f32)
            ws = torch.empty(lib.nb_segno_workspace_floats(ctypes.byref(cfg), 1), **f32)
            check(lib.nb_segno_backward(ctypes.byref(cfg), _ptr(flat), _ptr(seg_in[i]), _ptr(edge_attr), _ptr(seg_saved[i]),
                                        _ptr(gx), _ptr(gh), _ptr(gv), _ptr(target), _ptr(gx_in), _ptr(gv_in), _ptr(gh_in),
                                        _ptr(ws), st), "nb_segno_backward")
            if i != S - 1:
                check(lib.nb_accumulate(flat.numel(), _ptr(grad_flat), _ptr(tmp), st), "nb_accumulate")
            if i > 0:     # the merge that produced this segment's input: observed frame i, integrated state of segment i - 1
                ho, xo, vo = seg_out[i - 1]
                gh, gx, gv = torch.empty((n, 64), **f32), torch.empty((n, 3), **f32), torch.empty((n, 3), **f32)
                mws = torch.empty(lib.nb_segno_merge_backward_workspace_floats(n), **f32) if mode == 2 else None
                check(lib.nb_segno_merge_backward(mode, n, L, i, _ptr(h_all), _ptr(x), _ptr(v), _ptr(ho), _ptr(xo), _ptr(vo),
                                                  _ptr(attn_flat), _ptr(alphas[i - 1]), _ptr(gh_in), _ptr(gx_in), _ptr(gv_in),
                                                  _ptr(g_h_all), _ptr(g_x_all), _ptr(g_v_all), _ptr(gh), _ptr(gx), _ptr(gv),
                                                  _ptr(g_attn), 0 if i == S - 1 else 1, _ptr(mws), st), "nb_segno_merge_backward")
            else:         # frame 0 was copied into the first segment
                check(lib.nb_segno_merge_backward(0, n, L, 0, None, None, None, None, None, None, None, None, _ptr(gh_in),
                                                  _ptr(gx_in), _ptr(gv_in), _ptr(g_h_all), _ptr(g_x_all), _ptr(g_v_all),
                                                  None, None, None, None, 0, None, st), "nb_segno_merge_backward")
        ews = torch.empty(lib.nb_segno_embed_backward_workspace_floats(ctypes.byref(cfgs[0]), n * L), **f32)
        check(lib.nb_segno_embed_backward(ctypes.byref(cfgs[0]), n * L, _ptr(his), _ptr(g_h_all), _ptr(grad_flat), _ptr(ews), st),
              "nb_segno_embed_backward")
        _maybe_allreduce(grad_flat, ctx.dp_group)
        if g_attn is not None and ctx.dp_group is not None:
            _maybe_allreduce(g_attn, ctx.dp_group[:2])
        grads, o = [], 0
        for shp in ctx.param_shapes[:ctx.n_params]:
            k = shp.numel()
            grads.append(grad_flat[o:o + k].view(shp))
            o += k
        grads[-4:] = [None] * 4      # coord_mlp_vel never enters the computation (gcl.py:64-67)
        o = 0
        for shp in ctx.param_shapes[ctx.n_params:]:
            k = shp.numel()
            grads.append(g_attn[o:o + k].view(shp))
            o += k
        return (None, None, None, None, None, g_x_all, g_v_all, None, None, *grads)


class _EdgeCache:
    """Validates `edge_index` against the canonical fully connected list once per distinct tensor OBJECT: the cache holds
    weak references to the validated row / col tensors and their `_version`s, so a new tensor that happens to reuse a
    freed tensor's address is checked again.  Non-canonical graphs raise: the kernels reduce each receiver's N-1
    contiguous edge rows and have no general scatter path."""

    def __init__(self):
        self._ok = []   # [(weakref(row), weakref(col), row._version, col._version, E, B, N)]

    def _hit(self, row, col, E, B, N) -> bool:
        alive = []
        hit = False
        for ent in self._ok:
            r, c = ent[0](), ent[1]()
            if r is None or c is None:
                continue
            alive.append(ent)
            if r is row and c is col and ent[2:] == (row._version, col._version, E, B, N):
                hit = True
        self._ok = alive[-16:]
        return hit

    def validate(self, edge_index, B: int, N: int, device: torch.device) -> None:
        row, col = edge_index[0], edge_index[1]
        E = B * N * (N - 1)
        if row.dim() != 1 or row.numel() != E or col.numel() != E:
            raise ValueError(f"edge_index must hold B*N*(N-1) = {E} edges of a fully connected graph; got {row.numel()}")
        if self._hit(row, col, E, B, N):
            return
        if row.dtype != torch.int64 or col.dtype != torch.int64:
            raise ValueError("edge_index must be int64")
        if row.is_cuda:
            lib = load_library()
            flag = torch.zeros(1, device=row.device, dtype=torch.int32)
            check(lib.nb_check_canonical_edges(_ptr(row.contiguous()), _ptr(col.contiguous()), E, B, N, _ptr(flag),
                                               _stream_ptr(row.device)), "nb_check_canonical_edges")
            bad = int(flag.item())
        else:  # index tensors kept on the host by the caller (SEGNO/train_nbody.py:76-78): check them there
            e = torch.arange(E)
            b, rem = e // (N * (N - 1)), e % (N * (N - 1))
            i, jj = rem // (N - 1), rem % (N - 1)
            j = jj + (jj >= i).long()
            mism = (row != b * N + i) | (col != b * N + j)
            bad = int(mism.nonzero()[0].item()) + 1 if bool(mism.any()) else 0
        if bad:
            raise ValueError(f"edge_index is not the canonical fully connected list (first mismatch at edge {bad - 1}); "
                             "only `for i: for j != i` graphs offset by N*b are supported")
        import weakref

        try:
            self._ok.append((weakref.ref(row), weakref.ref(col), row._version, col._version, E, B, N))
        except TypeError:   # objects that cannot be weakly referenced are simply re-validated next time
            pass
