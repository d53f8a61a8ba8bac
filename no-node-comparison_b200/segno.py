"""Drop-in `SEGNO` module: constructor kwargs, forward signature, parameter names and shapes of the reference
class (SEGNO/models/model.py:6-102 with SEGNO_GCL, SEGNO/models/models/gcl.py:26-119).

Served semantics: `forward` returns the integrated state `forward_step(embedding(his), ...)` in the
reference's order (x, h, v).  The literal `forward` at reference HEAD (model.py:53-92) returns its *inputs*
and cannot be trained (SURVEY.md §0); the dead first definition (model.py:28-51), `rollout_fn` and the
training loop all assume the integrated state, which is what is computed here.
"""
from __future__ import annotations

import torch
from torch import nn

from .functional import SegnoFunction, SegnoMultiFunction, _EdgeCache, _ParamPack, _require_cuda_f32

_HIDDEN = 64


class _GCLHolder(nn.Module):
    """Parameters of SEGNO_GCL created in the reference's RNG order (gcl.py:39-67)."""

    def __init__(self, hidden: int, edges_in_d: int, act_fn: nn.Module):
        super().__init__()
        self.edge_mlp = nn.Sequential(nn.Linear(2 * hidden + 1 + edges_in_d, hidden), act_fn,
                                      nn.Linear(hidden, hidden), act_fn)
        self.node_mlp = nn.Sequential(nn.Linear(hidden + hidden, hidden), act_fn, nn.Linear(hidden, hidden))
        last = nn.Linear(hidden, 1, bias=True)                      # created BEFORE coord_mlp.0 (gcl.py:50-54)
        torch.nn.init.xavier_uniform_(last.weight, gain=0.001)
        self.coord_mlp = nn.Sequential(nn.Linear(hidden, hidden), act_fn, last)
        self.coord_mlp_vel = nn.Sequential(nn.Linear(hidden, hidden), act_fn, nn.Linear(hidden, 1))  # inert (gcl.py:64-67)
        self.n_layers = 8


class InvariantTemporalAttention(nn.Module):
    """model.py:127-139: softmax over the frames of an MLP on (|v|, h).  SEGNO.forward evaluates it (and its backward)
    in the merge kernels (csrc/nb_merge.cuh) from the flat view of these parameters; this torch forward is the
    reference's module interface, kept for callers that use the sub-module on its own."""

    def __init__(self, in_dim, hidden_dim=32):
        super().__init__()
        self.attn_mlp = nn.Sequential(nn.Linear(in_dim + 1, hidden_dim), nn.Tanh(), nn.Linear(hidden_dim, 1))

    def forward(self, vel_seq, his_seq):
        speed = vel_seq.norm(dim=-1, keepdim=True)
        return self.attn_mlp(torch.cat([speed, his_seq], dim=-1)).softmax(dim=1)


class SEGNO(nn.Module):
    def __init__(self, in_node_nf, in_edge_nf, hidden_nf, device='cpu', act_fn=nn.SiLU(), n_layers=4, coords_weight=1.0,
                 recurrent=False, norm_diff=False, tanh=False, invariant=True, norm_vel=True, varDT=False,
                 multiple_agg=None):
        super().__init__()
        if hidden_nf != _HIDDEN:
            raise ValueError(f"kernels are specialised for hidden_nf={_HIDDEN} (model_confs.yaml:23), got {hidden_nf}")
        if not isinstance(act_fn, nn.SiLU):
            raise ValueError("only the SiLU activation (reference default) is implemented")
        if tanh:
            raise ValueError("tanh=True (gcl.py:57-59) is not implemented (model_confs.yaml:27 uses False)")
        if norm_diff:
            # EGNN's coord2radial divides coord_diff by sqrt(radial) + 1: a different model, not computed by the kernels
            raise ValueError("norm_diff=True (coord2radial) is not implemented (model_confs.yaml uses False)")
        if multiple_agg not in (None, 'sum', 'attn'):
            raise ValueError(f"multiple_agg must be None, 'sum' or 'attn' (model.py:82-90), got {multiple_agg!r}")
        self.hidden_nf = hidden_nf
        self.varDT = varDT
        self.multiple_agg = multiple_agg
        if multiple_agg == 'attn':   # registered (and initialised) before everything else, as in model.py:14-15
            self.enc_attn_net = InvariantTemporalAttention(hidden_nf, hidden_dim=hidden_nf)
        self.device = device
        self.n_layers = n_layers
        self.in_node_nf = in_node_nf
        self.in_edge_nf = in_edge_nf
        self.recurrent = recurrent
        self.coords_weight = coords_weight
        self.embedding = nn.Linear(in_node_nf, hidden_nf)
        self.invariant = invariant
        self.norm_vel = norm_vel
        self.module = _GCLHolder(hidden_nf, in_edge_nf, act_fn)
        self.module.n_layers = n_layers
        self.to(self.device)
        self._pack = _ParamPack(self, skip_prefix="enc_attn_net")   # the C layout: embedding + module
        self._attn_pack = None                                       # enc_attn_net's four tensors as one flat buffer
        self._edges = _EdgeCache()
        self.process_group = None
        self.peer_bucket = None

    def enable_data_parallel(self, group=None, average=True, peer_memory=False):
        """Reduce parameter gradients over `group` once per backward.  Default: ONE NCCL all-reduce of the flat gradient
        buffer; average=True leaves the mean in `.grad` (any optimizer), average=False the sum, for
        FlatAdam(grad_scale=1 / world).  peer_memory=True: no collective call at all — the flat gradient buffer lives in
        symmetric memory (dataparallel.PeerGradBucket), `.grad` keeps the LOCAL gradient, and
        FlatAdam(..., peer_bucket=model.peer_bucket) sums all ranks' buffers over NVLink inside its update kernel
        (mean over the ranks)."""
        import torch.distributed as dist

        group = group if group is not None else dist.group.WORLD
        self.peer_bucket = None
        if peer_memory:
            from .dataparallel import PeerGradBucket

            if any(True for k, _ in self.named_parameters() if self._pack.skip_prefix and k.startswith(self._pack.skip_prefix)):
                raise ValueError("peer-memory data parallel needs every parameter inside the flat C layout")
            ps = self._pack.params()
            self.peer_bucket = PeerGradBucket(sum(p.numel() for p in ps), ps[0].device, group)
            self.process_group = (group, bool(average), self.peer_bucket)
        else:
            self.process_group = (group, bool(average))
        return self

    def forward(self, his, x, edges, v, edge_attr, T=10, in_steps=None):
        if x.dim() == 3:
            return self._forward_multi(his, x, edges, v, edge_attr, int(T), in_steps)
        return self._segment(his, x, edges, v, edge_attr, int(T), h_given=False)

    def _forward_multi(self, his, x, edges, v, edge_attr, T, in_steps):
        """Several input frames (model.py:65-90): integrate from frame i to frame i+1 (`diff(in_steps)` sub-steps),
        merge the result with the observed frame ('sum': add; 'attn': invariant temporal attention over the pair,
        model.py:105-139), and finally integrate T sub-steps from the last frame.  Embedding, integration segments and
        merges are all C calls behind ONE autograd node (functional.SegnoMultiFunction): no torch compute kernel runs.
        Returns the integrated state of the last segment (the intended semantics, see the module docstring)."""
        if in_steps is None or x.shape[1] < 2:
            raise ValueError("multi-input SEGNO needs x, v, his of shape [BN, n_inputs >= 2, .] and in_steps [n_inputs]")
        if self.multiple_agg is None:
            raise ValueError("multi-input SEGNO needs multiple_agg='sum' or 'attn' (main.py:110-114)")
        steps = [int(t) for t in torch.diff(torch.as_tensor(in_steps).cpu()).tolist()] + [int(T)]
        n0, L = x.shape[0], x.shape[1]
        if len(steps) != L:
            raise ValueError(f"in_steps has {len(steps)} entries for {L} input frames")
        if min(steps) < 1:
            raise ValueError(f"in_steps must increase strictly (sub-steps per segment: {steps})")
        if edge_attr.requires_grad or his.requires_grad:
            raise ValueError("gradients w.r.t. his / edge_attr are not implemented (the reference callers detach them)")
        dev = x.device
        x = _require_cuda_f32("x", x, (n0, L, 3))
        v = _require_cuda_f32("v", v, (n0, L, 3))
        his = _require_cuda_f32("his", his, (n0, L, self.in_node_nf))
        E = edge_attr.shape[0]
        if n0 == 0 or E % n0 != 0:
            raise ValueError(f"{E} edges / {n0} nodes is not a batch of fully connected graphs")
        N = E // n0 + 1
        if n0 % N != 0:
            raise ValueError(f"{n0} nodes do not divide into graphs of N={N}")
        B = n0 // N
        edge_attr = _require_cuda_f32("edge_attr", edge_attr, (E, self.in_edge_nf))
        self._edges.validate(edges, B, N, dev)
        self.module.n_layers = steps[-1]   # forward_step mutates these on every call (model.py:96-97)
        self.n_layers = steps[-1]
        from ._lib import load_library, check
        from . import _cabi
        import ctypes
        cfg0 = _cabi.NbSegnoConfig(B, N, steps[0], self.in_node_nf, self.in_edge_nf, 1 if self.recurrent else 0,
                                   float(self.coords_weight), 1)
        expected = load_library().nb_segno_param_count(ctypes.byref(cfg0))
        if expected < 0:
            check(-1, "SEGNO configuration")
        flat, params = self._pack.flat_params(expected, dev)
        attn_flat, attn_params = None, []
        if self.multiple_agg == 'attn':
            if self._attn_pack is None:
                self._attn_pack = _ParamPack(self.enc_attn_net)
            attn_flat, attn_params = self._attn_pack.flat_params(_HIDDEN * (_HIDDEN + 1) + 2 * _HIDDEN + 1, dev)
        meta = (B, N, tuple(steps), self.in_node_nf, self.in_edge_nf, 1 if self.recurrent else 0, float(self.coords_weight),
                2 if self.multiple_agg == 'attn' else 1)
        return SegnoMultiFunction.apply(meta, self.process_group, flat, attn_flat, his, x, v, edge_attr, len(params),
                                        *params, *attn_params)

    def _segment(self, his, x, edges, v, edge_attr, T, h_given):
        T = int(T)
        n0 = x.shape[0]
        dev = x.device
        x = _require_cuda_f32("x", x, (n0, 3))
        v = _require_cuda_f32("v", v, (n0, 3))
        his = _require_cuda_f32("his", his, (n0, _HIDDEN if h_given else self.in_node_nf))
        E = edge_attr.shape[0]
        # E = B*N*(N-1) and n0 = B*N  ->  N - 1 = E / n0
        if n0 == 0 or E % n0 != 0:
            raise ValueError(f"{E} edges / {n0} nodes is not a batch of fully connected graphs")
        N = E // n0 + 1
        if n0 % N != 0:
            raise ValueError(f"{n0} nodes do not divide into graphs of N={N}")
        B = n0 // N
        edge_attr = _require_cuda_f32("edge_attr", edge_attr, (E, self.in_edge_nf))
        self._edges.validate(edges, B, N, dev)
        # forward_step mutates these on every call (model.py:96-97)
        self.module.n_layers = T
        self.n_layers = T
        cfg = (B, N, T, self.in_node_nf, self.in_edge_nf, 1 if self.recurrent else 0, float(self.coords_weight),
               1 if h_given else 0)
        from ._lib import load_library, check
        from . import _cabi
        import ctypes
        expected = load_library().nb_segno_param_count(ctypes.byref(_cabi.NbSegnoConfig(*cfg)))
        if expected < 0:
            check(-1, "SEGNO configuration")
        flat, params = self._pack.flat_params(expected, dev)
        return SegnoFunction.apply(cfg, self.process_group, flat, his, x, v, edge_attr, *params)

    def forward_step(self, h, x, edges, v, edge_attr, T=10):
        """model.py:95-102: T weight-shared SEGNO_GCL sub-steps from an already embedded hidden state `h` [BN, 64];
        returns (x, h, v).  Differentiable w.r.t. h, x, v and edge_attr (the C call hands back dL/dh and dL/dedge_attr)."""
        return self._segment(h, x, edges, v, edge_attr, int(T), h_given=True)
