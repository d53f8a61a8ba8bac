"""Drop-in `EGNO` module: same constructor kwargs, forward signature, parameter names and shapes as the
reference class (EGNO/model/egno.py:8-111 on top of EGNN, EGNO/model/basic.py:189-212), so reference
checkpoints load unchanged and `EGNO/main_simulation_simple_no.py:267,360` can call it as is.

The submodules below only *hold* parameters (created in the reference's RNG order so that
`torch.manual_seed(s); EGNO(...)` gives the reference's initial weights); no torch op runs in forward —
the arithmetic is the CUDA kernel sequence behind `nb_egno_forward` / `nb_egno_backward`.
"""
from __future__ import annotations

import torch
from torch import nn

from .functional import EgnoFunction, _EdgeCache, _ParamPack, _require_cuda_f32

_HIDDEN = 64


class _MLPHolder(nn.Module):
    """Parameter container shaped like the reference's BaseMLP (basic.py:34-58): `.mlp.0`, `.mlp.2`."""

    def __init__(self, d_in: int, d_hidden: int, d_out: int, activation: nn.Module, last_act: bool = False):
        super().__init__()
        mods = [nn.Linear(d_in, d_hidden), activation, nn.Linear(d_hidden, d_out)]
        if last_act:
            mods.append(activation)
        self.mlp = nn.Sequential(*mods)


class _ScalarNetHolder(nn.Module):
    """`edge_message_net.scalar_net.mlp.*` (InvariantScalarNet, basic.py:107-123)."""

    def __init__(self, d_in: int, hidden: int, activation: nn.Module):
        super().__init__()
        self.scalar_net = _MLPHolder(d_in, hidden, hidden, activation, last_act=True)


class _EGNNLayerHolder(nn.Module):
    """Parameters of one EGNN_Layer (basic.py:147-165), created in the same order."""

    def __init__(self, in_edge_nf: int, hidden: int, activation: nn.Module):
        super().__init__()
        self.edge_message_net = _ScalarNetHolder(1 + 2 * hidden + in_edge_nf, hidden, activation)
        self.coord_net = _MLPHolder(hidden, hidden, 1, activation)
        self.node_v_net = _MLPHolder(hidden, hidden, 1, activation)
        self.node_net = _MLPHolder(2 * hidden, hidden, hidden, activation)


class _SpectralHolder(nn.Module):
    """`t_conv.weights1` of SpectralConv1d / SpectralConv1d_x (layer_no.py:92-94, :147-150)."""

    def __init__(self, c_in: int, c_out: int, modes: int, scale: float):
        super().__init__()
        self.weights1 = nn.Parameter(scale * torch.rand(c_in, c_out, modes, 2, dtype=torch.float))


class _TimeConvHolder(nn.Module):
    def __init__(self, c_in: int, c_out: int, modes: int, scale: float):
        super().__init__()
        self.t_conv = _SpectralHolder(c_in, c_out, modes, scale)


class EGNO(nn.Module):
    def __init__(self, n_layers, in_node_nf, in_edge_nf, hidden_nf, activation=nn.SiLU(), device='cpu', with_v=False,
                 flat=False, norm=False, use_time_conv=True, num_modes=2, num_timesteps=8, time_emb_dim=32,
                 num_inputs=1, varDT=False, fix_out_size=False):
        super().__init__()
        if hidden_nf != _HIDDEN:
            raise ValueError(f"kernels are specialised for hidden_nf={_HIDDEN} (model_confs.yaml:3), got {hidden_nf}")
        if not with_v:
            raise ValueError("only with_v=True (model_confs.yaml:9) is implemented")
        if flat or norm:
            raise ValueError("flat=True / norm=True are not implemented (model_confs.yaml:4-5 use False)")
        if not isinstance(activation, nn.SiLU):
            raise ValueError("only the SiLU activation (reference default) is implemented")
        if num_inputs < 1:
            raise ValueError("num_inputs must be >= 1")
        self.time_emb_dim = time_emb_dim
        self.num_inputs = num_inputs
        self.varDT = varDT
        self.in_node_nf = in_node_nf            # before the time embedding is appended (egno.py:13-16)
        self.in_edge_nf = in_edge_nf
        self.n_layers = n_layers
        self.with_v = with_v
        # --- EGNN.__init__ order (basic.py:193-203): `layers` registered first, `embedding` created first
        self.layers = nn.ModuleList()
        # egno.py:13-16: one time embedding, or two (input and output times) when there are several input frames
        self.embedding = nn.Linear(in_node_nf + time_emb_dim * (2 if num_inputs > 1 else 1), hidden_nf)
        for _ in range(n_layers):
            self.layers.append(_EGNNLayerHolder(in_edge_nf, hidden_nf, activation))
        self.use_time_conv = use_time_conv
        self.num_timesteps = num_timesteps if not fix_out_size else 10      # egno.py:22
        self.device = device
        self.hidden_nf = hidden_nf
        num_modes = min(num_timesteps, num_modes) if num_timesteps != 5 else min(num_modes, 3)   # egno.py:26
        self.num_modes = num_modes
        if use_time_conv:
            self.time_conv_modules = nn.ModuleList()
            self.time_conv_x_modules = nn.ModuleList()
            for _ in range(n_layers):
                self.time_conv_modules.append(_TimeConvHolder(hidden_nf, hidden_nf, num_modes, 1.0 / (hidden_nf * hidden_nf)))
                self.time_conv_x_modules.append(_TimeConvHolder(2, 2, num_modes, 0.1))
        self.to(self.device)
        self._pack = _ParamPack(self)
        self._edges = _EdgeCache()
        self.process_group = None   # set by enable_data_parallel(): one flat-bucket all-reduce per backward
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

    @staticmethod
    def _times(t, dev, floating):
        """The reference embeds `timesteps.float()` (layer_no.py:12).  Integer times go to the kernels as int64 frame
        indices (what every reference caller passes); floating-point times, integral or not, as that fp32 cast.  The
        cast is an autograd op, so dL/dtimes reaches the caller's tensor in its own dtype and on its own device."""
        return t.to(device=dev, dtype=torch.float32 if floating else torch.int64).contiguous()

    def forward(self, x, h, edge_index, edge_fea, v=None, loc_mean=None, timesteps_in=None, timesteps_out=None):
        T = self.num_timesteps
        if v is None or loc_mean is None:
            raise ValueError("v and loc_mean are required (with_v=True path, main_simulation_simple_no.py:267)")
        L = self.num_inputs
        if L > 1:   # several input frames (egno.py:42-47, main_simulation_simple_no.py:313-327): leading dimension L
            if x.dim() != 3 or x.shape[0] != L or x.shape[2] != 3:
                raise ValueError(f"x must be [num_inputs={L}, B*N, 3], got {tuple(x.shape)}")
            if timesteps_in is None or timesteps_in.dim() != 2 or timesteps_in.shape[1] != L:
                raise ValueError(f"timesteps_in must be [B, {L}] when num_inputs > 1")
            if L > T:
                raise ValueError(f"num_inputs={L} exceeds num_timesteps={T}")
        elif x.dim() != 2 or x.shape[1] != 3:
            raise ValueError(f"x must be [B*N, 3], got {tuple(x.shape)}")
        dev = x.device
        n0 = x.shape[-2]
        lead = (L,) if L > 1 else ()
        if timesteps_out is None:
            # the reference's default (egno.py:40) is 1-D and crashes in get_timestep_embedding; require [B, T]
            raise ValueError("timesteps_out [B, T] is required")
        if timesteps_out.dim() != 2 or timesteps_out.shape[1] != T:
            raise ValueError(f"timesteps_out must be [B, {T}], got {tuple(timesteps_out.shape)}")
        B = timesteps_out.shape[0]
        if n0 % B != 0:
            raise ValueError(f"{n0} nodes do not divide into B={B} graphs")
        N = n0 // B
        if self.use_time_conv and self.num_modes > T // 2 + 1:
            raise ValueError(f"num_modes={self.num_modes} exceeds T//2+1 for T={T} (the reference shape-errors too)")
        if L > 1:   # one input frame: the backward also returns dL/dh, dL/dedge_fea and dL/dloc_mean
            for name, t in (("h", h), ("edge_fea", edge_fea)):
                if t.requires_grad:
                    raise ValueError(f"gradients w.r.t. {name} are not implemented (the reference callers detach it)")
            if loc_mean.requires_grad:
                raise ValueError("gradients w.r.t. loc_mean are not implemented for num_inputs > 1")
        x = _require_cuda_f32("x", x, lead + (n0, 3))
        v = _require_cuda_f32("v", v, lead + (n0, 3))
        h = _require_cuda_f32("h", h, lead + (n0, self.in_node_nf))
        loc_mean = _require_cuda_f32("loc_mean", loc_mean, lead + (n0, 3))
        edge_fea = _require_cuda_f32("edge_fea", edge_fea, lead + (B * N * (N - 1), self.in_edge_nf))
        self._edges.validate(edge_index, B, N, dev)
        # one kind of time for the call: floating point when either tensor is (an integer tensor beside it is exact in fp32)
        floating = timesteps_out.is_floating_point() or (L > 1 and timesteps_in.is_floating_point())
        tsteps = self._times(timesteps_out, dev, floating)
        tsteps_in = None
        if L > 1:
            if timesteps_in.shape[0] != B:
                raise ValueError(f"timesteps_in must be [B={B}, {L}], got {tuple(timesteps_in.shape)}")
            tsteps_in = self._times(timesteps_in, dev, floating)
        cfg = (B, N, T, self.n_layers, self.num_modes if self.use_time_conv else 1, self.in_node_nf, self.in_edge_nf,
               self.time_emb_dim, 1 if self.use_time_conv else 0, L)
        from ._lib import load_library
        from . import _cabi
        import ctypes
        expected = load_library().nb_egno_param_count(ctypes.byref(_cabi.NbEgnoConfig(*cfg)))
        if expected < 0:
            from ._lib import check
            check(-1, "EGNO configuration")
        flat, params = self._pack.flat_params(expected, dev)
        return EgnoFunction.apply(cfg, self.process_group, flat, x, h, edge_fea, v, loc_mean, tsteps, tsteps_in, *params)
