"""CPU restatement of the reference EGNO / SEGNO forward (TEST INFRASTRUCTURE).

Plain PyTorch on CPU tensors, functional over a ``params`` dict keyed by the
reference's own ``state_dict`` names, differentiable (autograd supplies the
gradients the CUDA backward is checked against).  It runs in fp32 (the
reference's dtype) or fp64 (a tighter yardstick when judging which of two fp32
implementations is closer).

Every function cites the reference lines (relative to /root/reference) it
restates.  Pinned by tests/test_oracle_golden.py against vectors produced by the
reference's own modules (tests/golden/make_golden.py); the reference itself has
no tests or golden vectors for this path -> "parity unpinned by reference tests".
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import torch

Tensor = torch.Tensor


# ----------------------------------------------------------------------------- helpers
def silu(x: Tensor) -> Tensor:
    return x * torch.sigmoid(x)


def linear(x: Tensor, p: Dict[str, Tensor], name: str) -> Tensor:
    return x @ p[name + ".weight"].t() + p[name + ".bias"]


def canonical_edges(batch: int, n_nodes: int) -> Tuple[Tensor, Tensor]:
    """Fully connected edge list, per graph `for i: for j != i`, graphs offset by N*b.

    EGNO/simulation/dataset_simple.py:64-71 (single graph) and :101-111 (batch)."""
    i = torch.arange(n_nodes).repeat_interleave(n_nodes)
    j = torch.arange(n_nodes).repeat(n_nodes)
    keep = i != j
    i, j = i[keep], j[keep]
    off = (torch.arange(batch) * n_nodes).repeat_interleave(i.numel())
    return i.repeat(batch) + off, j.repeat(batch) + off


def segment_sum(data: Tensor, idx: Tensor, n: int) -> Tensor:
    """EGNO/model/basic.py:16-19 (aggregate, sum) == SEGNO/models/models/gcl.py:7-13."""
    out = data.new_zeros((n, data.shape[1]))
    return out.index_add(0, idx, data)


def segment_mean(data: Tensor, idx: Tensor, n: int) -> Tensor:
    """EGNO/model/basic.py:22-28: sum / count.clamp(min=1).

    SEGNO's gcl.py:16-23 builds a dense one-hot matrix, L1-normalises its rows and
    multiplies: the same mean (rows with no edge give 0 in both)."""
    s = segment_sum(data, idx, n)
    cnt = segment_sum(torch.ones_like(data), idx, n)
    return s / cnt.clamp(min=1)


# ----------------------------------------------------------------------------- EGNO pieces
def timestep_embedding(timesteps: Tensor, dim: int, max_positions: int = 10000) -> Tensor:
    """EGNO/model/layer_no.py:8-17.  timesteps [B,T] -> [B,T,dim] = [sin | cos]."""
    half = dim // 2
    scale = math.log(max_positions) / (half - 1)
    freq = torch.exp(torch.arange(half, dtype=torch.float32, device=timesteps.device) * -scale)
    arg = timesteps.float()[:, :, None] * freq[None, None, :]
    emb = torch.cat([torch.sin(arg), torch.cos(arg)], dim=-1)
    if dim % 2 == 1:
        emb = torch.nn.functional.pad(emb, (0, 1))
    return emb


def spectral_conv(x: Tensor, w: Tensor) -> Tensor:
    """SpectralConv1d / SpectralConv1d_x forward (layer_no.py:96-109, :151-162).

    x [T, N, ..., Cin]; w [Cin, Cout, modes, 2].  rfft over dim 0, keep the first
    `modes` coefficients, complex channel mix per mode, irfft back to length T."""
    T = x.shape[0]
    modes = w.shape[2]
    wc = torch.view_as_complex(w.contiguous())
    xf = torch.fft.rfft(x, dim=0)[:modes]
    yf = torch.einsum("m...i,iom->m...o", xf, wc.to(xf.dtype))
    return torch.fft.irfft(yf, n=T, dim=0)


def egnn_layer(p: Dict[str, Tensor], pre: str, x: Tensor, h: Tensor, row: Tensor, col: Tensor,
               edge_fea: Tensor, v: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """EGNN_Layer.forward, EGNO/model/basic.py:167-186 (with_v=True, norm=False, flat=False)."""
    n = x.shape[0]
    rij = x[row] - x[col]                                         # :169
    radial = (rij * rij).sum(-1, keepdim=True)                    # :93 (K=1 Gram matrix)
    # InvariantScalarNet: [radial | h_row | h_col | edge_fea]      :98, :170
    z = torch.cat([radial, h[row], h[col], edge_fea], dim=-1)
    en = pre + ".edge_message_net.scalar_net.mlp"
    m = silu(linear(silu(linear(z, p, en + ".0")), p, en + ".2"))  # last_act=True :46-51
    cn = pre + ".coord_net.mlp"
    c = linear(silu(linear(m, p, cn + ".0")), p, cn + ".2")        # :172
    f = rij * c                                                    # :173
    tot_f = segment_mean(f, row, n).clamp(-100, 100)               # :174-175 (clamp AFTER mean)
    vn = pre + ".node_v_net.mlp"
    s = linear(silu(linear(h, p, vn + ".0")), p, vn + ".2")
    x_new = x + s * v + tot_f                                      # :178 (pre-update h)
    tot_m = segment_sum(m, row, n)                                 # :182
    nn_ = pre + ".node_net.mlp"
    h_new = linear(silu(linear(torch.cat([h, tot_m], -1), p, nn_ + ".0")), p, nn_ + ".2")  # :183-185
    return x_new, v, h_new


def egno_forward(p: Dict[str, Tensor], x: Tensor, h: Tensor, row: Tensor, col: Tensor, edge_fea: Tensor,
                 v: Tensor, loc_mean: Tensor, timesteps_out: Tensor, *, n_layers: int, num_timesteps: int,
                 time_emb_dim: int = 32, use_time_conv: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
    """EGNO.forward, EGNO/model/egno.py:37-111, num_inputs == 1.

    Returns (x [T*BN,3], v [T*BN,3], h [T*BN,H]) in t-major node order."""
    T = num_timesteps
    nn_ = h.shape[0]
    ne = row.shape[0]
    B = timesteps_out.shape[0]
    temb = timestep_embedding(timesteps_out, time_emb_dim).to(x.dtype)           # :50  [B,T,D]
    # :66 -- [T,1,B,D].repeat(1, BN/B, 1, 1).reshape(T, BN, D): node k gets batch (k mod B)
    temb = temb.transpose(0, 1).unsqueeze(1).repeat(1, nn_ // B, 1, 1).reshape(T, -1, time_emb_dim)
    hh = torch.cat([h.unsqueeze(0).repeat(T, 1, 1), temb], dim=-1).reshape(T * nn_, -1)  # :63,:72,:74
    hh = linear(hh, p, "embedding")                                               # :76
    node_off = (torch.arange(T, device=row.device) * nn_).repeat_interleave(ne)   # :53-55, :91-92
    rr = row.repeat(T) + node_off
    cc = col.repeat(T) + node_off
    xx = x.repeat(T, 1)
    vv = v.repeat(T, 1)
    lm = loc_mean.repeat(T, 1)
    ef = edge_fea.repeat(T, 1)
    H = hh.shape[-1]
    for i in range(n_layers):
        if use_time_conv:
            # TimeConv: x + LeakyReLU(conv(x))  layer_no.py:121-126
            h3 = hh.view(T, nn_, H)
            conv = spectral_conv(h3, p[f"time_conv_modules.{i}.t_conv.weights1"])
            hh = (h3 + torch.nn.functional.leaky_relu(conv, 0.01)).reshape(T * nn_, H)
            # TimeConv_x on stack(x - mean, v): x + conv(x), no activation  egno.py:103-108, layer_no.py:173-178
            X = torch.stack([xx - lm, vv], dim=-1).view(T, nn_, 3, 2)
            X = X + spectral_conv(X, p[f"time_conv_x_modules.{i}.t_conv.weights1"])
            xx = X[..., 0].reshape(T * nn_, 3) + lm
            vv = X[..., 1].reshape(T * nn_, 3)
        xx, vv, hh = egnn_layer(p, f"layers.{i}", xx, hh, rr, cc, ef, vv)
    return xx, vv, hh


def frame_to_input(num_timesteps: int, num_inputs: int):
    """repeat_elements_to_exact_shape (EGNO/utils.py:115-131): frame t of the T outputs is fed by input
    min(t // (T // L), L - 1) — every input T // L times, the last one also covers the remainder."""
    reps = num_timesteps // num_inputs
    return [min(t // reps, num_inputs - 1) for t in range(num_timesteps)]


def egno_forward_multi(p: Dict[str, Tensor], x: Tensor, h: Tensor, row: Tensor, col: Tensor, edge_fea: Tensor,
                       v: Tensor, loc_mean: Tensor, timesteps_in: Tensor, timesteps_out: Tensor, *, n_layers: int,
                       num_timesteps: int, time_emb_dim: int = 32) -> Tuple[Tensor, Tensor, Tensor]:
    """EGNO.forward, EGNO/model/egno.py:37-111, num_inputs > 1.

    x, v, loc_mean [L,BN,3]; h [L,BN,F]; edge_fea [L,E,2]; timesteps_in [B,L]; timesteps_out [B,T]."""
    T, L = num_timesteps, x.shape[0]
    nn_ = h.shape[1]
    ne = row.shape[0]
    B = timesteps_out.shape[0]
    tmap = frame_to_input(T, L)
    ts_in = timesteps_in[:, tmap]                                                  # :45  [B,T]
    temb_in = timestep_embedding(ts_in, time_emb_dim).to(x.dtype)                 # :46
    temb_out = timestep_embedding(timesteps_out, time_emb_dim).to(x.dtype)        # :50
    bc = lambda e: e.transpose(0, 1).unsqueeze(1).repeat(1, nn_ // B, 1, 1).reshape(T, -1, time_emb_dim)  # :66,:69
    hh = torch.cat([h[tmap], bc(temb_in), bc(temb_out)], dim=-1).reshape(T * nn_, -1)   # :59-61,:70,:74
    hh = linear(hh, p, "embedding")
    node_off = (torch.arange(T, device=row.device) * nn_).repeat_interleave(ne)
    rr = row.repeat(T) + node_off
    cc = col.repeat(T) + node_off
    xx = x[tmap].reshape(T * nn_, 3)                                               # :80-83
    vv = v[tmap].reshape(T * nn_, 3)
    lm = loc_mean[tmap].reshape(T * nn_, 3)
    ef = edge_fea[tmap].reshape(T * ne, -1)
    H = hh.shape[-1]
    for i in range(n_layers):
        h3 = hh.view(T, nn_, H)
        conv = spectral_conv(h3, p[f"time_conv_modules.{i}.t_conv.weights1"])
        hh = (h3 + torch.nn.functional.leaky_relu(conv, 0.01)).reshape(T * nn_, H)
        X = torch.stack([xx - lm, vv], dim=-1).view(T, nn_, 3, 2)
        X = X + spectral_conv(X, p[f"time_conv_x_modules.{i}.t_conv.weights1"])
        xx = X[..., 0].reshape(T * nn_, 3) + lm
        vv = X[..., 1].reshape(T * nn_, 3)
        xx, vv, hh = egnn_layer(p, f"layers.{i}", xx, hh, rr, cc, ef, vv)
    return xx, vv, hh


def egno_features_multi(loc: Tensor, vel: Tensor, charges: Tensor, row: Tensor, col: Tensor):
    """prepare_inputs, EGNO/main_simulation_simple_no.py:313-327 (num_inputs > 1).
    loc, vel [L,B,N,3]; charges [B,N,1] -> (loc [L,BN,3], vel, edge_attr [L,E,2], nodes [L,BN,2], loc_mean [L,BN,3])."""
    L, B, N, _ = loc.shape
    loc_mean = loc.mean(dim=2, keepdim=True).repeat(1, 1, N, 1).reshape(L, -1, 3)
    loc = loc.reshape(L, -1, 3)
    vel = vel.reshape(L, -1, 3)
    q = charges.reshape(-1, 1)
    nodes = torch.cat([torch.sqrt((vel ** 2).sum(-1, keepdim=True)), q.repeat(L, 1, 1).reshape(L, -1, 1)], dim=-1)
    qq = (q[row] * q[col]).unsqueeze(0).repeat(L, 1, 1)
    dist = ((loc[:, row] - loc[:, col]) ** 2).sum(2, keepdim=True)
    return loc, vel, torch.cat([qq, dist], 2), nodes, loc_mean


# ----------------------------------------------------------------------------- SEGNO pieces
def segno_gcl(p: Dict[str, Tensor], h: Tensor, row: Tensor, col: Tensor, x: Tensor, v: Tensor,
              edge_attr: Tensor, n_layers: int, recurrent: bool = True,
              coords_weight: float = 1.0) -> Tuple[Tensor, Tensor, Tensor]:
    """SEGNO_GCL.forward, SEGNO/models/models/gcl.py:111-119 (one 2nd-order sub-step)."""
    n = x.shape[0]
    rij = x[row] - x[col]                                            # :106
    radial = (rij * rij).sum(1, keepdim=True)                        # :107
    z = torch.cat([h[row], h[col], radial, edge_attr], dim=1)        # :78  (h first)
    m = silu(linear(silu(linear(z, p, "module.edge_mlp.0")), p, "module.edge_mlp.2"))   # :39-43
    c = linear(silu(linear(m, p, "module.coord_mlp.0")), p, "module.coord_mlp.2")      # :50-60
    trans = (rij * c).clamp(-100, 100)                               # :99-100 (clamp per edge, BEFORE mean)
    agg = segment_mean(trans, row, n) * coords_weight                # :101-102
    v = v + agg * (1 / n_layers)                                     # :116
    x = x + v * (1 / n_layers)                                       # :117
    tot_m = segment_sum(m, row, n)                                   # :87
    out = linear(silu(linear(torch.cat([h, tot_m], 1), p, "module.node_mlp.0")), p, "module.node_mlp.2")  # :91-92
    h = h + out if recurrent else out                                # :93-94
    return h, x, v


def segno_forward(p: Dict[str, Tensor], his: Tensor, x: Tensor, row: Tensor, col: Tensor, v: Tensor,
                  edge_attr: Tensor, T: int, recurrent: bool = True,
                  coords_weight: float = 1.0) -> Tuple[Tensor, Tensor, Tensor]:
    """The *intended* SEGNO forward: forward_step(embedding(his), ...) (SEGNO/models/model.py:73,:95-102).

    (The literal SEGNO.forward at reference HEAD, model.py:53-92, returns its inputs — SURVEY.md §0.)
    Returns (x, h, v) in the reference's return order."""
    h = linear(his, p, "embedding")                                   # :73
    for _ in range(T):                                                # :96-100 (n_layers := T)
        h, x, v = segno_gcl(p, h, row, col, x, v, edge_attr, n_layers=T, recurrent=recurrent,
                            coords_weight=coords_weight)
    return x, h, v


def segno_forward_multi(p: Dict[str, Tensor], his: Tensor, x: Tensor, row: Tensor, col: Tensor, v: Tensor,
                        edge_attr: Tensor, T: int, in_steps, multiple_agg: str, recurrent: bool = True
                        ) -> Tuple[Tensor, Tensor, Tensor]:
    """The intended multi-input SEGNO forward (SEGNO/models/model.py:65-90 with :105-139): his [BN,L,F], x, v [BN,L,3].
    Integrate `diff(in_steps)` sub-steps between consecutive input frames, merge the prediction with the observed frame
    ('sum': add, 'attn': InvariantTemporalAttention over the pair), then T sub-steps from the last frame; returns the
    integrated state of the last segment (HEAD returns the segment's *inputs*, SURVEY.md 0)."""
    steps = torch.diff(torch.as_tensor(in_steps)).tolist() + [T]
    h = linear(his, p, "embedding")                                   # :73
    h_, x_, v_ = h[:, 0, :], x[:, 0, :], v[:, 0, :]
    xi = hi = vi = None
    for i, step in enumerate(steps):
        hi, xi, vi = h_, x_, v_
        for _ in range(int(step)):                                    # forward_step, :95-102
            hi, xi, vi = segno_gcl(p, hi, row, col, xi, vi, edge_attr, n_layers=int(step), recurrent=recurrent)
        if i < len(steps) - 1:
            if multiple_agg == "sum":                                 # :83-86
                h_, x_, v_ = h[:, i + 1, :] + hi, x[:, i + 1, :] + xi, v[:, i + 1, :] + vi
            else:                                                     # :87-90, :105-139
                hs = torch.stack([h[:, i + 1, :], hi], dim=1)
                xs = torch.stack([x[:, i + 1, :], xi], dim=1)
                vs = torch.stack([v[:, i + 1, :], vi], dim=1)
                feats = torch.cat([vs.norm(dim=-1, keepdim=True), hs], dim=-1)
                a = linear(torch.tanh(linear(feats, p, "enc_attn_net.attn_mlp.0")), p, "enc_attn_net.attn_mlp.2").softmax(dim=1)
                x_, v_, h_ = (a * xs).sum(1), (a * vs).sum(1), (a * hs).sum(1)
    return xi, hi, vi


def segno_features_multi(loc: Tensor, vel: Tensor, charges: Tensor, row: Tensor, col: Tensor):
    """SEGNO/train_nbody.py:110-118 (several input frames): loc, vel [L,B,N,3] -> his [BN,L,1], x, v [BN,L,3],
    edge_attr [E,2] (charge products and squared distances of the LAST input frame)."""
    L, B, N, _ = loc.shape
    x = loc.reshape(L, B * N, 3).transpose(0, 1).contiguous()
    v = vel.reshape(L, B * N, 3).transpose(0, 1).contiguous()
    q = charges.reshape(-1, 1)
    his = torch.sqrt((v ** 2).sum(-1, keepdim=True))
    dist = ((x[row, -1, :] - x[col, -1, :]) ** 2).sum(1, keepdim=True)
    return his, x, v, torch.cat([q[row] * q[col], dist], 1)


# ----------------------------------------------------------------------------- featurisation (callers)
def egno_features(loc: Tensor, vel: Tensor, charges: Tensor, row: Tensor, col: Tensor
                  ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """prepare_inputs, EGNO/main_simulation_simple_no.py:329-338 (num_inputs == 1).

    loc, vel [B,N,3]; charges [B,N,1] -> (loc[BN,3], vel[BN,3], edge_attr[E,2], nodes[BN,2], loc_mean[BN,3])."""
    B, N, _ = loc.shape
    loc_mean = loc.mean(dim=1, keepdim=True).repeat(1, N, 1).view(-1, 3)
    loc = loc.reshape(-1, 3)
    vel = vel.reshape(-1, 3)
    q = charges.reshape(-1, 1)
    nodes = torch.cat([torch.sqrt((vel ** 2).sum(1, keepdim=True)), q], dim=1)
    qq = q[row] * q[col]                      # dataset_simple.py:52-53 (edge_attr = q_i q_j)
    dist = ((loc[row] - loc[col]) ** 2).sum(1, keepdim=True)
    return loc, vel, torch.cat([qq, dist], 1), nodes, loc_mean


def segno_features(loc: Tensor, vel: Tensor, charges: Tensor, row: Tensor, col: Tensor
                   ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """SEGNO/train_nbody.py:93,119-123.  -> (his[BN,1], loc[BN,3], vel[BN,3], edge_attr[E,2])."""
    loc = loc.reshape(-1, 3)
    vel = vel.reshape(-1, 3)
    q = charges.reshape(-1, 1)
    his = torch.sqrt((vel ** 2).sum(1, keepdim=True))
    qq = q[row] * q[col]
    dist = ((loc[row] - loc[col]) ** 2).sum(1, keepdim=True)
    return his, loc, vel, torch.cat([qq, dist], 1)


# ----------------------------------------------------------------------------- energies (evaluation only)
def energy_charged(loc: Tensor, vel: Tensor, charges: Tensor) -> Tensor:
    """utils.py:126-144 (tot_energy_charged_batch): K + 0.5*sum_{i!=j} q_i q_j / |r_ij|.  [B,N,3] -> [B]."""
    K = 0.5 * (vel ** 2).sum((-1, -2))
    d = (loc[:, :, None, :] - loc[:, None, :, :]).norm(dim=-1)
    d = torch.where(d == 0, torch.full_like(d, float("inf")), d)
    q = charges.reshape(loc.shape[0], -1)
    U = 0.5 * ((q[:, :, None] * q[:, None, :]) / d).sum((-1, -2))
    return K + U


def energy_gravity(loc: Tensor, vel: Tensor, mass: Tensor, G: float = 1.0) -> Tensor:
    """utils.py:175-195 (tot_energy_gravity_batch).  [B,N,3], mass [B,N,1] -> [B]."""
    KE = 0.5 * (mass * vel ** 2).sum((-1, -2))
    d = (loc[:, :, None, :] - loc[:, None, :, :]).norm(dim=-1)
    inv = torch.where(d > 0, 1.0 / d, torch.zeros_like(d))
    m = mass.reshape(loc.shape[0], -1)
    pe = -(m[:, :, None] * m[:, None, :]) * inv
    PE = G * torch.triu(pe, 1).sum((-1, -2))
    return KE + PE


def trajectory_mse(pred_tmajor: Tensor, target_bnt3: Tensor, only_first: bool = False) -> Tuple[Tensor, Tensor]:
    """The callers' loss (EGNO/main_simulation_simple_no.py:268-276): pred [T*B*N, 3] frame-major as the model returns
    it, target [B*N, T, 3] as the loader holds it -> (loss, losses[T]) with
    losses = MSELoss(reduction='none')(pred, target).mean over (nodes, xyz); loss = losses[0] | losses.mean()."""
    bn, T = target_bnt3.shape[0], target_bnt3.shape[1]
    pred = pred_tmajor.reshape(T, bn, 3).transpose(0, 1)          # [BN, T, 3]   (:269)
    losses = ((pred - target_bnt3) ** 2).mean((0, 2))             # [T]          (:273)
    return (losses[0] if only_first else losses.mean()), losses   # (:276)
