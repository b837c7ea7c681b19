"""Torch (CPU) interpreter of the engine's four-sweep layer program.  TEST INFRASTRUCTURE ONLY.

The sm_100a engine does not replay PyTorch's reverse-over-reverse autograd graph.  It evaluates
``d Phi / d x`` for ``Phi(x) = h(G(x), g)``, ``G = grad_W L(x, W)`` as a *weight-direction tangent* of the
input gradient (SURVEY.md section 7.3, DESIGN.md section 3):

    v      = d h / d G                                  (elementwise in (G, g) + a few global scalars)
    dPhi/dx = d/d eps  grad_x L(x, W + eps v) |_{eps=0}

which needs exactly four sweeps over the static program produced by ``breaching_b200.compiler``:
forward (F), backward (B, gives G), tangent-forward (TF) and tangent-backward (TB).  This module
implements those sweeps op by op with plain torch functional calls so that

  * the lowering of ``nn.Module`` graphs can be validated on the CPU against autograd's double
    backward (``tests/test_program_interp.py``), in float64 to ~1e-12, and
  * every CUDA kernel has a one-to-one CPU restatement to be compared with in the ``-m gpu`` tests.

It mirrors what the reference computes at ``attacks/auxiliaries/objectives.py:40-46`` (G) and
``attacks/optimization_based_attack.py:165`` (second backward).
"""
import torch
import torch.nn.functional as F

from breaching_b200 import compiler as C
from oracle import transformer_interp as TI


def objective_direction(kind, G, g, scale=1.0, tag_scale=0.1, scale_scheme="linear", fudge=1e-7, mask_value=1e-6):
    """Return ``(value, v)`` with ``v_l = d value / d G_l`` for the matching objectives of
    ``attacks/auxiliaries/objectives.py`` (closed forms; SURVEY.md section 7.3)."""
    dot = sum((a * b).sum() for a, b in zip(G, g))
    if kind == "euclidean":
        val = 0.5 * sum((a - b).pow(2).sum() for a, b in zip(G, g)) * scale
        return val, [scale * (a - b) for a, b in zip(G, g)]
    if kind == "l1":
        val = 0.5 * sum((a - b).abs().sum() for a, b in zip(G, g)) * scale
        return val, [0.5 * scale * torch.sign(a - b) for a, b in zip(G, g)]
    if kind == "tag-euclidean":
        L = len(G)
        if scale_scheme == "linear":
            w = torch.arange(L, 0, -1, dtype=G[0].dtype) / L
        elif scale_scheme == "exp":
            w = torch.arange(L, 0, -1, dtype=G[0].dtype).softmax(dim=0)
            w = w / w[0]
        else:
            w = G[0].new_ones(L)
        val = 0.5 * scale * sum((a - b).pow(2).sum() + tag_scale * wl * (a - b).abs().sum() for a, b, wl in zip(G, g, w))
        return val, [scale * ((a - b) + 0.5 * tag_scale * wl * torch.sign(a - b)) for a, b, wl in zip(G, g, w)]
    if kind == "masked-cosine-similarity":
        masks = [(b.abs() > mask_value).to(b.dtype) for b in g]
        Gm = [a * m for a, m in zip(G, masks)]
        gm = [b * m for b, m in zip(g, masks)]
        val, v = objective_direction("cosine-similarity", Gm, gm, scale)
        return val, [vi * m for vi, m in zip(v, masks)]
    if kind in ("cosine-similarity", "angular", "fast-cosine-similarity"):
        nG = sum(a.pow(2).sum() for a in G).sqrt()
        ng = sum(b.pow(2).sum() for b in g).sqrt()
        cos = dot / (nG * ng)
        alpha = -1.0 / (nG * ng)  # d(1-cos)/dG = alpha * g + beta * G
        beta = dot / (nG.pow(3) * ng)
        if kind == "fast-cosine-similarity":
            beta = beta * 0
        if kind == "angular":
            c = cos.clamp(min=-1 + fudge, max=1 - fudge)
            val = torch.acos(c) / torch.pi * scale
            inside = (cos > -1 + fudge) & (cos < 1 - fudge)
            # d acos(c)/dc = -1/sqrt(1-c^2);  d cos/dG = -(alpha g + beta G)
            factor = (1.0 / torch.sqrt(1 - c * c)) / torch.pi * scale * inside
            return val, [factor * (alpha * b + beta * a) for a, b in zip(G, g)]
        return (1 - cos) * scale, [scale * (alpha * b + beta * a) for a, b in zip(G, g)]
    raise ValueError(kind)


class ProgramInterpreter:
    """Evaluates the program with torch ops.  Parameters / running stats are read from ``model``."""

    def __init__(self, model, prog, dtype=torch.float64):
        self.prog = prog
        self.dtype = dtype
        self.P = [p.detach().to(dtype) for p in model.parameters()]
        mods = C.bn_modules(model, prog)
        self.bn = [None if (m is None or m.running_mean is None) else (m.running_mean.detach().to(dtype), m.running_var.detach().to(dtype))
                   for m in mods]

    # ------------------------------------------------------------------ helpers
    def _flat_in(self, op, t):
        """Linear consumes the NCHW-flattened feature map (torch.flatten order)."""
        return t.reshape(t.shape[0], -1)

    def _bn_consts(self, i, op):
        rm, rv = self.bn[i]
        inv = 1.0 / torch.sqrt(rv + op.eps)
        return rm.view(1, -1, 1, 1), inv.view(1, -1, 1, 1)

    # ---- token-sequence helpers (rows = batch * seq_len; formulas verified in oracle/transformer_interp.py)
    @staticmethod
    def _pos_rows(pos, rows, T):
        return pos[:T].repeat(rows // T, 1).view(rows, -1, 1, 1)

    @staticmethod
    def _split_heads(t, heads, T):
        rows, three_d = t.shape[0], t.shape[1]
        d = three_d // 3
        q, k, v = t.view(rows // T, T, three_d).split(d, dim=-1)
        f = lambda u: u.reshape(rows // T, T, heads, d // heads).transpose(1, 2)  # noqa: E731  [B, h, T, dh]
        return f(q), f(k), f(v)

    @staticmethod
    def _merge_heads(t):
        B, h, T, dh = t.shape
        return t.transpose(1, 2).reshape(B * T, h * dh, 1, 1)

    def _token_loss(self, a, aux, targets, T):
        """CausalLoss (losses.py:7-26): row (b, t) predicts the target of row (b, t + 1); the last position of each sequence
        has no target.  ``targets``: token ids [B, T] or class probabilities [B, T, V]."""
        z = a[self.prog.logits].flatten(1)
        rows, V = z.shape
        keep = (torch.arange(rows) % T) != (T - 1)
        logp = torch.log_softmax(z, dim=1)
        if targets.dtype == torch.long:
            q = F.one_hot(targets.reshape(-1), V).to(self.dtype)
        else:
            q = targets.reshape(rows, V).to(self.dtype)
        q_next = torch.zeros_like(q)
        q_next[:-1] = q[1:]
        q_next = q_next * keep.view(-1, 1)
        M = int(keep.sum())
        loss = -(q_next * logp).sum() / M
        self.a, self.aux, self.p, self.onehot, self.loss = a, aux, logp.exp(), q_next, loss
        self.row_keep, self.M = keep.view(-1, 1).to(self.dtype), M
        return loss

    # ------------------------------------------------------------------ sweeps
    def forward(self, x, labels, soft_labels=None):
        prog = self.prog
        T = getattr(prog, "seq_len", 0)
        if T:   # token-sequence program: the candidate [B, T, d] becomes rows x features
            x = x.reshape(-1, x.shape[-1], 1, 1)
        a = {0: x.to(self.dtype)}
        aux = {}
        for i, op in enumerate(prog.ops):
            xin = a[op.tin]
            if op.kind == C.OP_CONV:
                b = None if op.b < 0 else self.P[op.b]
                a[op.tout] = F.conv2d(xin, self.P[op.w], b, stride=op.stride, padding=op.pad)
            elif op.kind == C.OP_BNACT:
                u = xin
                if op.has_bn:
                    if getattr(op, "bn_train", False):   # batch statistics of this very input (biased variance, F.batch_norm)
                        rm = xin.mean(dim=(0, 2, 3), keepdim=True)
                        inv = 1.0 / torch.sqrt(xin.var(dim=(0, 2, 3), unbiased=False, keepdim=True) + op.eps)
                        aux[("inv", i)] = inv
                    else:
                        rm, inv = self._bn_consts(i, op)
                    xhat = (xin - rm) * inv
                    u = self.P[op.gamma].view(1, -1, 1, 1) * xhat + self.P[op.beta].view(1, -1, 1, 1)
                    aux[i] = xhat
                if op.res >= 0:
                    u = u + a[op.res]
                a[op.tout] = torch.relu(u) if op.relu else u
            elif op.kind == C.OP_MAXPOOL:
                out, idx = F.max_pool2d(xin, op.R, op.stride, op.pad, return_indices=True)
                a[op.tout], aux[i] = out, idx
            elif op.kind == C.OP_AVGPOOL:
                a[op.tout] = xin.mean(dim=(2, 3), keepdim=True)
            elif op.kind == C.OP_LINEAR:
                b = None if op.b < 0 else self.P[op.b]
                a[op.tout] = F.linear(self._flat_in(op, xin), self.P[op.w], b).view(xin.shape[0], -1, 1, 1)
            elif op.kind == C.OP_POSADD:      # + learnable positional embedding of position (row mod T)
                a[op.tout] = xin + self._pos_rows(self.P[op.w], xin.shape[0], T)
            elif op.kind == C.OP_LAYERNORM:
                y, xh, inv = TI._ln_forward(xin.flatten(1), self.P[op.gamma], self.P[op.beta], op.eps)
                a[op.tout], aux[i] = y.view_as(xin), (xh, inv)
            elif op.kind == C.OP_ATTENTION:
                Q, K, Vv = self._split_heads(xin, op.R, T)
                P_ = torch.softmax(Q @ K.transpose(-1, -2) / (Q.shape[-1] ** 0.5), dim=-1)
                a[op.tout], aux[i] = self._merge_heads(P_ @ Vv), (Q, K, Vv, P_)
        if T:
            return self._token_loss(a, aux, soft_labels if soft_labels is not None else labels, T)
        z = a[prog.logits].view(x.shape[0], -1)
        logp = torch.log_softmax(z, dim=1)
        if soft_labels is None:
            loss = -logp.gather(1, labels.view(-1, 1)).mean()
            onehot = F.one_hot(labels, z.shape[1]).to(self.dtype)
        else:
            onehot = soft_labels.to(self.dtype)
            loss = -(onehot * logp).sum(dim=1).mean()
        self.a, self.aux, self.p, self.onehot, self.loss = a, aux, logp.exp(), onehot, loss
        return loss

    def _reverse(self, seed, V=None, d_prev=None, inject=None, want_G=True, want_dx=False):
        """Shared reverse sweep.

        * ``V is None``: ordinary backward (sweep B): returns parameter gradients ``G``, saves deltas.
        * ``V`` given (sweep TB): propagates tangent deltas; the additional ``v``-terms use the deltas
          ``d_prev`` saved by sweep B;  ``inject[tid]`` tensors (regulariser adjoints) are added to the
          stream when that tensor's delta is consumed.
        """
        prog = self.prog
        d = {prog.logits: seed.view(seed.shape[0], -1, 1, 1)}
        G = [None] * len(self.P)
        du_saved = {}
        if V is None:
            self.rsave = {}

        def add(tid, val):
            d[tid] = val if tid not in d else d[tid] + val

        for i in reversed(range(len(prog.ops))):
            op = prog.ops[i]
            dout = d[op.tout]
            if inject is not None and op.tout in inject:
                dout = dout + inject[op.tout]
            xin = self.a[op.tin]
            if op.kind == C.OP_CONV:
                if V is None:
                    if want_G:
                        G[op.w] = torch.nn.grad.conv2d_weight(xin, self.P[op.w].shape, dout, stride=op.stride, padding=op.pad)
                        if op.b >= 0:
                            G[op.b] = dout.sum(dim=(0, 2, 3))
                    if op.tin != 0 or want_dx:
                        add(op.tin, torch.nn.grad.conv2d_input(xin.shape, self.P[op.w], dout, stride=op.stride, padding=op.pad))
                else:
                    val = torch.nn.grad.conv2d_input(xin.shape, self.P[op.w], dout, stride=op.stride, padding=op.pad)
                    val = val + torch.nn.grad.conv2d_input(xin.shape, V[op.w], d_prev[op.tout], stride=op.stride, padding=op.pad)
                    add(op.tin, val)
            elif op.kind == C.OP_BNACT:
                du = dout * (self.a[op.tout] > 0).to(self.dtype) if op.relu else dout
                du_saved[i] = du
                if op.res >= 0:
                    add(op.res, du)
                if op.has_bn and getattr(op, "bn_train", False):
                    # train-mode BN: the statistics depend on the input.  With xh the normalised input, m(.) the mean over
                    # (N, H, W) per channel and inv = 1/sigma:
                    #   B :  dx  = gamma inv (du - m(du) - xh m(du xh))
                    #   TB:  dx' = (v_gamma inv + gamma inv') w + gamma inv (du' - m(du') - xh' m(du xh) - xh m(du' xh + du xh')),
                    #        w = du - m(du) - xh m(du xh),  inv' = -inv^2 m(xh x'),  xh' from the tangent-forward sweep
                    xh, inv = self.aux[i], self.aux[("inv", i)]
                    gam = self.P[op.gamma].view(1, -1, 1, 1)
                    m = lambda t: t.mean(dim=(0, 2, 3), keepdim=True)  # noqa: E731
                    if V is None:
                        if want_G:
                            G[op.gamma] = (du * xh).sum(dim=(0, 2, 3))
                            G[op.beta] = du.sum(dim=(0, 2, 3))
                        add(op.tin, gam * inv * (du - m(du) - xh * m(du * xh)))
                    else:
                        duB = self.du_B[i]
                        xhd, xd = self.taux[i], self.ta[op.tin]
                        vg = V[op.gamma].view(1, -1, 1, 1)
                        invd = -inv * inv * m(xh * xd)
                        w = duB - m(duB) - xh * m(duB * xh)
                        wd = du - m(du) - xhd * m(duB * xh) - xh * m(du * xh + duB * xhd)
                        add(op.tin, (vg * inv + gam * invd) * w + gam * inv * wd)
                elif op.has_bn:
                    rm, inv = self._bn_consts(i, op)
                    s = self.P[op.gamma].view(1, -1, 1, 1) * inv
                    if V is None:
                        if want_G:
                            G[op.gamma] = (du * self.aux[i]).sum(dim=(0, 2, 3))
                            G[op.beta] = du.sum(dim=(0, 2, 3))
                        add(op.tin, s * du)
                    else:
                        add(op.tin, s * du + V[op.gamma].view(1, -1, 1, 1) * inv * self.du_B[i])
                else:
                    add(op.tin, du)
            elif op.kind == C.OP_MAXPOOL:
                add(op.tin, _maxpool_scatter(dout, self.aux[i], xin.shape))
            elif op.kind == C.OP_AVGPOOL:
                add(op.tin, (dout / (xin.shape[2] * xin.shape[3])).expand_as(xin))
            elif op.kind == C.OP_POSADD:
                if V is None and want_G:
                    T = self.prog.seq_len
                    Gp = torch.zeros_like(self.P[op.w])
                    Gp[:T] = dout.flatten(1).view(-1, T, dout.shape[1]).sum(dim=0)
                    G[op.w] = Gp
                add(op.tin, dout)
            elif op.kind == C.OP_LAYERNORM:
                xh, inv = self.aux[i]
                gam = self.P[op.gamma]
                if V is None:
                    dx, Gg, Gb, t_, u_ = TI._ln_backward(dout.flatten(1)[None], xh[None], inv[None], gam)
                    self.rsave[i] = (dout.flatten(1), t_[0], u_[0])
                    if want_G:
                        G[op.gamma], G[op.beta] = Gg, Gb
                    add(op.tin, dx[0].view_as(xin))
                else:
                    dyB, t_, u_ = self.rsave[i]
                    xd, xhd = self.ta[op.tin].flatten(1), self.taux[i]
                    dxd = TI._ln_tangent_backward(dout.flatten(1), dyB, t_, u_, xd, xh, xhd, inv, gam, V[op.gamma])
                    add(op.tin, dxd.view_as(xin))
            elif op.kind == C.OP_ATTENTION:
                Q, K, Vv, P_ = self.aux[i]
                T, sc = self.prog.seq_len, 1.0 / (Q.shape[-1] ** 0.5)
                dO = dout.flatten(1).view(-1, T, op.R, Q.shape[-1]).transpose(1, 2)
                if V is None:
                    dV = P_.transpose(-1, -2) @ dO
                    dP = dO @ Vv.transpose(-1, -2)
                    r = (dP * P_).sum(dim=-1, keepdim=True)
                    dS = P_ * (dP - r)
                    dQ, dK = dS @ K * sc, dS.transpose(-1, -2) @ Q * sc
                    self.rsave[i] = (dO, dP, r, dS)
                else:
                    dOB, dP, r, dS = self.rsave[i]
                    Qd, Kd, Vd, Pd = self.taux[i]
                    dV = Pd.transpose(-1, -2) @ dOB + P_.transpose(-1, -2) @ dO
                    dPd = dO @ Vv.transpose(-1, -2) + dOB @ Vd.transpose(-1, -2)
                    rd = (dPd * P_ + dP * Pd).sum(dim=-1, keepdim=True)
                    dSd = Pd * (dP - r) + P_ * (dPd - rd)
                    dQ = (dSd @ K + dS @ Kd) * sc
                    dK = (dSd.transpose(-1, -2) @ Q + dS.transpose(-1, -2) @ Qd) * sc
                m = lambda u: u.transpose(1, 2).reshape(xin.shape[0], -1)  # noqa: E731
                add(op.tin, torch.cat([m(dQ), m(dK), m(dV)], dim=1).view_as(xin))
            elif op.kind == C.OP_LINEAR:
                do2 = dout.view(dout.shape[0], -1)
                xf = self._flat_in(op, xin)
                if V is None:
                    if want_G:
                        G[op.w] = do2.t() @ xf
                        if op.b >= 0:
                            G[op.b] = do2.sum(dim=0)
                    add(op.tin, (do2 @ self.P[op.w]).view_as(xin))
                else:
                    dprev2 = d_prev[op.tout].view(dout.shape[0], -1)
                    add(op.tin, (do2 @ self.P[op.w] + dprev2 @ V[op.w]).view_as(xin))
        return d, G, du_saved

    def backward(self, want_dx=False):
        n = self.p.shape[0]
        if getattr(self.prog, "seq_len", 0):
            seed = (self.p - self.onehot) * self.row_keep / self.M
            d, G, du = self._reverse(seed, want_dx=True)
            self.d_B, self.du_B, self.G = d, du, G
            return G
        seed = (self.p - self.onehot) / n
        d, G, du = self._reverse(seed, want_dx=want_dx)
        self.d_B, self.du_B, self.G = d, du, G
        return G

    def tangent_forward(self, V):
        prog = self.prog
        ta = {0: None}  # tangent of the candidate is zero
        self.taux = {}
        for i, op in enumerate(prog.ops):
            tin, xin = ta[op.tin], self.a[op.tin]
            if op.kind == C.OP_CONV:
                out = F.conv2d(xin, V[op.w], None if op.b < 0 else V[op.b], stride=op.stride, padding=op.pad)
                if tin is not None:
                    out = out + F.conv2d(tin, self.P[op.w], None, stride=op.stride, padding=op.pad)
                ta[op.tout] = out
            elif op.kind == C.OP_BNACT:
                u = tin if tin is not None else torch.zeros_like(xin)
                if op.has_bn and getattr(op, "bn_train", False):
                    #   TF:  xh' = inv (x' - m(x') - xh m(xh x'));   y' = v_gamma xh + gamma xh' + v_beta
                    xh, inv = self.aux[i], self.aux[("inv", i)]
                    m = lambda t: t.mean(dim=(0, 2, 3), keepdim=True)  # noqa: E731
                    xhd = inv * (u - m(u) - xh * m(xh * u))
                    self.taux[i] = xhd
                    ta[op.tin] = u
                    u = V[op.gamma].view(1, -1, 1, 1) * xh + self.P[op.gamma].view(1, -1, 1, 1) * xhd + V[op.beta].view(1, -1, 1, 1)
                elif op.has_bn:
                    rm, inv = self._bn_consts(i, op)
                    u = self.P[op.gamma].view(1, -1, 1, 1) * inv * u + V[op.gamma].view(1, -1, 1, 1) * self.aux[i] \
                        + V[op.beta].view(1, -1, 1, 1)
                if op.res >= 0 and ta[op.res] is not None:
                    u = u + ta[op.res]
                ta[op.tout] = u * (self.a[op.tout] > 0).to(self.dtype) if op.relu else u
            elif op.kind == C.OP_MAXPOOL:
                idx = self.aux[i]
                ta[op.tout] = tin.flatten(2).gather(2, idx.flatten(2)).view_as(idx).to(self.dtype)
            elif op.kind == C.OP_AVGPOOL:
                ta[op.tout] = tin.mean(dim=(2, 3), keepdim=True)
            elif op.kind == C.OP_LINEAR:
                out = F.linear(self._flat_in(op, xin), V[op.w], None if op.b < 0 else V[op.b])
                if tin is not None:
                    out = out + F.linear(self._flat_in(op, tin), self.P[op.w])
                ta[op.tout] = out.view(xin.shape[0], -1, 1, 1)
            elif op.kind == C.OP_POSADD:
                ta[op.tout] = self._pos_rows(V[op.w], xin.shape[0], self.prog.seq_len)
            elif op.kind == C.OP_LAYERNORM:
                xh, inv = self.aux[i]
                yd, xhd = TI._ln_tangent_forward(tin.flatten(1), xh, inv, self.P[op.gamma], V[op.gamma], V[op.beta])
                ta[op.tout], self.taux[i] = yd.view_as(xin), xhd
            elif op.kind == C.OP_ATTENTION:
                Q, K, Vv, P_ = self.aux[i]
                T, sc = self.prog.seq_len, 1.0 / (Q.shape[-1] ** 0.5)
                Qd, Kd, Vd = self._split_heads(tin, op.R, T)
                Sd = (Qd @ K.transpose(-1, -2) + Q @ Kd.transpose(-1, -2)) * sc
                Pd = P_ * (Sd - (P_ * Sd).sum(dim=-1, keepdim=True))
                ta[op.tout], self.taux[i] = self._merge_heads(Pd @ Vv + P_ @ Vd), (Qd, Kd, Vd, Pd)
        self.ta = ta
        return ta

    def tangent_backward(self, V, inject=None):
        n = self.p.shape[0]
        zdot = self.ta[self.prog.logits].view(n, -1)
        p = self.p
        if getattr(self.prog, "seq_len", 0):
            T = self.prog.seq_len
            centred = (zdot - (p * zdot).sum(dim=1, keepdim=True)) * self.row_keep
            seed = p * centred / self.M
            d, _, _ = self._reverse(seed, V=V, d_prev=self.d_B, inject=inject)
            self.d_TB = d
            # d objective / d (target probabilities): row (b, t) receives the term of the logits row (b, t - 1)
            dq = torch.zeros_like(centred)
            dq[1:] = -centred[:-1] / self.M
            self.dq = dq.view(n // T, T, -1)
            return d[0].flatten(1).view(n // T, T, -1)
        seed = (p * zdot - p * (p * zdot).sum(dim=1, keepdim=True)) / n
        d, _, _ = self._reverse(seed, V=V, d_prev=self.d_B, inject=inject)
        self.d_TB = d
        return d[0]

    # ------------------------------------------------------------------ regulariser adjoints
    def deep_inversion(self, scale, first_bn_multiplier=10):
        """Value and adjoints (w.r.t. each BN input tensor) of the DeepInversion prior
        (regularizers.py:222-227 + deepinversion.py:93-103)."""
        value, inject, first = 0.0, {}, True
        for i, op in enumerate(self.prog.ops):
            if op.kind != C.OP_BNACT or not op.has_bn:
                continue
            z = self.a[op.tin]
            rm, rv = self.bn[i]
            M = z.shape[0] * z.shape[2] * z.shape[3]
            mean = z.mean(dim=(0, 2, 3))
            var = z.var(dim=(0, 2, 3), unbiased=False)
            nv, nm = torch.norm(rv - var, 2), torch.norm(rm - mean, 2)
            mult = scale * (first_bn_multiplier if first else 1.0)
            first = False
            value = value + mult * (nv + nm)
            cm = (mean - rm) / nm / M
            cv = (var - rv) / nv * 2.0 / M
            adj = mult * (cm.view(1, -1, 1, 1) + cv.view(1, -1, 1, 1) * (z - mean.view(1, -1, 1, 1)))
            inject[op.tin] = inject.get(op.tin, 0) + adj
        return value, inject

    def feature_regularization(self, measured, scale):
        """regularizers.py:53-57: mean squared distance of the last linear layer's input to ``measured``."""
        lin = [op for op in self.prog.ops if op.kind == C.OP_LINEAR][-1]
        feat = self.a[lin.tin]
        f2 = feat.reshape(feat.shape[0], -1)
        diff = f2 - measured.to(self.dtype)
        value = diff.pow(2).mean() * scale
        return value, {lin.tin: (2.0 * scale / diff.numel() * diff).view_as(feat)}

    # ------------------------------------------------------------------ whole objective gradient
    def matching_gradient(self, x, labels, g, kind, scale=1.0, task_regularization=0.0, inject_fn=None, **kw):
        """Return (Phi_match (+task term), dPhi/dx, task_loss, G) via the four sweeps."""
        loss = self.forward(x, labels)
        G = self.backward(want_dx=task_regularization != 0)
        gg = [t.to(self.dtype) for t in g]
        val, V = objective_direction(kind, G, gg, scale=scale, **kw)
        self.tangent_forward(V)
        inject = inject_fn(self) if inject_fn is not None else None
        dx = self.tangent_backward(V, inject)
        if task_regularization != 0:
            val = val + task_regularization * loss
            dx = dx + task_regularization * self.d_B[0]
        return val, dx, loss, G


def _maxpool_scatter(dout, idx, in_shape):
    """Adjoint of max-pooling with overlapping windows: scatter-add by argmax index."""
    N, Cc, H, W = in_shape
    out = torch.zeros(N, Cc, H * W, dtype=dout.dtype)
    out.scatter_add_(2, idx.flatten(2), dout.flatten(2))
    return out.view(N, Cc, H, W)
