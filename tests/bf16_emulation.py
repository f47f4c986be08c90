"""fp64 emulation of the bf16 mode of the GraphSAGE / GCN encoders (csrc/encoder_bf16.cu, DESIGN §3.5 rounding points).

``emulate(encoder_module)`` switches an oracle GraphSAGE / GCN (oracle/scgib_oracle.py) to a forward that rounds to bf16
exactly where the product does, in the forward and - through straight-through rounding functions - in the backward:
  t                      rounded once (stored bf16), its gradient g_t not;
  every aggregation      output rounded; in the backward, the aggregated layer gradient rounded;
  every linear layer     weights rounded as MMA operands; inner outputs rounded, h3 not; in the backward every product
                         g W (the gradient arriving at each linear operand) rounded, and g_out rounded on entry.
With the switch off the forward is the oracle's own, operation for operation (bit-equal: tests/test_encoders_bf16_host.py)."""
import torch
import torch.nn.functional as F

from oracle.scgib_oracle import GCN, GraphSAGE


def _rnd(x):
    return x.to(torch.bfloat16).to(x.dtype)


class _RndF(torch.autograd.Function):
    """forward: round to bf16; backward: identity."""

    @staticmethod
    def forward(ctx, x):
        return _rnd(x)

    @staticmethod
    def backward(ctx, g):
        return g


class _RndB(torch.autograd.Function):
    """forward: identity; backward: round the gradient to bf16."""

    @staticmethod
    def forward(ctx, x):
        return x.clone()

    @staticmethod
    def backward(ctx, g):
        return _rnd(g)


def _ops(on):
    if on:
        return _RndF.apply, _RndB.apply, _RndF.apply
    ident = lambda x: x
    return ident, ident, ident


class EmulatedGraphSAGE(GraphSAGE):
    emulate_bf16 = True

    def forward(self, g, h):
        rf, rb, rw = _ops(self.emulate_bf16)
        h = rf(h)
        deg = None
        convs = (self.conv1, self.conv2, self.conv2)
        for i, c in enumerate(convs):
            if deg is None:
                deg = (g.indptr[1:] - g.indptr[:-1]).to(h.dtype).clamp(min=1)
            neigh = rf(torch.zeros_like(h).index_add(0, g.dst, h[g.src]) / deg[:, None])
            y = F.linear(rb(h), rw(c.fc_self.weight), c.fc_self.bias) + F.linear(rb(neigh), rw(c.fc_neigh.weight))
            if i == len(convs) - 1:
                return rb(y)
            h = rb(rf(F.relu(y)))


class EmulatedGCN(GCN):
    emulate_bf16 = True

    def forward(self, g, h):
        rf, rb, rw = _ops(self.emulate_bf16)
        h = rf(h)
        nrm = None
        convs = (self.conv1, self.conv2, self.conv3)
        for i, c in enumerate(convs):
            if nrm is None:
                nrm = torch.pow((g.indptr[1:] - g.indptr[:-1]).to(h.dtype).clamp(min=1), -0.5)
            hs = h * nrm[:, None]
            a = rf(torch.zeros_like(hs).index_add(0, g.dst, hs[g.src]) * nrm[:, None])
            y = rb(a) @ rw(c.weight) + c.bias
            if i == len(convs) - 1:
                return rb(y)
            h = rb(rf(F.relu(y)))


def emulate(enc, on=True):
    """switch an oracle GraphSAGE / GCN module (in place) to the emulated forward; returns it."""
    enc.__class__ = EmulatedGraphSAGE if isinstance(enc, GraphSAGE) else EmulatedGCN
    enc.emulate_bf16 = on
    return enc


# ------------------------------------------------------------------------------------------------ GIN layer in bf16 mode
def bf16_ulp(x):
    """spacing of bf16 numbers at |x| (8 significant bits); the smallest normal spacing at 0."""
    e = torch.floor(torch.log2(x.abs().clamp(min=2.0 ** -126)))
    return torch.pow(torch.full_like(e, 2.0), e - 7)


def gin_bn_act_terms(h, bn, bf16_mode):
    """The per-row terms f(h) the GIN forward kernels sum, in fp64, and the magnitude each term's fp32 rounding scales with.
    f = relu(BN(.)) with bn = {mean, rstd, gamma, beta} (fp32), or the identity (bn None).  The kernels form the BatchNorm scale
    rstd * gamma in fp32 (csrc/gin_tc3.cu: (h - mean) * scale + beta; csrc/gin_bf16.cu: h * scale + shift, shift = beta -
    mean * scale in fp32); the terms here use the same fp32 constants."""
    h = h.double()
    if bn is None:
        return h, h.abs()
    bn = bn.float()
    mean, rstd, gamma, beta = bn[0], bn[1], bn[2], bn[3]
    sc = rstd * gamma
    if bf16_mode:
        sh = beta - mean * sc
        t = h * sc.double() + sh.double()
        return torch.relu(t), (h * sc.double()).abs() + sh.double().abs()
    d = h - mean.double()
    return torch.relu(d * sc.double() + beta.double()), (d * sc.double()).abs() + beta.double().abs()


def gin_aggregate_ref(terms, src, dst, row_map=None):
    """a_v = f(h_map(v)) + sum_{u in N(v)} f(h_map(u)) (DGL GINConv 'sum', eps = 0) of per-input-row terms."""
    x = terms if row_map is None else terms[row_map]
    return x + torch.zeros_like(x).index_add(0, dst, x[src])


def gin_mlp_ref(a, W1, b1, W2, b2, emulate=True, r=None):
    """r = relu(W1 a + b1) and y = W2 r + b2 in fp64 with the bf16-mode rounding points of csrc/gin_bf16.cu (emulate): both
    weights are MMA operands (rounded), r and y are stored rounded; the accumulation and the biases are exact.  ``r`` given:
    y is computed from it (the kernel's own r).  With emulate False this is MLP (models.py:38-49) operation for operation."""
    rw = _rnd if emulate else (lambda x: x)
    if r is None:
        r = rw(F.relu(F.linear(a, rw(W1), b1)))
    return r, rw(F.linear(r, rw(W2), b2))


def gin_bwd_ref(g_next, src, dst, y, r, a, bn, W1, W2, ga_f32, emulate=True):
    """fp64 backward of one GINConv + BatchNorm(train) + ReLU layer with the rounding points of csrc/gin_bwd_bf16.cu
    (emulate):
      gin_bwd_pre_bf16 : G = g_next (direct mode) or g_next_v + sum_{u in N(v)} g_next_u (CSR mode, src / dst given);
                         g_o = G * [relu(BN(y)) > 0] rounded; d beta = sum g_o, d gamma = sum g_o * yhat of the ROUNDED g_o;
                         c1 = gamma * d beta / V, c2 = gamma * d gamma / V;
      gin_bwd_bf16     : g_y = rstd (gamma g_o - c1 - yhat c2) rounded (the G1 / G3 operand); db2 = sum g_y, dW2 = g_y^T r;
                         g_u = (g_y W2) * [r > 0] rounded (the G2 / G4 operand); db1 = sum g_u, dW1 = g_u^T a;
                         g_a = g_u W1, rounded unless ga_f32;
                         W1, W2 rounded (MMA operands); all accumulation exact.
    The ReLU mask is evaluated as the kernel does, relu(y * scale + shift) > 0 with fp32 scale / shift.  Returns the outputs
    (g_a, dW1, db1, dW2, db2, dgamma, dbeta) and, for each, the magnitude its fp32 accumulation error scales with."""
    rw = _rnd if emulate else (lambda x: x)
    V = y.shape[0]
    G = g_next if src is None else g_next + torch.zeros_like(g_next).index_add(0, dst, g_next[src])
    terms, _ = gin_bn_act_terms(y, bn, True)
    bn64 = bn.double()
    mean, rstd, gamma = bn64[0], bn64[1], bn64[2]
    g_o = rw(G * (terms > 0))
    yhat = (y - mean) * rstd
    dbeta, dgamma = g_o.sum(0), (g_o * yhat).sum(0)
    c1, c2 = gamma * dbeta / V, gamma * dgamma / V
    g_y = rw(rstd * (gamma * g_o - c1 - yhat * c2))
    g_u = rw((g_y @ rw(W2)) * (r > 0))
    g_a = g_u @ rw(W1)
    if not ga_f32:
        g_a = rw(g_a)
    out = (g_a, g_u.t() @ a, g_u.sum(0), g_y.t() @ r, g_y.sum(0), dgamma, dbeta)
    mag = (g_u.abs() @ rw(W1).abs(), g_u.abs().t() @ a.abs(), g_u.abs().sum(0), g_y.abs().t() @ r.abs(), g_y.abs().sum(0),
           (g_o * yhat).abs().sum(0), g_o.abs().sum(0))
    return out, mag
