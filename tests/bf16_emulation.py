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
