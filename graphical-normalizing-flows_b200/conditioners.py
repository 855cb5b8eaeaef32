"""Conditioner plugins with the reference's class names, constructor signatures, attributes and
state_dict keys (models/Conditionners/*.py), rebinding ``forward`` to the sm_100a kernels."""
import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from . import ops


class Conditioner(nn.Module):
    """Plugin ABC (models/Conditionners/Conditioner.py:4-23): forward(x [B,d], context) -> h [B,d,H]."""

    def __init__(self):
        super().__init__()
        self.is_invertible = True

    def forward(self, x, context=None):
        pass

    def depth(self):
        pass


def _linear_stack(sizes):
    layers = []
    for h1, h2 in zip(sizes[:-1], sizes[1:]):
        layers += [nn.Linear(h1, h2), nn.ReLU()]
    layers.pop()
    return nn.Sequential(*layers)


def _check_context(context, B, cond_in, who):
    """A conditional conditioner's context: [B, cond_in], CUDA, fp32, contiguous (ValueError for a missing or misshapen one,
    TypeError for the rest, like every op)."""
    if context is None:
        raise ValueError(f"{who}: built with cond_in={cond_in}, forward needs a [B, {cond_in}] context")
    L.require(context, "context")
    if tuple(context.shape) != (B, cond_in):
        raise ValueError(f"{who}: context must be [B, cond_in] = [{B}, {cond_in}], got {tuple(context.shape)}")
    return context


def _stack_params(net):
    """[W0, b0, W1, b1, ...] of the nn.Linear members of an nn.Sequential, rejecting anything that the
    fused kernels do not implement (only Linear/ReLU alternation)."""
    params = []
    mods = list(net)
    for i, m in enumerate(mods):
        if i % 2 == 0:
            if not isinstance(m, nn.Linear) or m.bias is None:
                raise NotImplementedError("fused MLP engine supports nn.Linear(bias=True)/nn.ReLU stacks only")
            params += [m.weight, m.bias]
        elif not isinstance(m, nn.ReLU):
            raise NotImplementedError("fused MLP engine supports nn.Linear/nn.ReLU stacks only")
    return params


class DAGMLP(nn.Module):
    """Parameter container + engine entry for DAGConditioner's embedding net (DAGConditioner.py:7-20)."""

    def __init__(self, in_size, hidden, out_size, cond_in=0):
        super().__init__()
        self.net = _linear_stack([in_size + cond_in] + list(hidden) + [out_size])

    def forward(self, x):
        return ops.MlpFn.apply(x.contiguous(), x.shape[1], *_stack_params(self.net))


class DAGConditioner(Conditioner):
    """models/Conditionners/DAGConditioner.py:23-293."""

    def __init__(self, in_size, hidden, out_size, cond_in=0, soft_thresholding=True, h_thresh=0., gumble_T=1.,
                 hot_encoding=False, l1=0., nb_epoch_update=1, A_prior=None):
        super().__init__()
        if A_prior is None:
            self.A = nn.Parameter(torch.ones(in_size, in_size) * 1.5 + torch.randn((in_size, in_size)) * .02)
        else:
            self.A = nn.Parameter(A_prior)
        self.in_size = in_size
        self.exponent = self.in_size % 50                    # quirk Q1: d % 50, kept for parity
        self.s_thresh = soft_thresholding
        self.h_thresh = h_thresh
        self.stoch_gate = True
        self.noise_gate = False
        in_net = in_size * 2 if hot_encoding else in_size
        self.cond_in = cond_in
        self._module_embedding = isinstance(hidden, nn.Module)
        if self._module_embedding:
            # an arbitrary embedding module (the reference's image flows pass MNISTCNN / CIFAR10CNN, DAGConditioner.py:38-39):
            # the gated, masked copies e[b,i,:] = x[b,:] * G[b,i,:] are produced by the fused DAG layer-1 kernels run with an
            # identity "first layer" (exact in fp32: one product by 1 plus zeros), then handed to the module as the reference does
            self.embedding_net = hidden
            self.register_buffer("_expand_weight", torch.eye(in_size), persistent=False)
            self.register_buffer("_expand_bias", torch.zeros(in_size), persistent=False)
        else:
            self.embedding_net = DAGMLP(in_net, hidden, out_size, cond_in)
        self.gumble = True
        self.hutchinson = False
        self.gumble_T = gumble_T
        self.hot_encoding = hot_encoding
        with torch.no_grad():
            self.constrainA(h_thresh)
        self.register_buffer("lambd", torch.tensor(.0))
        self.register_buffer("c", torch.tensor(1e-3))
        self.register_buffer("eta", torch.tensor(10.))
        self.register_buffer("gamma", torch.tensor(.9))
        self.register_buffer("l1_weight", torch.tensor(l1))
        self.register_buffer("dag_const", torch.tensor(1.))
        self.alpha_factor = 1.
        self.d = in_size
        self.tol = 1e-30
        self.register_buffer("alpha", self.getAlpha())
        self.register_buffer("prev_trace", self._power_trace_host())
        self.nb_epoch_update = nb_epoch_update
        self.no_update = 0
        self.is_invertible = False
        # Philox stream of the in-kernel Gumbel / Gaussian gate noise (replaces the reference's torch.rand calls)
        self._noise_seed = None
        self._noise_calls = 0
        self._noise_rank = 0
        self._replay_noise = None       # tests: tuple of [B,d,d] tensors replaying the reference's draws once
        self._noise_counter = None      # device int64 counter used instead of the host call count (CUDA graphs)

    # ---- small host helpers -------------------------------------------------------------------
    def getAlpha(self):
        return torch.tensor(1. / self.in_size)               # quirk Q2: the reference discards its SVD

    def get_dag(self):
        return self

    def _power_trace_host(self):
        """Constructor-time value of prev_trace on whatever device A lives on (CPU at construction: plain
        torch, init only — the per-step evaluations go through the K2 kernel)."""
        with torch.no_grad():
            if self.A.is_cuda or L._SIMULATOR:
                return self.get_power_trace().detach().clone()
            Bm = torch.eye(self.in_size) + min(1., 1. / self.in_size) * self.A.detach() ** 2
            return torch.diag(torch.matrix_power(Bm, self.exponent)).sum() - self.in_size

    def soft_thresholded_A(self):
        return 2 * (torch.sigmoid(2 * (self.A ** 2)) - .5)

    def hard_thresholded_A(self):
        if self.s_thresh:
            return self.soft_thresholded_A() * (self.soft_thresholded_A() > self.h_thresh).float()
        return self.A ** 2 * (self.A ** 2 > self.h_thresh).float()

    def constrainA(self, zero_threshold=.0001):
        self.A *= (self.A.clone().abs() > zero_threshold).float()
        self.A *= 1. - torch.eye(self.in_size, device=self.A.device)
        return

    # ---- hot path --------------------------------------------------------------------------------
    def _gate_spec(self, x):
        """Map the mutable Python flags onto (importance table, gate mode) — DAGConditioner.py:126-153."""
        if self.h_thresh > 0:
            imp = L.IMP_HARD_SOFT if self.s_thresh else L.IMP_HARD_SQ
        elif self.s_thresh:
            imp = L.IMP_SOFT
        else:
            return ops.GateSpec(L.GATE_TABLE, L.IMP_RAW)
        if self.stoch_gate:
            if not self.gumble:
                raise NotImplementedError("non-Gumbel stochastic gate (dead code in the reference) is not implemented")
            mode = L.GATE_GUMBEL
        elif self.noise_gate:
            mode = L.GATE_NOISER
        else:
            return ops.GateSpec(L.GATE_TABLE, imp, self.h_thresh)
        noise = self._replay_noise
        self._replay_noise = None
        if noise is not None:
            return ops.GateSpec(mode, imp, self.h_thresh, self.gumble_T, noise=tuple(noise))
        if self._noise_seed is None:
            self._noise_seed = int(torch.randint(0, 2 ** 62, (1,)).item())   # follows torch.manual_seed
        if self._noise_counter is not None:
            # graph-capturable: the Philox offset lives on the device.  Inside a capture the captured step bumps it itself and
            # its forward and backward replay together.  An EAGER call made after a graph was built draws fresh noise (bump)
            # and freezes the offset it used in a private scalar, so that its backward regenerates the same noise even if a
            # graph replay moves the shared counter in between.
            cnt = self._noise_counter
            if not torch.cuda.is_current_stream_capturing():
                ops.counter_add(cnt, 1)
                cnt = cnt.clone()
            return ops.GateSpec(mode, imp, self.h_thresh, self.gumble_T, seed=self._noise_seed,
                                offset=(self._noise_rank << 40), offset_dev=cnt)
        self._noise_calls += 1
        return ops.GateSpec(mode, imp, self.h_thresh, self.gumble_T, seed=self._noise_seed,
                            offset=(self._noise_rank << 40) + self._noise_calls)

    def forward(self, x, context=None):
        """h [B, d, H].  With cond_in = c > 0, context [B, c] joins layer 1's input: the row for sample b, variable i is
        [e[b,i,:] | onehot(i) (hot_encoding) | context[b,:]], the in_net + cond_in columns DAGMLP's first Linear is built with
        (see ops.DagMlpFn).  With cond_in = 0, or an nn.Module embedding, a context is accepted and ignored like the reference
        (quirk Q8)."""
        if self.cond_in > 0 and not self._module_embedding:
            _check_context(context, x.shape[0], self.cond_in, "DAGConditioner")
        gate = self._gate_spec(x)
        self._last_gate = gate          # lets tests dump the Philox draws this forward used
        if self._module_embedding:
            B, d = x.shape
            e = ops.DagMlpFn.apply(x.contiguous(), self.A, gate, False, self._expand_weight, self._expand_bias).reshape(B * d, d)
            if self.hot_encoding:       # DAGConditioner.py:155-166: the one-hot block goes in front of the embedding net
                e = torch.cat((e, torch.eye(d, device=e.device, dtype=e.dtype).repeat(B, 1)), 1)
            return self.embedding_net(e).view(B, d, -1)
        params = _stack_params(self.embedding_net.net)
        if self.cond_in > 0:
            params.append(context)
        return ops.DagMlpFn.apply(x.contiguous(), self.A, gate, self.hot_encoding, *params)

    def _alpha_host(self):
        # alpha is a registered buffer (checkpoint compatibility) but only ever holds 1/d; cache its host value
        # so that the per-step loss does not pay a device->host sync.
        key = (self.alpha.data_ptr(), self.alpha._version)
        if getattr(self, "_alpha_key", None) != key:
            self._alpha_key, self._alpha_val = key, float(self.alpha)
        return self._alpha_val

    def get_power_trace(self):
        alpha = min(1., self._alpha_host()) * self.alpha_factor
        if self.hutchinson != 0:
            raise NotImplementedError("Hutchinson trace estimator (disabled in the reference) is not implemented")
        return ops.PowerTraceFn.apply(self.A, alpha, int(self.exponent))

    def loss(self):
        lag_const = self.get_power_trace()
        duals = (self.lambd, self.c, self.dag_const, self.l1_weight)
        if all(torch.is_tensor(v) and v.dtype == torch.float32 and v.device == self.A.device and v.numel() == 1 for v in duals):
            return ops.DagLossFn.apply(self.A, lag_const, *duals)
        # a driver replaced a dual variable by something else than a one-element fp32 device tensor: the reference's formula
        return self.dag_const * (self.lambd * lag_const + self.c / 2 * lag_const ** 2) + self.l1_weight * self.A.abs().mean()

    # ---- dual-ascent control logic (host side; SURVEY.md §8f rank 1) -----------------------------
    def _adjacency(self, M):
        return (M.detach().abs() > 0).cpu().numpy()

    @staticmethod
    def _is_dag(adj):
        """Kahn topological sort on a boolean adjacency matrix (replaces networkx.is_directed_acyclic_graph)."""
        adj = np.array(adj, dtype=bool)
        n = adj.shape[0]
        indeg = adj.sum(0).astype(np.int64)
        stack = [i for i in range(n) if indeg[i] == 0]
        seen = 0
        while stack:
            u = stack.pop()
            seen += 1
            for v in np.nonzero(adj[u])[0]:
                indeg[v] -= 1
                if indeg[v] == 0:
                    stack.append(int(v))
        return seen == n

    @staticmethod
    def _longest_path(adj):
        adj = np.array(adj, dtype=bool)
        n = adj.shape[0]
        indeg = adj.sum(0).astype(np.int64)
        order, stack = [], [i for i in range(n) if indeg[i] == 0]
        while stack:
            u = stack.pop()
            order.append(u)
            for v in np.nonzero(adj[u])[0]:
                indeg[v] -= 1
                if indeg[v] == 0:
                    stack.append(int(v))
        dist = np.zeros(n, dtype=np.int64)
        for u in order:
            for v in np.nonzero(adj[u])[0]:
                dist[v] = max(dist[v], dist[u] + 1)
        return int(dist.max()) if n else 0

    def post_process(self, zero_threshold=None):
        """DAGConditioner.py:76-92 — threshold A to a binary DAG and switch to the deterministic branch."""
        with torch.no_grad():
            soft = self.soft_thresholded_A().detach().abs()
            if zero_threshold is None:
                zero_threshold = .1
                while not self._is_dag(self._adjacency((soft > zero_threshold).float())):
                    zero_threshold += .05
            self.stoch_gate = False
            self.noise_gate = False
            self.s_thresh = False
            self.h_thresh = 0.
            self.A.data.copy_((soft > zero_threshold).float())        # in place: A keeps its storage (captured graphs, optimizers)
            self.A *= 1. - torch.eye(self.in_size, device=self.A.device)
        self.A.requires_grad = False
        self.A.grad = None

    def depth(self):
        adj = self._adjacency((self.A.detach() > 0).float())
        if self.is_invertible or self._is_dag(adj):
            return self._longest_path(adj)
        return 0

    def _set_scalar(self, name, value):
        """In-place update of a one-element dual buffer: the device pointer stays valid for captured CUDA graphs and for the
        fused loss kernel (the reference rebinds the attribute to a fresh tensor; the value semantics are the same)."""
        buf = getattr(self, name)
        value = torch.as_tensor(value, dtype=buf.dtype, device=buf.device).reshape(buf.shape)
        buf.copy_(value)

    def graph_state(self):
        """Everything a captured step froze at capture time: host-side flags, the power-trace exponent, and the identity /
        address of A and of the dual buffers.  Graphed*Step compares it on every call and recaptures on change."""
        return (int(self.exponent), bool(self.s_thresh), float(self.h_thresh), bool(self.stoch_gate), bool(self.noise_gate),
                float(self.gumble_T), bool(self.hot_encoding), float(self.alpha_factor), self._alpha_host(), id(self.A),
                self.A.data_ptr(), bool(self.A.requires_grad), self.lambd.data_ptr(), self.c.data_ptr(),
                self.dag_const.data_ptr(), self.l1_weight.data_ptr())

    def update_dual_param(self):
        """Augmented-Lagrangian update (DAGConditioner.py:196-260).  The dual buffers are updated in place (stable device
        pointers); `self.A = nn.Parameter(A_before)` is kept as the reference has it -- a NEW Parameter object, which, exactly
        as in the reference, is no longer known to an optimizer built earlier."""
        with torch.no_grad():
            lag_const = self.get_power_trace()
            while self.dag_const > 0. and lag_const < self.tol and self.exponent < self.in_size:
                self.exponent += 50
                lag_const = self.get_power_trace()
            if self.dag_const > 0. and lag_const > self.tol:
                self._set_scalar("lambd", self.lambd + self.c * lag_const)
                if lag_const.abs() > self.gamma * self.prev_trace.abs():
                    self.c *= self.eta
                self._set_scalar("prev_trace", lag_const)
            elif self.dag_const > 0.:
                A_before = self.A.clone()
                self.post_process()
                self._set_scalar("alpha", self.getAlpha())
                lag_const = self.get_power_trace()
                if lag_const > 0.:
                    self.stoch_gate, self.noise_gate, self.s_thresh, self.h_thresh = True, False, True, 0.
                    self.A = nn.Parameter(A_before)
                    self.A.requires_grad = True
                    self.A.grad = self.A.clone()
                    self._set_scalar("alpha", self.getAlpha())
                    self._set_scalar("prev_trace", self.get_power_trace())
                    self.c *= 1 / self.eta
                    self._set_scalar("lambd", self.lambd + self.c * lag_const)
                    self._set_scalar("dag_const", 1.)
                else:
                    self._set_scalar("dag_const", 0.)
                    self._set_scalar("l1_weight", 0.)
            else:
                if not self._is_dag(self._adjacency(self.A.detach() ** 2)):
                    self.A.requires_grad = True
                    self.A.grad = self.A.clone()
                    self.stoch_gate, self.noise_gate, self.s_thresh, self.h_thresh = True, False, True, 0.
                    self._set_scalar("alpha", self.getAlpha())
                    self._set_scalar("prev_trace", self.get_power_trace())
                    self._set_scalar("dag_const", 1.)
                else:
                    self.is_invertible = True
        return lag_const

    def step(self, epoch_number, loss_avg=0.):
        """DAGConditioner.py:273-293 (without the reference's debug prints)."""
        with torch.no_grad():
            lag_const = self.get_power_trace()
            if lag_const > 50:
                self.exponent -= 5
                self.exponent = self.exponent if self.exponent > 3 else 3
            if epoch_number % self.nb_epoch_update == 0 and epoch_number > 0:
                loss_avg = torch.as_tensor(loss_avg)
                if self.loss().abs() < loss_avg.abs() / 2 or self.no_update > 10:
                    self.update_dual_param()
                    self.no_update = 0
                else:
                    self.no_update += 1


# ------------------------------------------------------------------------------------------------
# Autoregressive (MADE)
# ------------------------------------------------------------------------------------------------
class MaskedLinear(nn.Linear):
    """nn.Linear with a fixed 0/1 mask buffer (AutoregressiveConditioner.py:14-25)."""

    def __init__(self, in_features, out_features, bias=True):
        super().__init__(in_features, out_features, bias)
        self.register_buffer('mask', torch.ones(out_features, in_features))

    def set_mask(self, mask):
        self.mask.data.copy_(torch.from_numpy(mask.astype(np.uint8).T))

    def forward(self, input):
        W = ops.PackRowsFn.apply(self.weight, self.mask, None)
        return ops.MlpFn.apply(input.contiguous(), input.shape[1], W, self.bias)


class MADE(nn.Module):
    """Masked autoencoder, natural ordering (AutoregressiveConditioner.py:28-109)."""

    def __init__(self, nin, hidden_sizes, nout, num_masks=1, natural_ordering=False, random=False, device="cpu"):
        super().__init__()
        if random or num_masks != 1:
            raise NotImplementedError("random / multi-mask MADE is never used by the reference's conditioner")
        self.random, self.nin, self.nout, self.hidden_sizes = random, nin, nout, list(hidden_sizes)
        assert self.nout % self.nin == 0, "nout must be integer multiple of nin"
        net = []
        hs = [nin] + self.hidden_sizes + [nout]
        for h0, h1 in zip(hs, hs[1:]):
            net.extend([MaskedLinear(h0, h1), nn.ReLU()])
        net.pop()
        self.net = nn.Sequential(*net)
        self.natural_ordering, self.num_masks, self.seed = natural_ordering, num_masks, 0
        self.m = {}
        self.update_masks()

    def update_masks(self):
        if self.m and self.num_masks == 1:
            return
        Lh = len(self.hidden_sizes)
        self.m[-1] = np.arange(self.nin)
        for l in range(Lh):
            self.m[l] = np.array([self.nin - 1 - (i % self.nin) for i in range(self.hidden_sizes[l])])
        masks = [self.m[l - 1][:, None] <= self.m[l][None, :] for l in range(Lh)]
        masks.append(self.m[Lh - 1][:, None] < self.m[-1][None, :])
        if self.nout > self.nin:
            k = int(self.nout / self.nin)
            masks[-1] = np.concatenate([masks[-1]] * k, axis=1)
        layers = [l for l in self.net.modules() if isinstance(l, MaskedLinear)]
        for l, m in zip(layers, masks):
            l.set_mask(m)
        self.i_map = self.m[-1].copy()
        for k in range(len(self.m[-1])):
            self.i_map[self.m[-1][k]] = k

    def _packed_params(self, first_row=0):
        """mask*W per layer; the last layer's rows are permuted so that the GEMM writes h[b, i, k] directly
        (MADE.forward's view(B,-1,nin).permute(0,2,1), :108-109) and rows of dims < first_row are dropped
        (ConditionnalMADE's [:, cond_in:, :] slice, :140)."""
        layers = [m for m in self.net if isinstance(m, MaskedLinear)]
        key = (first_row, self.net[0].weight.device)
        if getattr(self, "_perm_key", None) != key:
            k_out = self.nout // self.nin
            i = torch.arange(first_row, self.nin).view(-1, 1)
            k = torch.arange(k_out).view(1, -1)
            self._perm = (k * self.nin + i).reshape(-1).to(torch.int32).to(key[1])
            self._perm_key = key
        params = []
        for li, m in enumerate(layers):
            last = li == len(layers) - 1
            params.append(ops.PackRowsFn.apply(m.weight, m.mask, self._perm if last else None))
            params.append(ops.PackVecFn.apply(m.bias, self._perm) if last else m.bias)
        return params

    def forward(self, x, first_row=0):
        out = ops.MlpFn.apply(x.contiguous(), x.shape[1], *self._packed_params(first_row))
        return out.view(x.shape[0], self.nin - first_row, self.nout // self.nin)


class ConditionnalMADE(MADE):
    """AutoregressiveConditioner.py:115-141."""

    def __init__(self, nin, cond_in, hidden_sizes, nout, num_masks=1, natural_ordering=False, random=False, device="cpu"):
        super().__init__(nin + cond_in, hidden_sizes, nout, num_masks, natural_ordering, random, device)
        self.nin_non_cond = nin
        self.cond_in = cond_in

    def forward(self, x, context):
        inp = torch.cat((context, x), 1) if context is not None else x
        return super().forward(inp, first_row=self.cond_in)


class AutoregressiveConditioner(Conditioner):
    """AutoregressiveConditioner.py:144-154."""

    def __init__(self, in_size, hidden, out_size, cond_in=0):
        super().__init__()
        self.in_size = in_size
        self.masked_autoregressive_net = ConditionnalMADE(in_size, cond_in=cond_in, hidden_sizes=hidden,
                                                          nout=out_size * in_size)

    def forward(self, x, context=None):
        return self.masked_autoregressive_net(x, context)

    def depth(self):
        return self.in_size - 1


# ------------------------------------------------------------------------------------------------
# Coupling
# ------------------------------------------------------------------------------------------------
class CouplingMLP(nn.Module):
    """CouplingConditioner.py:6-18."""

    def __init__(self, in_size, hidden, out_size, cond_in=0):
        super().__init__()
        self.net = _linear_stack([in_size - int(in_size / 2) + cond_in] + list(hidden) + [out_size * int(in_size / 2)])

    def forward(self, x):
        return ops.MlpFn.apply(x.contiguous(), x.shape[1], *_stack_params(self.net))


class _CouplingAssemble(torch.autograd.Function):
    """h = cat(constants broadcast over the batch, h2) (CouplingConditioner.py:33-36)."""

    @staticmethod
    def forward(ctx, constants, h2, B, d, indep, H):
        h = torch.empty(B, d, H, device=h2.device, dtype=h2.dtype)
        ops.broadcast_rows(constants.contiguous(), h, indep)
        h[:, indep:, :] = h2.view(B, d - indep, H)
        ctx.meta = (B, d, indep, H)
        return h

    @staticmethod
    def backward(ctx, gh):
        B, d, indep, H = ctx.meta
        gh = gh.contiguous()
        dT = ops.colsum(gh, H, B * d, H, period=d)          # [d, H] = sum over the batch
        return dT[:indep].contiguous(), gh[:, indep:, :].reshape(B, (d - indep) * H), None, None, None, None


class CouplingConditioner(Conditioner):
    """CouplingConditioner.py:21-39."""

    def __init__(self, in_size, hidden, out_size, cond_in=0):
        super().__init__()
        self.in_size = in_size
        self.out_size = out_size
        self.cond_size = int(in_size / 2)
        self.indep_size = in_size - self.cond_size
        self.cond_in = cond_in
        self.embeding_net = CouplingMLP(in_size, hidden, out_size, cond_in)
        self.constants = nn.Parameter(torch.randn(self.indep_size, out_size))

    def forward(self, x, context=None):
        """With cond_in = c > 0 the embedding net takes cat(x[:, :indep], context) (its indep + cond_in inputs); with c = 0 a
        context is concatenated and sliced away again, like the reference (quirk Q8)."""
        if self.cond_in > 0:
            _check_context(context, x.shape[0], self.cond_in, "CouplingConditioner")
            inp = torch.cat((x[:, :self.indep_size], context), 1)
            h2 = ops.MlpFn.apply(inp, inp.shape[1], *_stack_params(self.embeding_net.net))
            return _CouplingAssemble.apply(self.constants, h2, x.shape[0], self.in_size, self.indep_size, self.out_size)
        if context is not None:
            x = torch.cat((x, context), 1)                  # then sliced away again, like the reference (quirk Q8)
        x = x.contiguous()
        h2 = ops.MlpFn.apply(x, self.indep_size, *_stack_params(self.embeding_net.net))
        return _CouplingAssemble.apply(self.constants, h2, x.shape[0], self.in_size, self.indep_size, self.out_size)

    def depth(self):
        return 1
