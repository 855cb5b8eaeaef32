"""CUDA-graph capture of a whole training step (zero_grad -> forward -> loss -> backward -> [all-reduce] -> optimizer)
and of the log-likelihood evaluation step.

The step of the small configs is launch-bound (tens of kernels of a few microseconds each): replaying one captured
graph removes the per-launch gaps.  Everything inside the step is already asynchronous on the current stream and
allocation-stable; the one host-side quantity that changed per step, the Philox offset of the DAG gate noise, is moved
to a device counter (gnf_gate_t.offset_dev) that the captured step bumps itself.
"""
import torch

from . import ops


def _device_noise_counters(model, dev):
    """Move every DAG conditioner's Philox offset to a device counter (created once; later graphs share it)."""
    counters = []
    for c in model.getConditioners():
        if hasattr(c, "_noise_counter"):
            if c._noise_seed is None:
                c._noise_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            if c._noise_counter is None:
                c._noise_counter = torch.full((1,), c._noise_calls + 1, dtype=torch.int64, device=dev)
            counters.append(c._noise_counter)
    return counters


def model_graph_state(model):
    """Host-side state a captured step froze (ADVICE r1): conditioner flags / exponents / buffer addresses
    (DAGConditioner.graph_state), quadrature steps and precision of the normalizers, and the engine switches."""
    st = [ops._GEMM_MODE, ops.UMNN_ENGINE, ops.UMNN_FWD_FUSED_TC3]
    for c in model.getConditioners():
        st.append(c.graph_state() if hasattr(c, "graph_state") else None)
    for n in model.getNormalizers():
        st.append((getattr(n, "nb_steps", None), getattr(n, "precision", None), getattr(n, "solver", None)))
    return tuple(st)


def _capture(body, warmup, stream=None):
    """Warm-up runs and the capture on ONE side stream (`stream`, or a fresh one).  A training loop that keeps capturing new graphs
    (one per quadrature-step count, recaptures after model.step()) should pass the stream it runs its eager steps on: autograd
    binds a parameter's gradient accumulator to the stream of the backward that created it, and a capture that has to
    synchronise with another stream for it -- the legacy default stream in particular -- is invalidated."""
    s = stream if stream is not None else torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warmup):
            body()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        out = body()
    return graph, out


class GraphedEvalStep:
    """compute_ll (NormalizingFlow.py:48-50 / UCIExperiments.py:152-162) of a fixed batch shape as one captured graph: the
    evaluation step of the small configs is nine launches of 7-80 us, i.e. launch-bound when issued one by one.
    Returns (ll [B], z [B,d]) -- static tensors overwritten by the next call."""

    def __init__(self, model, example_x, warmup=3):
        self.model, self.warmup = model, warmup
        self.static_x = example_x.clone()
        self.recaptures = 0
        self._capture()

    def _capture(self):
        model = self.model
        self.counters = _device_noise_counters(model, self.static_x.device)

        def body():
            for cnt in self.counters:
                ops.counter_add(cnt, 1)
            with torch.no_grad():
                return model.compute_ll(self.static_x)

        self.graph, self.static_out = _capture(body, self.warmup)
        self.state = model_graph_state(model)

    def __call__(self, x):
        if model_graph_state(self.model) != self.state:      # e.g. model.step() moved an exponent / a gate flag / A
            self.recaptures += 1
            self._capture()
        self.static_x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.static_out


class GraphedTrainStep:
    """One training step as one captured graph.  The capture freezes host-side model state (DAG gate flags, the power-trace
    exponent, quadrature steps, the addresses of A and of the dual buffers): `model.step()` / `update_dual_param()` /
    `post_process()` may change it, so every call compares `model_graph_state` with the captured one and RECAPTURES when it
    differs (`recaptures` counts them).  Note the reference's own quirk: when update_dual_param re-creates A as a new
    Parameter, an optimizer built earlier no longer owns it -- here as there."""

    def __init__(self, model, optimizer, bucket, example_x, allreduce=True, warmup=3, stream=None, side_branch=True):
        self.model, self.opt, self.bucket = model, optimizer, bucket
        has_penalty = any(hasattr(c, "get_power_trace") for c in model.getConditioners())
        self.side = torch.cuda.Stream() if (side_branch and has_penalty and example_x.is_cuda) else None
        if self.side is not None and hasattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch"):
            # A receives one gradient from the side branch (penalty) and one from the main branch (layer 1): intended, and neither
            # stream is the default stream
            torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
        self.static_x = example_x.clone()
        self.allreduce, self.warmup, self.stream = allreduce, warmup, stream
        self.recaptures = 0
        self._capture()

    def _capture(self):
        model, optimizer, bucket, allreduce = self.model, self.opt, self.bucket, self.allreduce
        self.counters = _device_noise_counters(model, self.static_x.device)
        self._one = torch.ones((), device=self.static_x.device, dtype=self.static_x.dtype)

        def body():
            for cnt in self.counters:
                ops.counter_add(cnt, 1)
            bucket.begin_step()
            if self.side is not None:
                # the acyclicity / sparsity penalty depends on A only (a ~40-us chain of one-CTA kernels at d = 63: power trace, loss
                # formula, and their backward): it runs as a parallel branch of the captured step, next to the forward
                cur = torch.cuda.current_stream()
                self.side.wait_stream(cur)
                with torch.cuda.stream(self.side):
                    c = model.constraintsLoss()
                z, jac = model(self.static_x)
                cur.wait_stream(self.side)
                loss = model.loss(z, jac, constraint=c)
            else:
                z, jac = model(self.static_x)
                loss = model.loss(z, jac)
            loss.backward(gradient=self._one)          # a resident cotangent: no ones_like fill launch per step
            if allreduce:
                bucket.finish_step()
            optimizer.step()
            return loss.detach()

        self.graph, self.static_loss = _capture(body, self.warmup, self.stream)
        self.state = model_graph_state(model)

    def __call__(self, x):
        if model_graph_state(self.model) != self.state:
            self.recaptures += 1
            self._capture()
        self.static_x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.static_loss
