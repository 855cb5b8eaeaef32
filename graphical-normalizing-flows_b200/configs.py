"""The five BASELINE.json workload shapes (SURVEY.md App. D) and a builder for each."""
import torch

from .conditioners import AutoregressiveConditioner, CouplingConditioner, DAGConditioner
from .flow import MNIST_A_prior, buildFCNormalizingFlow
from .normalizers import AffineNormalizer, MonotonicNormalizer

CONFIGS = {
    "cfg1": dict(nb_flow=3, d=2, cond="DAG", hidden=[150, 150], out=150, hot_encoding=True, gumble_T=.5, l1=1.,
                 norm="affine"),
    "cfg2": dict(nb_flow=1, d=6, cond="DAG", hidden=[60, 60, 60], out=30, hot_encoding=True, gumble_T=.5, l1=0.,
                 norm="monotonic", int_net=[100, 100, 100], nb_steps=20, solver="CC"),
    "cfg3": dict(nb_flow=1, d=21, cond="Autoregressive", hidden=[210, 210, 210], out=30, norm="monotonic",
                 int_net=[200, 200, 200], nb_steps=20, solver="CCParallel"),
    "cfg4": dict(nb_flow=1, d=63, cond="DAG", hidden=[630, 630, 630], out=30, hot_encoding=True, gumble_T=.5, l1=0.,
                 norm="monotonic", int_net=[150, 150, 150], nb_steps=20, solver="CCParallel"),
    "cfg5": dict(nb_flow=1, d=784, cond="DAG", hidden=[1024, 1024, 1024], out=2, hot_encoding=True, gumble_T=1.,
                 l1=0., norm="affine", A_prior="mnist"),
}

_COND = {"DAG": DAGConditioner, "Autoregressive": AutoregressiveConditioner, "Coupling": CouplingConditioner}


def build_from_spec(spec, device=None, seed=None):
    """buildFCNormalizingFlow(...) for a spec dict (same dict format the oracle uses)."""
    if seed is not None:
        torch.manual_seed(seed)
    cargs = {"in_size": spec["d"], "hidden": list(spec["hidden"]), "out_size": spec["out"]}
    if spec.get("cond_in", 0):
        cargs["cond_in"] = spec["cond_in"]          # conditional flow: every forward takes a [B, cond_in] context
    if spec["cond"] == "DAG":
        cargs.update(l1=spec.get("l1", 0.), gumble_T=spec.get("gumble_T", 1.), nb_epoch_update=10,
                     hot_encoding=spec.get("hot_encoding", False))
        if spec.get("A_prior") == "mnist":
            cargs["A_prior"] = MNIST_A_prior(int(round(spec["d"] ** .5)), 2)
    if spec["norm"] == "monotonic":
        ntype = MonotonicNormalizer
        nargs = {"integrand_net": list(spec["int_net"]), "cond_size": spec["out"], "nb_steps": spec["nb_steps"],
                 "solver": spec.get("solver", "CC")}
    else:
        ntype, nargs = AffineNormalizer, {}
    model = buildFCNormalizingFlow(spec["nb_flow"], _COND[spec["cond"]], cargs, ntype, nargs)
    return model.to(device) if device is not None else model
