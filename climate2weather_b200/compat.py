"""Makes the reference's import paths resolve to this package, so `exp/downscaling.py` / `training_loop.py` and
pickled snapshots (training_loop.py:250-266: util.EasyDict{"ema": model.score.ScoreUNet (fp16), "pipeline":
thor.pipelines.SDAPipeline, "dataset_kwargs": ...}) work unchanged:

    import climate2weather_b200.compat as compat; compat.install()
    import thor.score, thor.pipelines, model.score        # -> this package
    snapshot = pickle.load(open("network-snapshot-....pkl", "rb"))   # ema is a climate2weather_b200.ScoreUNet

Pickle resolves classes by qualified name.  The snapshot's `ema` carries the reference's whole module tree
(`model.nn.UNet`, `ModResidualBlock`, `AttentionBlock`, `QKVAttention`, `zuko.nn.LayerNorm`, `torch.nn.*`): those names are
bound to parameter-holding stand-ins (their arithmetic lives in the CUDA library), and `ScoreUNet.__setstate__` rebuilds
the architecture description from the parameter names and shapes.
"""
from __future__ import annotations

import sys
import types

import torch

from . import model as _model
from . import pipelines as _pipelines
from . import score as _score


class EasyDict(dict):
    """util.EasyDict of the reference (util.py:36-49): a dict with attribute access."""

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    def __setattr__(self, name, value):
        self[name] = value

    def __delattr__(self, name):
        del self[name]


def _holder(name: str, module: str, base=torch.nn.Module):
    """A parameter container standing in for a reference module class when unpickling."""
    cls = type(name, (base,), {"__doc__": f"stand-in for the reference's {module}.{name} (state only; no forward)",
                               "forward": lambda self, *a, **k: (_ for _ in ()).throw(
                                   NotImplementedError(f"{module}.{name} is a state holder; call the ScoreUNet"))})
    cls.__module__ = module
    return cls


def install(force: bool = False) -> None:
    def mod(name: str, **attrs) -> types.ModuleType:
        if name in sys.modules and not force:
            m = sys.modules[name]
        else:
            m = types.ModuleType(name)
            sys.modules[name] = m
        for k, v in attrs.items():
            if force or not hasattr(m, k):
                setattr(m, k, v)
        return m

    thor = mod("thor")
    thor.score = mod("thor.score", AbstractScoreFunction=_score.AbstractScoreFunction,
                     DefaultScoreFunction=_score.DefaultScoreFunction,
                     BatchedScoreFunction=_score.BatchedScoreFunction, CoarseGrain=_score.CoarseGrain,
                     PointObservation=_score.PointObservation)
    thor.pipelines = mod("thor.pipelines", SDAPipeline=_pipelines.SDAPipeline)
    m = mod("model")
    m.score = mod("model.score", ScoreUNet=_model.ScoreUNet)
    m.nn = mod("model.nn", UNet=_holder("UNet", "model.nn"), ModResidualBlock=_holder("ModResidualBlock", "model.nn"),
               AttentionBlock=_holder("AttentionBlock", "model.nn"), QKVAttention=_holder("QKVAttention", "model.nn"),
               ResidualBlock=_holder("ResidualBlock", "model.nn", torch.nn.Sequential))
    zuko = mod("zuko")
    zuko.nn = mod("zuko.nn", LayerNorm=_holder("LayerNorm", "zuko.nn"))
    mod("util", EasyDict=EasyDict)
