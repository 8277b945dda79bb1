"""climate2weather_b200 — B200-native (sm_100a) guided score-based sampling hot path of Climate2Weather.

Public API mirrors the reference's classes on this path (SURVEY.md §8(b)):
    ScoreUNet                                   <- model.score.ScoreUNet
    DefaultScoreFunction, BatchedScoreFunction  <- thor.score.*            (aliases: MCScoreNet)
    SDAPipeline                                 <- thor.pipelines.SDAPipeline (alias: VPSDE)
    CoarseGrain                                 <- the observation operator of exp/downscaling.py:129-132
    PointObservation                            <- observations at single grid points (stations, masked data)
The arithmetic lives in libc2w_b200.so (csrc/, C ABI in include/c2w_b200.h); importing this package on a machine
without the built library works, calling into the path raises.
"""
from .model import ScoreUNet, build_from_reference
from .pipelines import SDAPipeline
from .score import (AbstractScoreFunction, BatchedScoreFunction, CoarseGrain, DefaultScoreFunction,
                    PointObservation)
from .sharding import ShardPlan, make_plan

# names used by BASELINE.json's north_star (francois-rozet/sda vocabulary) for the same objects
MCScoreNet = DefaultScoreFunction
VPSDE = SDAPipeline

__all__ = ["ScoreUNet", "build_from_reference", "SDAPipeline", "AbstractScoreFunction", "DefaultScoreFunction",
           "BatchedScoreFunction", "CoarseGrain", "PointObservation", "ShardPlan", "make_plan", "MCScoreNet", "VPSDE"]
