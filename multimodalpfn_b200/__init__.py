"""mmpfn-b200: sm_100a implementation of MMPFN's in-context inference hot path.

Importing the package does not need a GPU; constructing a model or classifier does.
"""
from .synth import Geometry  # noqa: F401

__all__ = ["Geometry", "MMPFNClassifier", "MMPFNRegressor", "B200PerFeatureTransformer", "B200InferenceEngine"]


def __getattr__(name):
    if name == "MMPFNClassifier":
        from .classifier import MMPFNClassifier
        return MMPFNClassifier
    if name == "MMPFNRegressor":
        from .regressor import MMPFNRegressor
        return MMPFNRegressor
    if name == "B200PerFeatureTransformer":
        from .model import B200PerFeatureTransformer
        return B200PerFeatureTransformer
    if name == "B200InferenceEngine":
        from .engine import B200InferenceEngine
        return B200InferenceEngine
    raise AttributeError(name)
