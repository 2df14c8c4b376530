"""B200-native (sm_100a) hot path of the EB-NeRD news recommender: the reference's
`models/` nn.Module surface computed by hand-written CUDA kernels behind a C ABI."""
from .models import (MLP, PointwiseAttention, PointwiseAttentionExpanded, UserInstantInterestModel,
                     UserInvariantInterestModel, UserModel)
from .optim import FusedAdam
from .trainer import FusedTrainStep
from ._lib import NrmError, build
from . import dp, explain, metrics, scoring, wire

__all__ = ['MLP', 'PointwiseAttention', 'PointwiseAttentionExpanded', 'UserInstantInterestModel',
           'UserInvariantInterestModel', 'UserModel', 'FusedAdam', 'FusedTrainStep', 'NrmError', 'build', 'dp', 'explain', 'metrics', 'scoring', 'wire']
