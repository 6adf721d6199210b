"""Drop-in counterparts of the reference's `models` package for the episode hot path."""
from .dgcnn import DGCNN, conv1d, conv2d, get_edge_feature, get_graph_feature, knn  # noqa: F401
from .attention import SelfAttention  # noqa: F401
from .mpti import BaseLearner, MPTI_SelfAtten, SupportSet  # noqa: F401
from .protonet import ProtoNet_Contrast  # noqa: F401
