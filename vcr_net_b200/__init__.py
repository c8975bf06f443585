"""vcr_net_b200 -- B200-native (sm_100a) drop-in for VCR-Net's registration inference path.

Same class / function names as the reference's ``model`` and ``util`` packages
(VCRNet, LPDNet, LPD, Transformer, VcpTopK, SVDHead, vcrnetIter, knn, get_graph_feature,
farthest_point_sample, transform_point_cloud, quat2mat); the compute runs in hand-written
CUDA kernels behind the C ABI of include/vcr_b200.h.  There is no CPU fallback.
"""
from .model.lpdnet_model import LPD, LPDNet, TranformNet  # noqa: F401
from .model.icp_model import ICP  # noqa: F401
from .model.transformer import Transformer  # noqa: F401
from .model.vcrnet_model import (DGCNN, PointNet, SVDHead, VcpAtt, VcpByDis, VcpTopK, VCRNet,  # noqa: F401
                                 vcrnetIcpNet, vcrnetIter, vcrnetIterRagged,
                                 vcrnetIterRaggedPartial)
from .util.util import (farthest_point_sample, get_graph_feature, knn, quat2mat,  # noqa: F401
                        transform_point_cloud)

__all__ = ["VCRNet", "LPDNet", "LPD", "DGCNN", "PointNet", "VcpAtt", "VcpByDis", "Transformer", "VcpTopK", "SVDHead", "vcrnetIter", "vcrnetIterRagged", "vcrnetIterRaggedPartial", "vcrnetIcpNet", "ICP", "knn",
           "get_graph_feature", "farthest_point_sample", "transform_point_cloud", "quat2mat"]
