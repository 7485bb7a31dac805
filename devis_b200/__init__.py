"""devis_b200 -- B200-native (sm_100a) temporal multi-scale deformable attention, the hot path of
acaelles97/DeVIS (src/models/ops), behind the reference's own Python API.

  devis_b200.MultiScaleDeformableAttention   the compiled-module mirror (ms_deform_attn_forward/backward)
  devis_b200.functions.MSDeformAttnFunction  reference signature, reference autograd contract
  devis_b200.functions.TemporalMSDeformAttnFunction   the whole-clip op (one launch per layer-clip)
  devis_b200.modules.*                       MSDeformAttn, TemporalMSDeformAttn{Encoder,Decoder}
  devis_b200.devis_transformer               DeVISTransformer and its encoder / decoder (layers): the direct callers
  devis_b200.clip_geometry                   host-side level / frame tables for the whole-clip op
  devis_b200.GraphedLayer                    CUDA-graph replay (forward + backward) of a layer for fixed shapes
  devis_b200.build                           nvcc recipe for libdevis_msda.so (include/devis_msda.h)
  devis_b200.deform_conv                     deform_conv2d (torchvision's signature) for the mask head

Every op is a torch.library custom op in the ``devis`` namespace (torch.ops.devis.*, registered on import, without
loading the library), so torch.compile and torch.export trace the attention and the deformable convolution as single
nodes.

There is no CPU or PyTorch fallback: the ops raise if libdevis_msda.so is absent.
"""
from . import _lib, clip_geometry  # noqa: F401
from . import MultiScaleDeformableAttention  # noqa: F401
from . import deform_conv  # noqa: F401
from .functions import (MSDeformAttnFunction, TemporalMSDeformAttnFunction,  # noqa: F401
                        TemporalMSDeformAttnFusedFunction, temporal_ms_deform_attn)
from .modules import (MSDeformAttn, TemporalMSDeformAttnBase, TemporalMSDeformAttnDecoder,  # noqa: F401
                      TemporalMSDeformAttnEncoder)
from .graphed import GraphedLayer  # noqa: F401
from .devis_transformer import (DeVISTransformer, DeVISTransformerDecoder, DeVISTransformerDecoderLayer,  # noqa: F401
                                DeVISTransformerEncoder, DeVISTransformerEncoderLayer)

__all__ = ["MSDeformAttnFunction", "TemporalMSDeformAttnFunction", "TemporalMSDeformAttnFusedFunction", "temporal_ms_deform_attn", "MSDeformAttn",
           "TemporalMSDeformAttnBase", "TemporalMSDeformAttnEncoder", "TemporalMSDeformAttnDecoder",
           "MultiScaleDeformableAttention", "clip_geometry", "DeVISTransformer", "DeVISTransformerEncoder",
           "DeVISTransformerEncoderLayer", "DeVISTransformerDecoder", "DeVISTransformerDecoderLayer", "GraphedLayer"]
