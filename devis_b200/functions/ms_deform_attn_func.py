"""``MSDeformAttnFunction`` with the reference's signature and autograd contract
(functions/ms_deform_attn_func.py:21-38): ``apply(value, spatial_shapes, level_start_index,
sampling_locations, attention_weights, im2col_step)``; saves the five input tensors and nothing
else, backward is once-differentiable and returns ``(grad_value, None, None, grad_sampling_loc,
grad_attn_weight, None)``.  The arithmetic runs in the sm_100a kernels behind the C ABI.

(The reference file also holds ``ms_deform_attn_core_pytorch``; that is the oracle and lives in
oracle/msda_torch.py -- the product package has no PyTorch implementation of the op.)
"""
from .. import MultiScaleDeformableAttention as MSDA


class MSDeformAttnFunction:
    """Entry point of the op ``devis::ms_deform_attn`` (MultiScaleDeformableAttention._forward_op), whose registered
    autograd formula is this contract; torch.compile and torch.export trace it as one node."""

    @staticmethod
    def apply(value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights,
              im2col_step):
        return MSDA._forward_op(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                                attention_weights, int(im2col_step), False)
