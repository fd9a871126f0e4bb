"""mdn_sfm_b200 -- the MDN_SfM self-supervised geometric loss path as hand-written sm_100a CUDA.

Drop-in modules (same names / signatures as the reference):
    mdn_sfm_b200.loss_functions   Loss, LossModule
    mdn_sfm_b200.loss_utils       inverse_warp, get_epipolar_new, post_process_epipolar_*, smooth_loss, ...
    mdn_sfm_b200.layers           SSIM, get_scale_factor, transformation_from_parameters
    mdn_sfm_b200.utils            gauss_distance_weight, binary_image, FlowWarp
Evaluation:
    mdn_sfm_b200.metrics          mask_confusion, mask_metrics, MaskMetrics (binary_image(mobile, thr) vs moving masks)
There is no CPU implementation: everything raises unless libmdn_loss.so is built and the tensors live on a GPU.
"""
__version__ = "0.1.0"
