"""dcae_b200: B200 (sm_100a) implementation of the DCAE entropy-model hot path.

Public surface (mirrors the reference's operator interface for this path only):
  EntropySliceLoop      -- the channel-slice loop of DCAE.forward/compress/decompress
  HostPipeline          -- pinned-host-in / pinned-host-out streaming front end (overlapped copies)
  GaussianConditional   -- compressai-compatible quantise / likelihood / build_indexes (kernel 3)
  EntropyBottleneck     -- compressai-compatible factorised prior for the hyper-latent z (one fused pass + the native coder)
  accelerate, DictCrossAttention, ConvStack -- module-level drop-ins for a reference DCAE instance (dcae_b200/modules.py)
  EntropyModel, SliceLoopFunction -- the training form (autograd: kernels forward, torch-graph recompute backward)
  ans.BufferedRansEncoder / RansDecoder -- the native range coder with compressai.ans' interface
  init_entropy_params   -- deterministic random-init weights with the reference's state-dict keys
  TransformStack, accelerate_transforms, init_transform_params -- g_a / g_s / h_a / h_z_s1 / h_z_s2 on the library (dcae_b200/transforms.py);
                        accelerate_transforms also trains: under autograd each stack call is a recompute node
  TransformModel        -- one transform stack as a trainable module (kernels forward, recompute backward with the
                           window-attention backward kernel; dcae_b200/training.py)
  EntropyBottleneckModel, DCAEModel, dcae_rate_distortion_loss -- the trainable bottleneck (backward kernel
                           dcae_eb_backward) and the whole DCAE as one trainable module (dcae_b200/training.py)
  ms_ssim, MSSSIMStatsFunction -- MS-SSIM with the library's forward and backward kernels (dcae_b200/msssim.py); the
                           distortion of dcae_rate_distortion_loss(..., metric="ms-ssim")
  DCAECodec             -- the whole model (forward / compress / decompress / update, image <-> .bin container) from a reference state dict
  container             -- the reference's bitstream container and image padding (compress_and_decompress.py:48-148)
"""
from .params import init_entropy_params, entropy_param_shapes  # noqa: F401


def __getattr__(name):
    # CUDA-facing classes are imported lazily so that `import dcae_b200` works on a build box
    if name in ("EntropySliceLoop", "get_scale_table", "bits_per_pixel"):
        from . import entropy_model
        return getattr(entropy_model, name)
    if name == "HostPipeline":
        from .pipeline import HostPipeline
        return HostPipeline
    if name in ("accelerate", "DictCrossAttention", "ConvStack"):
        from . import modules
        return getattr(modules, name)
    if name in ("EntropyModel", "SliceLoopFunction", "GaussianLikelihoodFunction", "rate_distortion_loss", "TransformModel",
                "EntropyBottleneckFunction", "EntropyBottleneckModel", "DCAEModel", "dcae_rate_distortion_loss"):
        from . import training
        return getattr(training, name)
    if name in ("ms_ssim", "MSSSIMStatsFunction"):
        from . import msssim
        return getattr(msssim, name)
    if name == "EntropyBottleneck":
        from .entropy_bottleneck import EntropyBottleneck
        return EntropyBottleneck
    if name in ("TransformStack", "accelerate_transforms", "init_transform_params", "transform_param_shapes"):
        from . import transforms
        return getattr(transforms, name)
    if name == "container":
        import importlib
        return importlib.import_module(".container", __name__)
    if name == "DCAECodec":
        from .codec import DCAECodec
        return DCAECodec
    if name == "GaussianConditional":
        from .gaussian_conditional import GaussianConditional
        return GaussianConditional
    raise AttributeError(name)
