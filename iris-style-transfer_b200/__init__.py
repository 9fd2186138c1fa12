"""iris_b200 -- B200-native (sm_100a) drop-in for the NST hot path of AnonymWriter/Iris-Style-Transfer.

The arithmetic lives in libisx.so (hand-written CUDA, C ABI in include/isx.h); this package is the
host-side mirror of the reference's Python surface (pipelines.py, utils.py, models/vgg/vgg.py)."""
from . import _lib  # noqa: F401
from . import synthetic  # noqa: F401

try:  # torch-dependent surface (the ctypes layer and the synthetic generators import without torch)
    from .pipelines import (composite_irises, crop_resize_irises, iris_masks_and_bboxes, mask_and_crop_iris,  # noqa: F401
                            nst)
    from .utils import (ContentLoss_L2, GramMatrix, StyleLoss_BN, StyleLoss_Gram, angular_distance, cal_IoUs,  # noqa: F401
                        crop_image, style_features)
    from .vgg import VGG19, random_vgg19_weights  # noqa: F401
    from .frames import stylize_frames  # noqa: F401
    from .ritnet import RITnet  # noqa: F401
    from .classifiers import Classifier1, Classifier2  # noqa: F401
    from .resnet import ResNet50  # noqa: F401
    from .gaze import (GazeEstimator1, GazeEstimator2, extract_eye_landmarks,  # noqa: F401
                       extract_eye_landmarks_batch)
    from . import features, frames, sharding  # noqa: F401
except ImportError:  # pragma: no cover
    pass
