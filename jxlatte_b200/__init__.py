"""jxlatte_b200 -- B200-native (sm_100a) replacement for jxlatte's post-entropy VarDCT reconstruction path
(and the Modular inverse transforms), behind a C ABI (include/jxlb200.h, libjxlb200.so)."""
from .params import FrameParams, default_frame_params, TRANSFORM_TYPES, TRANSFORM_NAMES  # noqa: F401
from .decoder import BatchResult, decode_batch  # noqa: F401,E402
