"""ctypes signatures of the training entry points of libfact_sm100.so."""
from __future__ import annotations

import ctypes as C

_vp, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float

SIGNATURES: dict = {
    "fact_sdpa_lse": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "fact_wgrad_gemm": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "fact_sdpa_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "fact_layernorm_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "fact_embed_backward": (_i, [_vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "fact_cast_colsum": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _vp]),
    "fact_cast_weight": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "fact_adam_step": (_i, [_vp, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _ll, _f, _vp, _vp]),
    "fact_dp_adam_step": (_i, [C.POINTER(_vp), _vp, _ll, _ll, _ll, _vp, _vp, _ll, _i, _i, _f, _f, _f, _f, _ll, _f, _vp]),
    "fact_dp_adam_range": (_i, [C.POINTER(_vp), _vp, _ll, _ll, _ll, _vp, _vp, _ll, _ll, _i, _i, _f, _f, _f, _f, _ll, _f,
                                _i, _vp]),
    "fact_sum_squares": (_i, [_vp, _ll, _vp, _vp]),
    "fact_train_workspace_bytes": (C.c_size_t, [_vp, _i]),
    "fact_clip_scale": (_i, [_vp, _ll, _vp, _f, _vp]),
    "fact_train_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp, _vp, C.c_size_t, C.POINTER(_vp), _i, _vp]),
    "fact_gather_windows": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
}


def bind(lib) -> None:
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
