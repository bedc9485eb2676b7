"""mdqtplasmasims_b200 -- B200-native engine for the per-timestep MDQT hot path of tlangin/MDQTPlasmaSims.

Only what the hot path needs: ``csrc/`` (hand-written sm_100a CUDA kernels + the C ABI of include/mdqt.h),
``engine.py`` (ctypes mirror of the reference's forces()/step()/qstep() interface), ``synthetic.py`` (synthetic
random-start inputs of the reference's shapes) and ``build.py`` (in-tree nvcc build).
"""
from .engine import (Engine, MDQTError, Params, axis_wavevectors, load_library, md_params, philox_uniforms, su_params,  # noqa: F401
                     ts_params, SCHEME_NONE, SCHEME_SR7, SCHEME_SR12, SCHEME_CA5, SCHEME_V3, ABI_SYMBOLS, LIB_PATH)
