"""fhe_string_bounty_b200 -- B200-native (sm_100a) engine for the shortint KS-PBS hot path of the
tfhe-rs 0.5.0 fork Lcressot/fhe-string-bounty.

The product is the C-ABI shared library ``libtfhe_b200.so`` (``include/tfhe_b200.h``); this package is a
thin ctypes loader plus host-side mirrors of the reference interfaces that sit on the path.  There is no
CPU fallback: every compute entry point fails loudly if the CUDA library or a GPU is missing.
"""
from ._native import Engine, Params, build_native, load_native, many_lut_accumulator, NativeError, PARAM_MESSAGE_2_CARRY_2_KS_PBS, PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS, classic_params, multi_bit_params  # noqa: F401

__all__ = ["Engine", "Params", "build_native", "load_native", "many_lut_accumulator", "NativeError", "PARAM_MESSAGE_2_CARRY_2_KS_PBS", "PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS", "classic_params", "multi_bit_params"]
