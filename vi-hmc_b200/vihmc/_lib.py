"""ctypes binding of libvihmc.so (C ABI: include/vihmc.h).  No torch types cross this boundary:
only raw device pointers, sizes and a cudaStream_t handle."""
from __future__ import annotations

import ctypes as C
import os

MAX_LAYERS = 16
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VIHMC_LIB_PATH", os.path.join(_HERE, "libvihmc.so"))  # override: A/B builds only


class VihmcError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libvihmc error {code}: {message}")
        self.code = code


class Problem(C.Structure):
    _fields_ = [
        ("model_kind", C.c_int32), ("act", C.c_int32), ("loss", C.c_int32), ("last_bias", C.c_int32),
        ("impose_bc", C.c_int32), ("n_layers_a", C.c_int32), ("n_layers_b", C.c_int32), ("in_a", C.c_int32),
        ("in_b", C.c_int32), ("dims_a", C.c_int32 * MAX_LAYERS), ("dims_b", C.c_int32 * MAX_LAYERS),
        ("D", C.c_int64), ("d", C.c_int64), ("N", C.c_int64), ("P", C.c_int64),
        ("tau_out", C.c_float), ("prior_scale", C.c_float), ("prior_sigma_scalar", C.c_float),
        ("prior_log_norm", C.c_float),
        ("x", C.c_void_p), ("x2", C.c_void_p), ("y", C.c_void_p), ("frozen", C.c_void_p), ("sens_ind", C.c_void_p),
        ("prior_mu", C.c_void_p), ("prior_sigma", C.c_void_p), ("frozen_chain_stride", C.c_int64),
    ]


class SamplerCfg(C.Structure):
    _fields_ = [
        ("num_samples", C.c_int32), ("num_steps", C.c_int32), ("burn", C.c_int32), ("integrator", C.c_int32),
        ("adapt_step_size", C.c_int32), ("hamiltorch_fallback_rule", C.c_int32),
        ("step_size", C.c_float), ("desired_accept_rate", C.c_float), ("seed", C.c_uint64), ("chain_offset", C.c_int64),
    ]


class SamplerIO(C.Structure):
    _fields_ = [
        ("accepted", C.c_void_p), ("hamiltonians", C.c_void_p), ("logp", C.c_void_p), ("step_sizes", C.c_void_p),
        ("inject_momenta", C.c_void_p), ("inject_uniforms", C.c_void_p),
        ("vi_sigma", C.c_void_p), ("vi_params", C.c_void_p), ("inject_vi_normals", C.c_void_p),
        ("inv_mass", C.c_void_p),
    ]


class ViCfg(C.Structure):
    _fields_ = [
        ("num_ens", C.c_int32), ("patience", C.c_int32), ("kl_form", C.c_int32), ("reserved", C.c_int32),
        ("lr_start", C.c_float), ("min_lr", C.c_float), ("lr_factor", C.c_float), ("plateau_threshold", C.c_float),
        ("beta", C.c_float), ("prior_mu", C.c_float), ("prior_sigma", C.c_float),
        ("adam_b1", C.c_float), ("adam_b2", C.c_float), ("adam_eps", C.c_float), ("seed", C.c_uint64),
    ]


# every symbol include/vihmc.h declares: name -> (restype, argtypes)
_PP, _PC, _PIO = C.POINTER(Problem), C.POINTER(SamplerCfg), C.POINTER(SamplerIO)
_V, _I64, _U64, _F, _I32, _SZ = C.c_void_p, C.c_int64, C.c_uint64, C.c_float, C.c_int32, C.c_size_t
SYMBOLS = {
    "vihmc_version": (C.c_char_p, []),
    "vihmc_last_error": (C.c_char_p, []),
    "vihmc_device_check": (C.c_int, []),
    "vihmc_prior_log_norm": (C.c_double, [_V, _I64, _F]),
    "vihmc_workspace_bytes": (_SZ, [_PP, _I64]),
    "vihmc_logp_grad": (C.c_int, [_PP, _I64, _V, _V, _V, _V, _SZ, _V]),
    "vihmc_predict": (C.c_int, [_PP, _I64, _V, _V, _V, _SZ, _V]),
    "vihmc_mlp_sample": (C.c_int, [_PP, _PC, _I64, _V, _V, _PIO, _V]),
    "vihmc_sample": (C.c_int, [_PP, _I32, _PC, _I64, _V, _V, _PIO, _V, _SZ, _V]),
    "vihmc_momentum_philox": (C.c_int, [_U64, _I64, _I64, _I64, _I64, _V, _V]),
    "vihmc_uniform_philox": (C.c_int, [_U64, _I64, _I64, _I64, _V, _V]),
    "vihmc_vi_redraw_philox": (C.c_int, [_U64, _I64, _I64, _I64, _I64, _V, _V, _V, _V]),
    "vihmc_scatter_vi": (C.c_int, [_V, _V, _V, _V, _I64, _I64, _I64, _V]),
    "vihmc_gather_vi": (C.c_int, [_V, _V, _V, _I64, _I64, _I64, _V]),
    "vihmc_ke_partials": (_I64, [_I64]),
    "vihmc_leapfrog_update": (C.c_int, [_V, _V, _V, _F, _V, _F, _F, _I64, _I64, _V, _V, _V]),
    "vihmc_mh_accept": (C.c_int, [_V, _V, _V, _V, _V, _V, _V, _I32, _V, _V, _V, _V, _I64, _I64, _V]),
    "vihmc_sample_host": (C.c_int, [_PP, _I32, _PC, _I64, _V, _V, _PIO]),
    "vihmc_mlp_sensitivity_workspace_bytes": (_SZ, [_PP]),
    "vihmc_mlp_sensitivity": (C.c_int, [_PP, _V, _V, _V, _V, _SZ, _V]),
    "vihmc_deeponet_sensitivity_workspace_bytes": (_SZ, [_PP]),
    "vihmc_deeponet_sensitivity": (C.c_int, [_PP, _V, _V, _V, _V, _SZ, _V]),
    "vihmc_vi_workspace_bytes": (_SZ, [_I64, _I32]),
    "vihmc_vi_buffer": (_V, [_V, _I64, _I32, _I32]),
    "vihmc_vi_init": (C.c_int, [C.POINTER(ViCfg), _I64, _V, _SZ, _V]),
    "vihmc_vi_draw": (C.c_int, [C.POINTER(ViCfg), _I64, _V, _V, _V, _V, _SZ, _V]),
    "vihmc_vi_step": (C.c_int, [C.POINTER(ViCfg), _I64, _F, _V, _V, _V, _SZ, _V]),
    "vihmc_vi_epoch_end": (C.c_int, [C.POINTER(ViCfg), _I64, _V, _I32, _F, _V, _V, _V, _V, _SZ, _V]),
    "vihmc_debug_umma": (C.c_int, [_V, _V] + [C.c_uint32] * 7 + [_V, _V]),
    "vihmc_kinetic_energy": (C.c_int, [_V, _I64, _I64, _V, _V, _V]),
    "vihmc_momentum_philox_mass": (C.c_int, [_U64, _I64, _I64, _I64, _I64, _V, _V, _V]),
    "vihmc_kinetic_energy_mass": (C.c_int, [_V, _V, _I64, _I64, _V, _V, _V]),
    "vihmc_leapfrog_update_mass": (C.c_int, [_V, _V, _V, _V, _F, _V, _F, _F, _I64, _I64, _V, _V, _V]),
    "vihmc_debug_tanh": (C.c_int, [_I32, _V, _V, _I64, _V]),
    "vihmc_debug_xgemm_workspace_bytes": (_SZ, [_I32, _I32, _I32]),
    "vihmc_debug_xgemm": (C.c_int, [_V, _I64, _V, _I64, _V, _I64, _I32, _I32, _I32, _I32, _V, _SZ, _V]),
    "vihmc_gemm_batched": (C.c_int, [_V, _I64, _I64, _I64, _V, _I64, _I64, _I64, _V, _I64, _I64, _I32, _I32, _I32, _I32, _I32, _V, _V]),
}

_lib = None


def load() -> C.CDLL:
    """Load libvihmc.so; there is deliberately no fallback if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VihmcError(-1, f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise VihmcError(rc, load().vihmc_last_error().decode())
