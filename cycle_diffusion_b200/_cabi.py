"""ctypes binding of include/cdx.h (libcdx.so).  Thin by design: no arithmetic happens in Python.

There is NO CPU fallback: if the shared library is missing the import of this module raises, and
``Engine()`` raises when no CUDA device is usable (cdx_engine_create returns CDX_E_CUDA).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libcdx.so')

CDX_UNET_OPENAI = 1
CDX_UNET_IDDPM = 2
CDX_UNET_DDPM = 3


class UnetConfig(C.Structure):
    _fields_ = [('kind', C.c_int), ('in_channels', C.c_int), ('out_channels', C.c_int), ('model_channels', C.c_int),
                ('num_res_blocks', C.c_int), ('n_mult', C.c_int), ('channel_mult', C.c_int * 8), ('n_attn', C.c_int),
                ('attention_ds', C.c_int * 8), ('num_heads', C.c_int), ('num_head_channels', C.c_int),
                ('context_dim', C.c_int)]


class VaeConfig(C.Structure):
    _fields_ = [('ch', C.c_int), ('n_mult', C.c_int), ('ch_mult', C.c_int * 8), ('num_res_blocks', C.c_int),
                ('in_channels', C.c_int), ('out_ch', C.c_int), ('z_channels', C.c_int), ('embed_dim', C.c_int), ('vq', C.c_int), ('n_embed', C.c_int)]


class TextConfig(C.Structure):
    _fields_ = [('vocab_size', C.c_int), ('width', C.c_int), ('layers', C.c_int), ('heads', C.c_int), ('max_len', C.c_int),
                ('mlp_width', C.c_int), ('kind', C.c_int), ('dim_head', C.c_int), ('proj_dim', C.c_int), ('patch', C.c_int), ('image_size', C.c_int)]


class DdimCoef(C.Structure):
    _fields_ = [('sqrt_at', C.c_float), ('sqrt_1m_at', C.c_float), ('sqrt_1m_at_tab', C.c_float),
                ('sqrt_aprev', C.c_float), ('dir_coef', C.c_float), ('sigma', C.c_float)]


class PixelCoef(C.Structure):
    _fields_ = [('ddpm', C.c_int), ('sqrt_at', C.c_float), ('sqrt_1m_at', C.c_float), ('sqrt_at_next', C.c_float),
                ('c1', C.c_float), ('c2', C.c_float), ('w0', C.c_float), ('wt', C.c_float), ('post_std', C.c_float),
                ('weight', C.c_float), ('inv_sqrt_1m_bt', C.c_float), ('std_model', C.c_float), ('mask', C.c_float)]


class GemmPlan(C.Structure):
    _fields_ = [('path', C.c_int), ('halo', C.c_int), ('epi_tma', C.c_int), ('tn_w', C.c_int), ('splits', C.c_int), ('tail16', C.c_int),
                ('side_done', C.c_int)]


GEMM_PATHS = {0: 'FFMA', 1: 'SS', 2: 'TS', 3: 'H16', 4: 'H16_PAIR'}


class GemmTest(C.Structure):
    _fields_ = [('conv', C.c_int), ('M', C.c_int), ('B', C.c_int), ('H', C.c_int), ('W', C.c_int), ('stride', C.c_int), ('pad', C.c_int),
                ('up', C.c_int), ('N', C.c_int), ('C1', C.c_int), ('C2', C.c_int), ('A', C.c_void_p), ('A2', C.c_void_p),
                ('a_amax', C.c_void_p), ('a2_amax', C.c_void_p), ('w', C.c_void_p), ('bias', C.c_void_p), ('rowvec', C.c_void_p),
                ('ld_rowvec', C.c_int), ('rows_per_batch', C.c_int), ('residual', C.c_void_p), ('ldr', C.c_int), ('alpha', C.c_float),
                ('geglu', C.c_int), ('C', C.c_void_p), ('ldc', C.c_int), ('out_nchw', C.c_int), ('rows_per_img', C.c_int),
                ('C_lo', C.c_void_p), ('Ct_hi', C.c_void_p), ('Ct_lo', C.c_void_p), ('t_col0', C.c_int), ('ldt', C.c_longlong),
                ('c_amax', C.c_void_p), ('c_stats', C.c_void_p), ('plan', C.POINTER(GemmPlan))]


_P = C.c_void_p          # device / opaque pointers
_F = C.c_float
_I = C.c_int
_S = C.c_size_t

# name -> (restype, argtypes); every symbol include/cdx.h declares (tests/test_cabi.py checks the list against the header)
SIGNATURES = {
    'cdx_abi_version': (_I, []),
    'cdx_last_error': (C.c_char_p, []),
    'cdx_engine_create': (_I, [_I, C.POINTER(_P)]),
    'cdx_engine_destroy': (None, [_P]),
    'cdx_engine_workspace_bytes': (_S, [_P]),
    'cdx_engine_launch_count': (C.c_uint64, [_P]),
    'cdx_engine_set_mma_mode': (_I, [_P, _I]),
    'cdx_engine_profile': (_I, [_P, _I]),
    'cdx_engine_profile_read': (_I, [_P, _I, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    'cdx_unet_create': (_I, [_P, C.POINTER(UnetConfig), C.POINTER(_P)]),
    'cdx_vae_create': (_I, [_P, C.POINTER(VaeConfig), C.POINTER(_P)]),
    'cdx_text_create': (_I, [_P, C.POINTER(TextConfig), C.POINTER(_P)]),
    'cdx_net_destroy': (None, [_P]),
    'cdx_net_num_params': (_I, [_P]),
    'cdx_net_param_name': (C.c_char_p, [_P, _I]),
    'cdx_net_param_shape': (_I, [_P, _I, C.POINTER(C.c_int64)]),
    'cdx_net_load_param': (_I, [_P, C.c_char_p, _P, _I, C.POINTER(C.c_int64), _I]),
    'cdx_net_finalize': (_I, [_P]),
    'cdx_net_weight_blob': (_I, [_P, C.POINTER(_P), C.POINTER(_S)]),
    'cdx_net_adopt_blob': (_I, [_P]),
    'cdx_unet_set_time_freqs': (_I, [_P, C.POINTER(_F), _I]),
    'cdx_unet_forward': (_I, [_P, _P, _P, _P, _I, _P, _I, _I, _I, _P]),
    'cdx_vae_encode': (_I, [_P, _P, _P, _I, _I, _P]),
    'cdx_text_encode': (_I, [_P, _P, _I, _I, _P, _P]),
    'cdx_vae_decode': (_I, [_P, _P, _P, _I, _I, _P]),
    'cdx_affine': (_I, [_P, _P, _F, _F, _P, _S, _P]),
    'cdx_shift_scale': (_I, [_P, _P, _F, _F, _P, _S, _P]),
    'cdx_q_sample': (_I, [_P, _P, _P, _F, _F, _P, _S, _P]),
    'cdx_vae_posterior': (_I, [_P, _P, _P, _F, _P, _I, _I, _I, _P]),
    'cdx_ddim_posterior_sample': (_I, [_P, _P, _P, _P, C.POINTER(DdimCoef), _P, _S, _P]),
    'cdx_ddim_compute_eps': (_I, [_P, _P, _P, _P, _P, _F, C.POINTER(DdimCoef), _P, _S, _P]),
    'cdx_ddim_step_with_eps': (_I, [_P, _P, _P, _P, _F, _P, C.POINTER(DdimCoef), _P, _S, _P]),
    'cdx_pixel_posterior_sample': (_I, [_P, _P, _P, _P, C.POINTER(PixelCoef), _P, _S, _P]),
    'cdx_pixel_compute_eps': (_I, [_P, _P, _P, _P, C.POINTER(PixelCoef), _P, _I, _I, _I, _P]),
    'cdx_pixel_step_with_eps': (_I, [_P, _P, _P, _P, C.POINTER(PixelCoef), _P, _I, _I, _I, _P]),
    'cdx_latent_encode': (_I, [_P, _P, _P, _P, _I, _F, C.POINTER(DdimCoef), C.POINTER(_F), _I, _I, _P, _F, _F, _P, _I, _I,
                               _I, _I, _P]),
    'cdx_latent_decode': (_I, [_P, _P, _I, _P, _P, _I, _F, C.POINTER(DdimCoef), C.POINTER(_F), _I, _P, _P, _I, _I, _I, _I,
                               _P]),
    'cdx_cycle_lockstep': (_I, [_P, _P, _P, _P, _P, _I, _F, _F, C.POINTER(DdimCoef), C.POINTER(_F), _I, _P, _F, _F, _P, _P, _I, _I, _I, _I,
                                _P]),
    'cdx_cycle_lockstep_pair': (_I, [_P, _P, _P, _P, _P, _P, _I, _F, _F, C.POINTER(DdimCoef), C.POINTER(_F), _I, _P, _F, _F, _P, _P, _I, _I,
                                     _I, _I, _P]),
    'cdx_latent_loop_ens': (_I, [_P, _I, _P, _P, _P, _P, _I, _P, _P, C.POINTER(DdimCoef), C.POINTER(_F), _I, _I, _P, _F, _F, _P, _I, _P, _P, _P,
                                 _I, _I, _I, _I, _P]),
    'cdx_clip_preprocess': (_I, [_P, _P, _I, _I, _I, _P, _P]),
    'cdx_clip_image_features': (_I, [_P, _P, _I, _P, _P]),
    'cdx_text_features': (_I, [_P, _P, _I, _I, _P, _P]),
    'cdx_dclip_scores': (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P]),
    'cdx_image_metrics': (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    'cdx_pixel_encode': (_I, [_P, _P, C.POINTER(PixelCoef), C.POINTER(_F), _I, _P, _F, _F, _P, _I, _I, _I, _P]),
    'cdx_pixel_decode': (_I, [_P, _P, _I, C.POINTER(PixelCoef), C.POINTER(_F), _I, _P, _P, _I, _I, _I, _P]),
    'cdx_pixel_cycle_lockstep': (_I, [_P, _P, _P, C.POINTER(PixelCoef), C.POINTER(_F), _I, _P, _F, _F, _P, _P, _P, _I, _I, _I, _P]),
    'cdx_op_gemm': (_I, [_P, C.POINTER(GemmTest), _P]),
    'cdx_op_groupnorm': (_I, [_P, _P, _I, _P, _I, _P, _P, _F, _I, _P, _P, _I, _P, _P, _P, _P, _I, _I, _P]),
    'cdx_op_layernorm': (_I, [_P, _P, _P, _P, _P, _I, _I, _P]),
    'cdx_op_attention': (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
    'cdx_op_nchw_to_nhwc': (_I, [_P, _P, _P, _I, _I, _I, _P]),
    'cdx_op_nhwc_to_nchw': (_I, [_P, _P, _P, _I, _I, _I, _P]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            f'(nvcc, sm_100a).  The engine has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


class CdxError(RuntimeError):
    pass


def check(rc):
    """Translate a CDX_E_* status into the exception type the reference's own checks raise."""
    if rc == 0:
        return
    msg = (lib.cdx_last_error() or b'').decode('utf-8', 'replace')
    if rc == -1:
        raise AssertionError(msg)     # the reference uses assert for preconditions (SDW:178, DDIM:268, DW:472)
    raise CdxError(f'libcdx error {rc}: {msg}')
