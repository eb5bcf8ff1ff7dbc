"""Python handles over the libcdx C ABI: Engine (per device), UNet / VAE networks, per-step kernels, loop drivers.

PyTorch is used only as plumbing: device memory (``torch.empty(..., device='cuda')``), streams and
``torch.distributed``.  Every compute call goes through ctypes into hand-written sm_100a kernels; there is no
torch.nn / CPU fallback anywhere on this path.
"""
import ctypes as C
import math

import torch

from . import _cabi
from ._cabi import lib, check, UnetConfig, VaeConfig, TextConfig, DdimCoef, PixelCoef


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f32c(t, device):
    assert t.dtype == torch.float32, f'expected float32, got {t.dtype}'
    if t.device != device:
        t = t.to(device)
    return t.contiguous()


class Engine:
    """One per CUDA device / rank.  Not thread-safe; all work is enqueued on the current torch stream."""

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise RuntimeError('cycle_diffusion_b200 needs a CUDA device: the engine has no CPU fallback')
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        torch.cuda.set_device(self.device)
        h = C.c_void_p()
        check(lib.cdx_engine_create(self.device.index, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, 'h', None):
            lib.cdx_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launches(self):
        return int(lib.cdx_engine_launch_count(self.h))

    @property
    def workspace_bytes(self):
        return int(lib.cdx_engine_workspace_bytes(self.h))

    def set_mma_mode(self, mode):
        check(lib.cdx_engine_set_mma_mode(self.h, int(mode)))

    PROF_TAGS = ['conv3x3_ffma', 'dense_ffma', 'batched_ffma', 'conv3x3_tc', 'dense_tc', 'batched_tc', 'groupnorm', 'layernorm',
                 'softmax', 'other']

    def profile(self, enable):
        check(lib.cdx_engine_profile(self.h, int(enable)))

    def profile_read(self):
        """{tag: dict(ms, flops, bytes, launches)} of everything recorded since profile(True)."""
        out = {}
        for i, name in enumerate(self.PROF_TAGS):
            ms, fl, by, n = C.c_double(), C.c_double(), C.c_double(), C.c_uint64()
            check(lib.cdx_engine_profile_read(self.h, i, C.byref(ms), C.byref(fl), C.byref(by), C.byref(n)))
            if n.value:
                out[name] = dict(ms=ms.value, flops=fl.value, bytes=by.value, launches=int(n.value))
        return out

    def empty(self, *shape):
        return torch.empty(*shape, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ per-step kernels
    def affine(self, x, a, b):
        x = _f32c(x, self.device)
        out = torch.empty_like(x)
        check(lib.cdx_affine(self.h, _ptr(x), a, b, _ptr(out), x.numel(), self.stream))
        return out

    def shift_scale(self, x, b, a):
        x = _f32c(x, self.device)
        out = torch.empty_like(x)
        check(lib.cdx_shift_scale(self.h, _ptr(x), b, a, _ptr(out), x.numel(), self.stream))
        return out

    def q_sample(self, x0, noise, sqrt_a, sqrt_1ma):
        x0, noise = _f32c(x0, self.device), _f32c(noise, self.device)
        out = torch.empty_like(x0)
        check(lib.cdx_q_sample(self.h, _ptr(x0), _ptr(noise), sqrt_a, sqrt_1ma, _ptr(out), x0.numel(), self.stream))
        return out

    def vae_posterior(self, moments, noise, scale_factor):
        moments = _f32c(moments, self.device)
        B, C2, h, w = moments.shape
        out = self.empty(B, C2 // 2, h, w)
        if noise is not None:
            noise = _f32c(noise, self.device)
            assert noise.shape == out.shape
        check(lib.cdx_vae_posterior(self.h, _ptr(moments), _ptr(noise), scale_factor, _ptr(out), B, C2 // 2, h * w, self.stream))
        return out

    def ddim_posterior_sample(self, x0, xt, noise, coef):
        x0, xt, noise = (_f32c(t, self.device) for t in (x0, xt, noise))
        out = torch.empty_like(x0)
        check(lib.cdx_ddim_posterior_sample(self.h, _ptr(x0), _ptr(xt), _ptr(noise), C.byref(coef), _ptr(out), x0.numel(), self.stream))
        return out

    def ddim_compute_eps(self, xt, xt_next, e_c, e_uc, scale, coef):
        xt, xt_next, e_c = (_f32c(t, self.device) for t in (xt, xt_next, e_c))
        e_uc = _f32c(e_uc, self.device) if e_uc is not None else None
        out = torch.empty_like(xt)
        check(lib.cdx_ddim_compute_eps(self.h, _ptr(xt), _ptr(xt_next), _ptr(e_c), _ptr(e_uc), scale, C.byref(coef), _ptr(out),
                                       xt.numel(), self.stream))
        return out

    def ddim_step_with_eps(self, x, e_c, e_uc, scale, eps, coef):
        x, e_c, eps = (_f32c(t, self.device) for t in (x, e_c, eps))
        e_uc = _f32c(e_uc, self.device) if e_uc is not None else None
        out = torch.empty_like(x)
        check(lib.cdx_ddim_step_with_eps(self.h, _ptr(x), _ptr(e_c), _ptr(e_uc), scale, _ptr(eps), C.byref(coef), _ptr(out),
                                         x.numel(), self.stream))
        return out

    def pixel_posterior_sample(self, x0, xt, noise, coef):
        x0, xt, noise = (_f32c(t, self.device) for t in (x0, xt, noise))
        out = torch.empty_like(x0)
        check(lib.cdx_pixel_posterior_sample(self.h, _ptr(x0), _ptr(xt), _ptr(noise), C.byref(coef), _ptr(out), x0.numel(), self.stream))
        return out

    def pixel_compute_eps(self, xt, xt_next, et, coef):
        xt, xt_next, et = (_f32c(t, self.device) for t in (xt, xt_next, et))
        B = xt.shape[0]
        out = torch.empty_like(xt)
        check(lib.cdx_pixel_compute_eps(self.h, _ptr(xt), _ptr(xt_next), _ptr(et), C.byref(coef), _ptr(out), B, xt[0].numel(),
                                        et[0].numel(), self.stream))
        return out

    def pixel_step_with_eps(self, xt, et, eps, coef):
        xt, et = _f32c(xt, self.device), _f32c(et, self.device)
        eps = _f32c(eps, self.device) if eps is not None else None
        B = xt.shape[0]
        out = torch.empty_like(xt)
        check(lib.cdx_pixel_step_with_eps(self.h, _ptr(xt), _ptr(et), _ptr(eps), C.byref(coef), _ptr(out), B, xt[0].numel(),
                                          et[0].numel(), self.stream))
        return out

    # ------------------------------------------------------------------ unit-test hooks (NHWC)
    def op_conv3x3(self, x_nhwc, w_oihw, bias, stride=1, pad_lo=1, upsample=1):
        return self.op_gemm(x_nhwc, w_oihw, bias, conv=dict(stride=stride, pad=pad_lo, up=upsample))['C']

    def op_linear(self, x, w, bias):
        return self.op_gemm(x, w, bias)['C']

    def op_gemm(self, x, w, bias=None, *, conv=None, x2=None, a_amax=None, a2_amax=None, rowvec=None, rows_per_batch=0, residual=None,
                alpha=1.0, geglu=False, out_nchw=False, planes=False, t_col0=None, c_amax=False, c_stats=False, ldc=0):
        """One GEMM through cdx_op_gemm with the networks' epilogue options.

        x: dense [M, C1] (x2: optional second source [M, C2]) or, with conv=dict(stride, pad, up), NHWC [B, H, W, C1] and w OIHW.
        a_amax / a2_amax: optional one-element device tensors (tracked ranges).  geglu: w / bias in the reference [value; gate] layout.
        planes: C and C_lo receive TF32 hi / lo planes; t_col0: columns >= t_col0 go transposed to Ct_hi / Ct_lo [N - t_col0, M]
        (C then holds the first t_col0 columns, ldc = t_col0).  Returns a dict with C (and C_lo, Ct_hi, Ct_lo, c_amax, c_stats when
        asked for) and `plan`, the variant that ran (_cabi.GemmPlan fields, path as a name)."""
        dev = self.device
        x, w = _f32c(x, dev), _f32c(w, dev)
        opt = lambda t: _f32c(t, dev) if t is not None else None
        bias, x2, rowvec, residual = opt(bias), opt(x2), opt(rowvec), opt(residual)
        N = w.shape[0]
        t = _cabi.GemmTest()
        if conv is not None:
            B, H, W, C1 = x.shape
            stride, pad, up = conv.get('stride', 1), conv.get('pad', 1), conv.get('up', 1)
            Ho, Wo = (H * up, W * up) if stride == 1 else (H * up // 2, W * up // 2)
            M, lead = B * Ho * Wo, (B, Ho, Wo)
            t.conv, t.B, t.H, t.W, t.stride, t.pad, t.up = 1, B, H, W, stride, pad, up
        else:
            M, C1 = x.shape
            lead = (M,)
            t.M = M
        ncols = N // 2 if geglu else (t_col0 if t_col0 is not None else N)
        imgs = lead[0] if conv is not None else 1               # images (rows_per_batch default: one image per conv sample)
        rpb = rows_per_batch or M // imgs
        out = {'C': self.empty(imgs, N, M // imgs) if out_nchw else self.empty(*lead, ldc or ncols)}
        t.N, t.C1 = N, C1
        t.A, t.w, t.bias = _ptr(x), _ptr(w), _ptr(bias)
        if x2 is not None:
            t.A2, t.C2 = _ptr(x2), x2.shape[-1]
        t.a_amax, t.a2_amax = _ptr(a_amax), _ptr(a2_amax)
        if rowvec is not None:
            t.rowvec, t.ld_rowvec = _ptr(rowvec), rowvec.shape[-1]
        t.rows_per_batch = rpb
        if residual is not None:
            t.residual, t.ldr = _ptr(residual), residual.shape[-1]
        t.alpha, t.geglu, t.out_nchw = float(alpha), int(geglu), int(out_nchw)
        t.C, t.ldc = _ptr(out['C']), ldc or (0 if t_col0 is None else t_col0)
        if planes:
            out['C_lo'] = torch.empty_like(out['C'])
            t.C_lo = _ptr(out['C_lo'])
        if t_col0 is not None:
            out['Ct_hi'], out['Ct_lo'] = self.empty(N - t_col0, M), self.empty(N - t_col0, M)
            t.Ct_hi, t.Ct_lo, t.t_col0, t.ldt = _ptr(out['Ct_hi']), _ptr(out['Ct_lo']), t_col0, M
        if c_amax:
            out['c_amax'] = self.empty(1)
            t.c_amax = _ptr(out['c_amax'])
        if c_stats:
            out['c_stats'] = torch.empty(M // rpb, N, 2, dtype=torch.float64, device=dev)
            t.c_stats = _ptr(out['c_stats'])
        plan = _cabi.GemmPlan()
        t.plan = C.pointer(plan)
        check(lib.cdx_op_gemm(self.h, C.byref(t), self.stream))
        out['plan'] = {f: getattr(plan, f) for f, _ in _cabi.GemmPlan._fields_}
        out['plan']['path'] = _cabi.GEMM_PATHS.get(plan.path, plan.path)
        return out

    # ---- Directional-CLIP ranking / evaluation metrics (SURVEY 8f-3)
    def clip_preprocess(self, img, size=224):
        """clean_clip.py:14-17 on a float batch in [0,1]: bicubic resize to size x size + CLIP normalisation."""
        x = _f32c(img, self.device)
        B, Cc, R, R2 = x.shape
        assert Cc == 3 and R == R2, 'square RGB batches (the reference feeds R x R sampler outputs)'
        out = self.empty(B, 3, size, size)
        check(lib.cdx_clip_preprocess(self.h, _ptr(x), B, R, size, _ptr(out), self.stream))
        return out

    def dclip_scores(self, img_f, orig_f, enc_f, dec_f):
        fs = [_f32c(t, self.device) for t in (img_f, orig_f, enc_f, dec_f)]
        B, D = fs[0].shape
        clip, dclip = self.empty(B), self.empty(B)
        check(lib.cdx_dclip_scores(self.h, *[_ptr(t) for t in fs], B, D, _ptr(clip), _ptr(dclip), self.stream))
        return clip, dclip

    def image_metrics(self, a, b):
        """-> [B, 3] = (psnr, ssim, l2) per image pair (evaluation/translate_text.py:76-89)."""
        a, b = _f32c(a, self.device), _f32c(b, self.device)
        B, Cc, H, W = a.shape
        assert Cc == 3 and a.shape == b.shape
        out = self.empty(B, 3)
        check(lib.cdx_image_metrics(self.h, _ptr(a), _ptr(b), B, H, W, _ptr(out), self.stream))
        return out

    def op_groupnorm(self, x_nhwc, gamma, beta, eps, silu, x2=None, scale_shift=None, st1=None, st2=None, amax=False):
        """GroupNorm(32) of x (or of the channel concat [x | x2]) -> [silu](gn * (1 + scale) + shift).  scale_shift: optional
        [B, 2C] rows (scale first, as the improved-DDPM ResBlock chunks its embedding); st1 / st2: optional fp64 [B, C, 2] channel
        statistics of the sources; amax=True returns (y, max |y| as a one-element tensor)."""
        x, gamma, beta = (_f32c(t, self.device) for t in (x_nhwc, gamma, beta))
        x2, ss = (_f32c(t, self.device) if t is not None else None for t in (x2, scale_shift))
        st1, st2 = (t.to(self.device).contiguous() if t is not None else None for t in (st1, st2))
        B, H, W, C1 = x.shape
        C2 = x2.shape[-1] if x2 is not None else 0
        y = self.empty(B, H, W, C1 + C2)
        am = self.empty(1) if amax else None
        scale, shift, ld_ss = (ss, ss[:, C1 + C2:], ss.shape[-1]) if ss is not None else (None, None, 0)
        check(lib.cdx_op_groupnorm(self.h, _ptr(x), C1, _ptr(x2), C2, _ptr(gamma), _ptr(beta), eps, int(silu), _ptr(scale), _ptr(shift), ld_ss,
                                   _ptr(st1), _ptr(st2), _ptr(am), _ptr(y), B, H * W, self.stream))
        return (y, am) if amax else y

    def op_layernorm(self, x, gamma, beta):
        x, gamma, beta = (_f32c(t, self.device) for t in (x, gamma, beta))
        M, Cc = x.shape
        y = torch.empty_like(x)
        check(lib.cdx_op_layernorm(self.h, _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), M, Cc, self.stream))
        return y

    def op_attention(self, q, k, v, heads, scale):
        q, k, v = (_f32c(t, self.device) for t in (q, k, v))
        B, Nq, Cc = q.shape
        Nk = k.shape[1]
        out = torch.empty_like(q)
        check(lib.cdx_op_attention(self.h, _ptr(q), _ptr(k), _ptr(v), _ptr(out), B, Nq, Nk, heads, Cc // heads, scale, self.stream))
        return out

    def op_nchw_to_nhwc(self, x):
        x = _f32c(x, self.device)
        B, Cc, H, W = x.shape
        y = self.empty(B, H, W, Cc)
        check(lib.cdx_op_nchw_to_nhwc(self.h, _ptr(x), _ptr(y), B, Cc, H * W, self.stream))
        return y

    def op_nhwc_to_nchw(self, x):
        x = _f32c(x, self.device)
        B, H, W, Cc = x.shape
        y = self.empty(B, Cc, H, W)
        check(lib.cdx_op_nhwc_to_nchw(self.h, _ptr(x), _ptr(y), B, Cc, H * W, self.stream))
        return y


def _int_arr8(vals):
    a = (C.c_int * 8)()
    for i, v in enumerate(vals):
        a[i] = int(v)
    return a


class Net:
    """A network living in the engine: parameter inventory + packed weight blob."""

    def __init__(self, engine, handle):
        self.engine = engine
        self.h = handle
        self.finalized = False

    def close(self):
        if getattr(self, 'h', None):
            lib.cdx_net_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def inventory(self):
        """[(name, shape)] in the reference checkpoint's key names."""
        out = []
        dims = (C.c_int64 * 4)()
        for i in range(lib.cdx_net_num_params(self.h)):
            name = lib.cdx_net_param_name(self.h, i).decode()
            rank = lib.cdx_net_param_shape(self.h, i, dims)
            out.append((name, tuple(int(dims[k]) for k in range(rank))))
        return out

    def load_state_dict(self, sd, prefix='', strict=True):
        """Load a reference-style state_dict (keys optionally under ``prefix``, e.g. 'model.diffusion_model.')."""
        inv = self.inventory()
        names = {n for n, _ in inv}
        if strict:
            extra = [k[len(prefix):] for k in sd if k.startswith(prefix) and k[len(prefix):] not in names]
            assert not extra, f'unexpected keys in state_dict: {extra[:5]}...'
        for name, shape in inv:
            key = prefix + name
            assert key in sd, f'missing key in state_dict: {key}'
            t = sd[key]
            assert tuple(t.shape) == shape, f'{key}: shape {tuple(t.shape)} != {shape}'
            t = t.detach().to(torch.float32).contiguous()
            dims = (C.c_int64 * 4)(*(list(shape) + [1] * (4 - len(shape))))
            check(lib.cdx_net_load_param(self.h, name.encode(), _ptr(t), 1 if t.is_cuda else 0, dims, len(shape)))
        self.finalize()
        return self

    def finalize(self):
        check(lib.cdx_net_finalize(self.h))
        self.finalized = True

    def weight_blob(self):
        """(device pointer, bytes) of the packed weights -- the buffer rank 0 broadcasts over NCCL."""
        p, n = C.c_void_p(), C.c_size_t()
        check(lib.cdx_net_weight_blob(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def blob_tensor(self):
        """A torch view of the packed weight blob (no copy), for torch.distributed.broadcast."""
        p, n = self.weight_blob()

        class _Blob:
            __cuda_array_interface__ = {'shape': (n // 4,), 'typestr': '<f4', 'data': (p, False), 'version': 2}
        return torch.as_tensor(_Blob(), device=self.engine.device)

    def adopt_blob(self):
        check(lib.cdx_net_adopt_blob(self.h))
        self.finalized = True


class UNet(Net):
    """SD/LDM (kind='openai') or improved-DDPM (kind='iddpm') eps-prediction U-Net."""

    def __init__(self, engine, cfg, kind='openai'):
        self.cfg = dict(cfg)
        self.kind = kind
        c = UnetConfig()
        c.kind = {'openai': _cabi.CDX_UNET_OPENAI, 'iddpm': _cabi.CDX_UNET_IDDPM, 'ddpm': _cabi.CDX_UNET_DDPM}[kind]
        c.in_channels, c.out_channels = cfg['in_channels'], cfg['out_channels']
        c.model_channels, c.num_res_blocks = cfg['model_channels'], cfg['num_res_blocks']
        c.n_mult = len(cfg['channel_mult'])
        c.channel_mult = _int_arr8(cfg['channel_mult'])
        c.n_attn = len(cfg['attention_resolutions'])
        c.attention_ds = _int_arr8(cfg['attention_resolutions'])
        c.num_heads = cfg.get('num_heads', 0)
        c.num_head_channels = cfg.get('num_head_channels', 0)
        c.context_dim = cfg.get('context_dim', 0)
        h = C.c_void_p()
        check(lib.cdx_unet_create(engine.h if engine is not None else None, C.byref(c), C.byref(h)))
        super().__init__(engine, h)
        if engine is not None:
            # sinusoid frequencies with the reference expression (util.py:161-163 / nn.py:112-114), evaluated by torch on
            # the host so that they are bit-identical to what the reference / oracle computes on this machine
            half = cfg['model_channels'] // 2
            if kind == 'ddpm':          # get_timestep_embedding, ddpm/diffusion.py:15-18: log(10000) / (half - 1)
                freqs = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
            else:
                freqs = torch.exp(-math.log(10000) * torch.arange(start=0, end=half, dtype=torch.float32) / half)
            arr = (C.c_float * half)(*freqs.tolist())
            check(lib.cdx_unet_set_time_freqs(self.h, arr, half))

    def forward(self, x, timesteps, context=None):
        e = self.engine
        x = _f32c(x, e.device)
        B, _, H, W = x.shape
        t = timesteps.to(device=e.device, dtype=torch.float32).contiguous()
        assert t.shape == (B,)
        L = 0
        if context is not None:
            context = _f32c(context, e.device)
            assert context.shape[0] == B and context.shape[2] == self.cfg['context_dim']
            L = context.shape[1]
        out = e.empty(B, self.cfg['out_channels'], H, W)
        check(lib.cdx_unet_forward(self.h, _ptr(x), _ptr(t), _ptr(context), L, _ptr(out), B, H, W, e.stream))
        return out

    __call__ = forward

    # ---- loop drivers (whole chains enqueued inside libcdx)
    def latent_encode(self, x0, c, uc, scale, sched, n_rec, noise):
        """-> z [B, n_rec+1, C, h, w]; noise [n_rec+1, B, C, h, w] in the reference's draw order."""
        e = self.engine
        x0, noise = _f32c(x0, e.device), _f32c(noise, e.device)
        c = _f32c(c, e.device) if c is not None else None            # None: unconditional model (no context)
        uc = _f32c(uc, e.device) if uc is not None else None
        B, Cc, h, w = x0.shape
        assert noise.shape == (n_rec + 1, B, Cc, h, w), f'noise shape {tuple(noise.shape)}'
        z = e.empty(B, n_rec + 1, Cc, h, w)
        check(lib.cdx_latent_encode(self.h, _ptr(x0), _ptr(c), _ptr(uc), c.shape[1] if c is not None else 0, float(scale), sched.coef_array(), sched.t_array(),
                                    sched.refine_steps, n_rec, _ptr(noise), sched.sqrt_a_T, sched.sqrt_1ma_T, _ptr(z), B, Cc, h, w,
                                    e.stream))
        return z

    def latent_decode(self, z, c, uc, scale, sched, extra_noise=None):
        """z [B, n_eps+1, C, h, w] -> x0 [B, C, h, w]."""
        e = self.engine
        z = _f32c(z, e.device)
        c = _f32c(c, e.device) if c is not None else None
        uc = _f32c(uc, e.device) if uc is not None else None
        extra_noise = _f32c(extra_noise, e.device) if extra_noise is not None else None
        B, n1, Cc, h, w = z.shape
        out = e.empty(B, Cc, h, w)
        check(lib.cdx_latent_decode(self.h, _ptr(z), n1 - 1, _ptr(c), _ptr(uc), c.shape[1] if c is not None else 0, float(scale), sched.coef_array(),
                                    sched.t_array(), sched.refine_steps, _ptr(extra_noise), _ptr(out), B, Cc, h, w, e.stream))
        return out

    def latent_refine(self, x0, c, uc, scale, S, refine_steps, noise, alphas_cumprod=None):
        """DDIMSampler.refine / _refine (ddim.py:114-168, 339-393) as the latentdiff wrappers call it (eta = 1): re-noise x0 to the
        level of step `refine_steps - 1` of the S-step eta-1 schedule and run the last `refine_steps` stochastic DDIM steps with
        fresh noise.  noise [refine_steps + 1, B, C, h, w]: the x_t draw (ddim.py:349), then one per step (p_sample_ddim)."""
        from .schedule import DDIMSchedule
        assert 0 < refine_steps < S                                   # ddim.py:364
        sched = DDIMSchedule(S, 1.0, S - refine_steps, alphas_cumprod)
        noise = _f32c(noise, self.engine.device)
        assert noise.shape[0] == refine_steps + 1
        xt = self.engine.q_sample(x0, noise[0], sched.sqrt_a_T, sched.sqrt_1ma_T)
        return self.latent_decode(xt.unsqueeze(1).contiguous(), c, uc, scale, sched, extra_noise=noise[1:].contiguous())

    # ---- ensemble members batched along B (per-sample guidance scales; cdx_latent_loop_ens)
    def latent_encode_ens(self, x0, c, uc, scales, sched, n_rec, noise):
        """latent_encode with one guidance scale per sample: scales [B] -> z [B, n_rec+1, C, h, w]."""
        e = self.engine
        x0, c, uc, noise = (_f32c(t, e.device) for t in (x0, c, uc, noise))
        sc = _f32c(torch.as_tensor(scales, dtype=torch.float32), e.device)
        B, Cc, h, w = x0.shape
        assert noise.shape == (n_rec + 1, B, Cc, h, w) and sc.shape == (B,)
        z = e.empty(B, n_rec + 1, Cc, h, w)
        check(lib.cdx_latent_loop_ens(self.h, 1, _ptr(x0), _ptr(c), None, _ptr(uc), c.shape[1], _ptr(sc), None, sched.coef_array(), sched.t_array(),
                                      sched.refine_steps, n_rec, _ptr(noise), sched.sqrt_a_T, sched.sqrt_1ma_T, None, 0, None, _ptr(z), None,
                                      B, Cc, h, w, e.stream))
        return z

    def latent_decode_ens(self, z, c, uc, scales, sched, extra_noise=None):
        """latent_decode with one guidance scale per sample: z [B, n_eps+1, C, h, w], scales [B] -> x0 [B, C, h, w]."""
        e = self.engine
        z, c, uc = (_f32c(t, e.device) for t in (z, c, uc))
        sc = _f32c(torch.as_tensor(scales, dtype=torch.float32), e.device)
        extra_noise = _f32c(extra_noise, e.device) if extra_noise is not None else None
        B, n1, Cc, h, w = z.shape
        assert sc.shape == (B,)
        out = e.empty(B, Cc, h, w)
        check(lib.cdx_latent_loop_ens(self.h, 2, None, None, _ptr(c), _ptr(uc), c.shape[1], None, _ptr(sc), sched.coef_array(), sched.t_array(),
                                      sched.refine_steps, 0, None, 0.0, 0.0, _ptr(z), n1 - 1, _ptr(extra_noise), None, _ptr(out),
                                      B, Cc, h, w, e.stream))
        return out

    def cycle_lockstep(self, x0, c_src, c_tgt, uc, src_scale, tgt_scale, sched, noise, return_z=False):
        """Both chains in one loop (one U-Net call + one fused elementwise kernel per step, no z buffer unless asked for):
        x0 [B,C,h,w] -> translated latent [B,C,h,w] (and z [B, n+1, C,h,w] when return_z).  noise as for latent_encode with
        n_rec == sched.refine_steps."""
        e = self.engine
        x0, c_src, c_tgt, noise = (_f32c(t, e.device) for t in (x0, c_src, c_tgt, noise))
        uc = _f32c(uc, e.device) if uc is not None else None
        B, Cc, h, w = x0.shape
        n = sched.refine_steps
        assert noise.shape == (n + 1, B, Cc, h, w), f'noise shape {tuple(noise.shape)}'
        assert c_src.shape == c_tgt.shape
        out = e.empty(B, Cc, h, w)
        z = e.empty(B, n + 1, Cc, h, w) if return_z else None
        check(lib.cdx_cycle_lockstep(self.h, _ptr(x0), _ptr(c_src), _ptr(c_tgt), _ptr(uc), c_src.shape[1], float(src_scale), float(tgt_scale),
                                     sched.coef_array(), sched.t_array(), n, _ptr(noise), sched.sqrt_a_T, sched.sqrt_1ma_T, _ptr(out), _ptr(z),
                                     B, Cc, h, w, e.stream))
        return (out, z) if return_z else out

    def cycle_lockstep_pair(self, target, x0, c_src, c_tgt, uc, src_scale, tgt_scale, sched, noise, return_z=False):
        """cycle_lockstep with this U-Net on the source chain and `target` (a UNet, possibly on another engine of the same device)
        on the target chain: bit-equal to latent_encode on self followed by latent_decode on target.  Context-free U-Nets pass
        c_src = c_tgt = uc = None."""
        e = self.engine
        x0, noise = _f32c(x0, e.device), _f32c(noise, e.device)
        c_src, c_tgt, uc = (_f32c(t, e.device) if t is not None else None for t in (c_src, c_tgt, uc))
        B, Cc, h, w = x0.shape
        n = sched.refine_steps
        assert noise.shape == (n + 1, B, Cc, h, w), f'noise shape {tuple(noise.shape)}'
        assert (c_src is None) == (c_tgt is None) and (c_src is None or c_src.shape == c_tgt.shape)
        out = e.empty(B, Cc, h, w)
        z = e.empty(B, n + 1, Cc, h, w) if return_z else None
        check(lib.cdx_cycle_lockstep_pair(self.h, target.h, _ptr(x0), _ptr(c_src), _ptr(c_tgt), _ptr(uc), c_src.shape[1] if c_src is not None else 0,
                                          float(src_scale), float(tgt_scale), sched.coef_array(), sched.t_array(), n, _ptr(noise), sched.sqrt_a_T,
                                          sched.sqrt_1ma_T, _ptr(out), _ptr(z), B, Cc, h, w, e.stream))
        return (out, z) if return_z else out

    def pixel_cycle_lockstep(self, target, x0, sched, noise, last_noise, return_z=False):
        """pixel_encode on this U-Net feeding pixel_decode on `target` (a UNet, possibly on another engine of the same device) as one
        loop: two U-Net calls and one fused kernel per step, no z buffer unless asked for.  x0 [B,C,R,R], noise [es_steps, B,C,R,R]
        as for pixel_encode, last_noise [1, B,C,R,R] (or None) as for pixel_decode -> target chain result [B,C,R,R] (and
        z [B, es_steps, C,R,R] when return_z), bit-equal to the two calls."""
        e = self.engine
        x0, noise = _f32c(x0, e.device), _f32c(noise, e.device)
        last_noise = _f32c(last_noise, e.device) if last_noise is not None else None
        B, Cc, R, _ = x0.shape
        n = sched.es_steps
        assert noise.shape == (n, B, Cc, R, R), f'noise shape {tuple(noise.shape)}'
        assert last_noise is None or last_noise.shape == (1, B, Cc, R, R)
        out = e.empty(B, Cc, R, R)
        z = e.empty(B, n, Cc, R, R) if return_z else None
        t = (C.c_float * n)(*sched.t_loop[:n])
        check(lib.cdx_pixel_cycle_lockstep(self.h, target.h, _ptr(x0), sched.coef_array(sched.coef[:n]), t, n, _ptr(noise), sched.sqrt_a_T,
                                           sched.sqrt_1ma_T, _ptr(last_noise), _ptr(out), _ptr(z), B, Cc, R, e.stream))
        return (out, z) if return_z else out

    def pixel_encode(self, x0, sched, noise):
        e = self.engine
        x0, noise = _f32c(x0, e.device), _f32c(noise, e.device)
        B, Cc, R, _ = x0.shape
        n_rec = sched.es_steps - 1
        assert noise.shape == (n_rec + 1, B, Cc, R, R)
        z = e.empty(B, n_rec + 1, Cc, R, R)
        t = (C.c_float * max(n_rec, 1))(*sched.t_loop[:n_rec])
        check(lib.cdx_pixel_encode(self.h, _ptr(x0), sched.coef_array(sched.coef[:n_rec]) if n_rec else None, t, n_rec, _ptr(noise),
                                   sched.sqrt_a_T, sched.sqrt_1ma_T, _ptr(z), B, Cc, R, e.stream))
        return z

    def pixel_decode(self, z, sched, coefs=None, t_loop=None, last_noise=None):
        e = self.engine
        z = _f32c(z, e.device)
        last_noise = _f32c(last_noise, e.device) if last_noise is not None else None
        B, n1, Cc, R, _ = z.shape
        coefs = sched.coef if coefs is None else coefs
        t_loop = sched.t_loop if t_loop is None else t_loop
        out = e.empty(B, Cc, R, R)
        t = (C.c_float * len(t_loop))(*t_loop)
        check(lib.cdx_pixel_decode(self.h, _ptr(z), n1 - 1, sched.coef_array(coefs), t, len(coefs), _ptr(last_noise), _ptr(out), B, Cc,
                                   R, e.stream))
        return out


class VAE(Net):
    """KL-f8 autoencoder (AutoencoderKL)."""

    def __init__(self, engine, cfg):
        self.cfg = dict(cfg)
        c = VaeConfig()
        c.ch, c.n_mult = cfg['ch'], len(cfg['ch_mult'])
        c.ch_mult = _int_arr8(cfg['ch_mult'])
        c.num_res_blocks = cfg['num_res_blocks']
        c.in_channels, c.out_ch = cfg['in_channels'], cfg['out_ch']
        c.z_channels, c.embed_dim = cfg['z_channels'], cfg['embed_dim']
        c.vq, c.n_embed = int(bool(cfg.get('vq', False))), cfg.get('n_embed', 0)
        h = C.c_void_p()
        check(lib.cdx_vae_create(engine.h if engine is not None else None, C.byref(c), C.byref(h)))
        super().__init__(engine, h)
        self.down = 2 ** (len(cfg['ch_mult']) - 1)

    def encode_moments(self, img):
        e = self.engine
        img = _f32c(img, e.device)
        B, _, R, R2 = img.shape
        assert R == R2
        out = e.empty(B, (1 if self.cfg.get('vq') else 2) * self.cfg['embed_dim'], R // self.down, R // self.down)      # vq: h itself
        check(lib.cdx_vae_encode(self.h, _ptr(img), _ptr(out), B, R, e.stream))
        return out

    def decode(self, z):
        e = self.engine
        z = _f32c(z, e.device)
        B, _, h, h2 = z.shape
        assert h == h2
        out = e.empty(B, self.cfg['out_ch'], h * self.down, h * self.down)
        check(lib.cdx_vae_decode(self.h, _ptr(z), _ptr(out), B, h, e.stream))
        return out


class TextEncoder(Net):
    """Text conditioning towers: CLIP (HF CLIPTextModel layout -> last_hidden_state; FrozenCLIPEmbedder,
    ldm/modules/encoders/modules.py:140-158) or, with ``cfg['kind'] == 'xtransformer'``, the LDM BERTEmbedder's in-tree
    encoder (modules.py:79-98, x_transformer.py).  Tokenisation stays on the host (vocabulary files are not part of the engine)."""

    def __init__(self, engine, cfg):
        self.cfg = dict(cfg)
        c = TextConfig()
        c.vocab_size, c.width, c.layers = cfg['vocab_size'], cfg['width'], cfg['layers']
        c.heads, c.max_len, c.mlp_width = cfg['heads'], cfg['max_len'], cfg['mlp_width']
        c.kind = {'clip': 1, 'xtransformer': 2, 'clip_vision': 3}[cfg.get('kind', 'clip')]
        c.dim_head = cfg.get('dim_head', cfg['width'] // cfg['heads'])
        c.proj_dim, c.patch, c.image_size = cfg.get('proj_dim', 0), cfg.get('patch', 0), cfg.get('image_size', 0)
        h = C.c_void_p()
        check(lib.cdx_text_create(engine.h if engine is not None else None, C.byref(c), C.byref(h)))
        super().__init__(engine, h)

    def load_state_dict(self, sd, prefix='', strict=True):
        # older transformers versions register `embeddings.position_ids` as a persistent buffer: not a parameter
        # (and x_transformer's TransformerWrapper carries an unused `to_logits` head)
        sd = {k: v for k, v in sd.items() if not k.endswith('embeddings.position_ids') and '.to_logits.' not in k}
        return super().load_state_dict(sd, prefix, strict)

    def forward(self, input_ids):
        """input_ids [B, L] integer tensor -> [B, L, width] fp32 on the engine's device."""
        e = self.engine
        ids = input_ids.to(device=e.device, dtype=torch.int32).contiguous()
        B, L = ids.shape
        assert L <= self.cfg['max_len'], f'{L} tokens > {self.cfg["max_len"]} positions'
        out = torch.empty(B, L, self.cfg['width'], device=e.device, dtype=torch.float32)
        check(lib.cdx_text_encode(self.h, _ptr(ids), B, L, _ptr(out), e.stream))
        return out

    __call__ = forward

    def features(self, input_ids):
        """CLIP.encode_text: ids [B, L] -> [B, proj_dim] (final-LN state at the EOT token @ text_projection); needs cfg['proj_dim']."""
        e = self.engine
        ids = input_ids.to(device=e.device, dtype=torch.int32).contiguous()
        B, L = ids.shape
        out = torch.empty(B, self.cfg['proj_dim'], device=e.device, dtype=torch.float32)
        check(lib.cdx_text_features(self.h, _ptr(ids), B, L, _ptr(out), e.stream))
        return out


class ClipVision(TextEncoder):
    """CLIP ViT image tower (cfg: width, layers, heads, mlp_width, patch, image_size, proj_dim): CLIP.encode_image."""

    def __init__(self, engine, cfg):
        cfg = dict(cfg, kind='clip_vision', vocab_size=cfg.get('vocab_size', 0), max_len=cfg.get('max_len', 0))
        super().__init__(engine, cfg)

    def forward(self, pixels):
        """pixels [B,3,S,S] (already preprocessed) -> image features [B, proj_dim]."""
        e = self.engine
        x = _f32c(pixels, e.device)
        B, _, S, S2 = x.shape
        assert S == S2 == self.cfg['image_size'], f'{tuple(x.shape)} vs image_size {self.cfg["image_size"]}'
        out = torch.empty(B, self.cfg['proj_dim'], device=e.device, dtype=torch.float32)
        check(lib.cdx_clip_image_features(self.h, _ptr(x), B, _ptr(out), e.stream))
        return out

    __call__ = forward
