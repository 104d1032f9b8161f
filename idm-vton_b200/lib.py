"""ctypes binding of libb200vton.so (include/b200vton.h) plus thin torch-tensor wrappers.

PyTorch is used for device memory and streams only: every wrapper passes `tensor.data_ptr()` and the current CUDA
stream to the C ABI. There is no fallback: if the library is missing or an op fails, a RuntimeError is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200vton.so")

_c = ctypes
_vp, _i, _i64, _f = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float

# name -> argtypes; restype is int for every op. Mirrors include/b200vton.h one to one.
SIGNATURES = {
    "b200vton_gemm_f16": [_vp, _i64, _vp, _i64, _vp, _i64, _i, _i, _i, _vp, _vp, _i64, _vp, _i64, _i, _i, _i, _vp],
    "b200vton_conv3x3_nhwc": [_vp, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _i64, _vp, _i, _vp, _i, _vp, _vp, _vp, _i64,
                              _vp, _i64, _i, _i, _vp],
    "b200vton_attention": [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _f, _i,
                           _vp],
    "b200vton_cross_attention": [_vp, _i64, _vp, _vp, _i64, _i, _vp, _vp, _i64, _i, _vp, _i64, _i, _i, _i, _f, _f, _vp],
    "b200vton_encoder_attention": [_vp, _i64, _vp, _vp, _i64, _vp, _i64, _i, _i, _i, _i, _f, _i, _vp],
    "b200vton_patchify": [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp],
    "b200vton_token_embedding": [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "b200vton_conv3x3_nhwc_f32": [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp],
    "b200vton_split_tf32": [_vp, _i64, _i, _i64, _f, _vp, _vp, _vp],
    "b200vton_softmax_split_tf32": [_vp, _i64, _i, _vp, _vp, _vp],
    "b200vton_groupnorm_nhwc_f32": [_vp, _i, _i, _i, _vp, _vp, _f, _i, _vp, _i64, _vp, _i, _vp],
    "b200vton_conv3x3_nhwc_f16in_f32": [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp],
    "b200vton_groupnorm": [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _f, _i, _vp, _vp, _vp],
    "b200vton_layernorm": [_vp, _i64, _i, _i, _vp, _vp, _f, _vp, _i64, _vp],
    "b200vton_nchw_to_nhwc": [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp],
    "b200vton_nhwc_to_nchw": [_vp, _i, _i, _i, _i, _i, _vp, _vp],
    "b200vton_upsample2x_nhwc": [_vp, _i, _i, _i, _i, _vp, _vp],
    "b200vton_im2col3x3_s2_nhwc": [_vp, _i, _i, _i, _i, _vp, _vp],
    "b200vton_timestep_embedding": [_vp, _i, _i, _i, _vp, _vp],
    "b200vton_skinny_linear": [_vp, _i, _i, _i, _vp, _i64, _i, _vp, _i, _i, _vp, _i, _vp, _i, _vp],
    "b200vton_cfg_ddpm_step": [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp],
    "b200vton_cfg_sched_step": [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp],
    "b200vton_nchw_to_nhwc_scaled": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp],
    "b200vton_preprocess_inpaint": [_vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "b200vton_postprocess_image": [_vp, _i, _i, _i, _i, _vp, _vp, _vp],
}

_lib = None
ABI_VERSION = 107      # must equal b200vton_version() of the loaded library (bumped with every SIGNATURES change)


def load(build_if_missing=True):
    """Load (building first if needed) libb200vton.so and declare every exported symbol. The build runs under an
    exclusive file lock (several ranks may import at once); a library whose sources changed and that cannot be rebuilt,
    or whose ABI version differs from this binding, raises instead of being called with a stale argument layout."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from . import build as _build
        if _build.needs_build():
            import fcntl
            os.makedirs(os.path.join(_HERE, "build"), exist_ok=True)
            with open(os.path.join(_HERE, "build", ".lock"), "w") as lock:
                fcntl.flock(lock, fcntl.LOCK_EX)
                try:
                    _build.build()          # re-checks the source hash under the lock
                finally:
                    fcntl.flock(lock, fcntl.LOCK_UN)
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: the CUDA extension must be built (python idm-vton_b200/build.py); "
                           "there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    lib.b200vton_version.restype = _i
    got = lib.b200vton_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"{LIB_PATH} reports ABI version {got}, this binding expects {ABI_VERSION}: rebuild it "
                           "(python idm-vton_b200/build.py --force)")
    lib.b200vton_last_error.restype = _c.c_char_p
    lib.b200vton_launch_count.restype = _c.c_longlong
    lib.b200vton_set_option.argtypes = [_c.c_char_p, _i]
    lib.b200vton_set_option.restype = _i
    if os.environ.get("B200VTON_GEMM2", "1") == "0":
        lib.b200vton_set_option(b"gemm_2cta_auto", 0)
    if os.environ.get("B200VTON_CLUSTER4", "1") == "0":
        lib.b200vton_set_option(b"gemm_cluster4", 0)
    if os.environ.get("B200VTON_PDL", "0") == "1":
        lib.b200vton_set_option(b"programmatic_launch", 1)
        _options["programmatic_launch"] = 1
    if os.environ.get("B200VTON_ATTN2", "1") == "0":
        lib.b200vton_set_option(b"attention_pingpong", 0)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _i
    _lib = lib
    return lib


_options = {}


def set_option(name, value):
    _check(load().b200vton_set_option(name.encode(), int(value)), "b200vton_set_option")
    _options[name] = int(value)


def get_option(name, default=0):
    """Last value set through set_option / the B200VTON_* environment switches (the C library has no getter)."""
    return _options.get(name, default)


def launch_count():
    """Kernels launched (or captured) by libb200vton.so since load."""
    return int(load().b200vton_launch_count())


def _check(rc, name):
    if rc != 0:
        msg = _lib.b200vton_last_error().decode()
        raise RuntimeError(f"{name} failed (code {rc}): {msg}")


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f16(t, name):
    if t is not None:
        if t.dtype != torch.float16 or not t.is_cuda:
            raise TypeError(f"{name} must be a CUDA fp16 tensor, got {t.dtype} on {t.device}")
    return t


# ------------------------------------------------------------------------------------------------
# op wrappers
# ------------------------------------------------------------------------------------------------
def gemm(a, w, bias=None, residual=None, rowvec=None, rows_per_sample=0, geglu=False, gelu=False, out=None, force_bn=0,
         quick_gelu=False):
    """out[M,N] = epi(a[M,K] @ w[N,K]^T). a / residual / out may be row-strided 2-D views (last dim contiguous)."""
    lib = load()
    _f16(a, "a"); _f16(w, "w")
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K and a.stride(1) == 1 and w.stride(1) == 1
    n_out = N // 2 if geglu else N
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.float16, device=a.device)
    assert out.shape == (M, n_out) and out.stride(1) == 1
    if residual is not None:
        assert residual.shape == (M, n_out) and residual.stride(1) == 1
    rc = lib.b200vton_gemm_f16(_p(a), a.stride(0), _p(w), w.stride(0), _p(out), out.stride(0), M, N, K, _p(bias),
                               _p(residual), residual.stride(0) if residual is not None else 0, _p(rowvec),
                               rowvec.stride(0) if rowvec is not None else 0, rows_per_sample,
                               int(geglu) | (2 if gelu else 0) | (4 if quick_gelu else 0), force_bn,
                               _stream())
    _check(rc, "b200vton_gemm_f16")
    return out


def conv3x3(x, w_packed, bias=None, temb=None, sc0=None, sc1=None, w_sc=None, bias_sc=None, residual=None, out=None,
            force_bn=0, stride=1):
    """x: [B,H,W,Cin] NHWC fp16 (contiguous); w_packed: [9,Cout,Cin]; returns [B,Ho,Wo,Cout] (stride 1 or 2, pad 1)."""
    lib = load()
    _f16(x, "x"); _f16(w_packed, "w_packed")
    B, H, W, Cin = x.shape
    assert x.is_contiguous() and w_packed.is_contiguous() and w_packed.shape[0] == 9 and w_packed.shape[2] == Cin
    Cout = w_packed.shape[1]
    if out is None:
        out = torch.empty((B, (H - 1) // stride + 1, (W - 1) // stride + 1, Cout), dtype=torch.float16, device=x.device)
    C0 = sc0.shape[-1] if sc0 is not None else 0
    C1 = sc1.shape[-1] if sc1 is not None else 0
    rc = lib.b200vton_conv3x3_nhwc(_p(x), Cin, B, H, W, Cin, _p(w_packed), Cout, _p(bias), _p(temb),
                                   temb.stride(0) if temb is not None else 0, _p(sc0), C0, _p(sc1), C1, _p(w_sc),
                                   _p(bias_sc), _p(residual), residual.shape[-1] if residual is not None else 0,
                                   _p(out), out.shape[-1], force_bn, stride, _stream())
    _check(rc, "b200vton_conv3x3_nhwc")
    return out


def attention(q, k0, v0, k1=None, v1=None, n1=0, kv1_off=0, heads=None, scale=None, accumulate=False, out=None,
              kv1_mod=0, kv1_base=None):
    """q: [B,Nq,*], k0/v0: [B,N0,*], k1/v1: [B1,N1,*] 3-D views with contiguous last dim (row strides may exceed
    heads*64, e.g. slices of a fused QKV buffer). n1 > 0 with k1 None => all-zero segment-1 tokens for every sample."""
    lib = load()
    B, Nq = q.shape[0], q.shape[1]
    N0 = k0.shape[1]
    H = heads
    assert q.stride(2) == 1 and k0.stride(2) == 1 and v0.stride(2) == 1
    assert q.stride(0) == Nq * q.stride(1) and k0.stride(0) == N0 * k0.stride(1) and v0.stride() == k0.stride()
    if scale is None:
        scale = 64 ** -0.5
    if out is None:
        out = torch.empty((B, Nq, H * 64), dtype=torch.float16, device=q.device)
    B1 = 0
    ld1 = 0
    if k1 is not None:
        B1, n1 = k1.shape[0], k1.shape[1]
        ld1 = k1.stride(1)
        assert k1.stride(2) == 1 and k1.stride(0) == n1 * ld1 and v1.stride() == k1.stride()
    rc = lib.b200vton_attention(_p(q), q.stride(1), _p(k0), _p(v0), k0.stride(1), _p(k1), _p(v1), ld1, _p(out),
                                out.stride(1), B, H, Nq, N0, n1, B1, kv1_off, kv1_mod, _p(kv1_base), float(scale),
                                int(accumulate), _stream())
    _check(rc, "b200vton_attention")
    return out


def encoder_attention(q, k, v, heads, head_dim, scale=None, causal=False, out=None):
    """CLIP-tower self-attention. q / k / v: [B,N,heads*head_dim] views with contiguous last dim (e.g. the three column
    blocks of a fused QKV buffer); head_dim 16..96, multiple of 16."""
    lib = load()
    _f16(q, "q"); _f16(k, "k"); _f16(v, "v")
    B, N = q.shape[0], q.shape[1]
    assert q.stride(2) == 1 and k.stride(2) == 1 and v.stride() == k.stride() and k.shape[:2] == (B, N)
    assert q.stride(0) == N * q.stride(1) and k.stride(0) == N * k.stride(1)
    if scale is None:
        scale = head_dim ** -0.5
    if out is None:
        out = torch.empty((B, N, heads * head_dim), dtype=torch.float16, device=q.device)
    rc = lib.b200vton_encoder_attention(_p(q), q.stride(1), _p(k), _p(v), k.stride(1), _p(out), out.stride(1), B, heads, N,
                                        head_dim, float(scale), int(causal), _stream())
    _check(rc, "b200vton_encoder_attention")
    return out


def patchify(x, patch, ldk):
    """x: [B,C,H,W] fp16 -> [B*(H/P)*(W/P), ldk] rows of (c, ky, kx), zero-padded to ldk columns."""
    lib = load()
    _f16(x, "x")
    B, C, H, W = x.shape
    assert x.is_contiguous()
    out = torch.empty((B * (H // patch) * (W // patch), ldk), dtype=torch.float16, device=x.device)
    _check(lib.b200vton_patchify(_p(x), B, C, H, W, patch, _p(out), ldk, _stream()), "b200vton_patchify")
    return out


def token_embedding(ids, tok, pos, T):
    """ids: int64 [rows] (rows = B*T); out[r] = fp16(tok[ids[r]] + pos[r % T])."""
    lib = load()
    _f16(tok, "tok"); _f16(pos, "pos")
    assert ids.dtype == torch.int64 and ids.is_cuda and ids.is_contiguous() and tok.is_contiguous() and pos.is_contiguous()
    rows, C = ids.numel(), tok.shape[1]
    out = torch.empty((rows, C), dtype=torch.float16, device=tok.device)
    _check(lib.b200vton_token_embedding(_p(ids), rows, T, C, tok.shape[0], _p(tok), _p(pos), _p(out), _stream()),
           "b200vton_token_embedding")
    return out


def conv3x3_f32_supported(x, cin, cout):
    """Shapes the TF32 convolution kernel covers (everything else stays on the caller's fallback)."""
    return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and cin % 32 == 0 and cout % 32 == 0 and cout >= 64
            and x.shape[3] % 8 == 0)


def pack_conv3x3_f32(weight):
    """[Cout,Cin,3,3] fp32 -> [9,Cout,Cin] (tap-major rows for the kernel's weight map)."""
    return weight.detach().permute(2, 3, 0, 1).reshape(9, weight.shape[0], weight.shape[1]).contiguous()


def conv3x3_f32(x, w_packed, bias=None, residual=None):
    """x: logical [B,Cin,H,W] fp32 (any strides; converted to channels_last = NHWC memory); residual: logical [B,Cout,H,W]
    fp32 or None, added after the bias in the epilogue; returns a channels_last [B,Cout,H,W] fp32 tensor."""
    lib = load()
    B, Cin, H, W = x.shape
    Cout = w_packed.shape[1]
    assert w_packed.dtype == torch.float32 and w_packed.is_contiguous() and w_packed.shape == (9, Cout, Cin)
    x = x.contiguous(memory_format=torch.channels_last)
    if residual is not None:
        assert residual.shape == (B, Cout, H, W) and residual.dtype == torch.float32
        residual = residual.contiguous(memory_format=torch.channels_last)
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    rc = lib.b200vton_conv3x3_nhwc_f32(_p(x), B, H, W, Cin, _p(w_packed), Cout, _p(bias), _p(residual), _p(out), _stream())
    _check(rc, "b200vton_conv3x3_nhwc_f32")
    return out


def split_tf32(x, scale=1.0):
    """x: fp32 [B, ...] whose per-batch block is contiguous (a dense tensor or a row slice x[:, a:b] of a dense [B,N,C] one).
    Returns dense (hi, lo) with hi = tf32(x*scale), lo = tf32(x*scale - hi)."""
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() >= 2
    B = x.shape[0]
    per = x[0].numel()
    if not x[0].is_contiguous():
        x = x.contiguous()
    hi = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    lo = torch.empty_like(hi)
    rc = lib.b200vton_split_tf32(_p(x), x.stride(0) if B > 1 else per, B, per, float(scale), _p(hi), _p(lo), _stream())
    _check(rc, "b200vton_split_tf32")
    return hi, lo


def softmax_split_tf32(scores):
    """scores: dense fp32 [..., N]; returns (p_hi, p_lo), the TF32 parts of softmax(scores, -1)."""
    lib = load()
    assert scores.is_cuda and scores.dtype == torch.float32 and scores.is_contiguous()
    N = scores.shape[-1]
    hi = torch.empty_like(scores)
    lo = torch.empty_like(scores)
    rc = lib.b200vton_softmax_split_tf32(_p(scores), scores.numel() // N, N, _p(hi), _p(lo), _stream())
    _check(rc, "b200vton_softmax_split_tf32")
    return hi, lo


_gn32_ws = {}


def conv3x3_f16in(x16, w_packed16, bias=None, residual=None):
    """x16: logical [B,Cin,H,W] fp16 in channels_last memory (the fp16 output of groupnorm_f32_nhwc); w_packed16: [9,Cout,Cin]
    fp16; bias [Cout] fp32; residual logical [B,Cout,H,W] fp32 or None. Returns a channels_last [B,Cout,H,W] fp32 tensor."""
    lib = load()
    B, Cin, H, W = x16.shape
    Cout = w_packed16.shape[1]
    assert x16.dtype == torch.float16 and x16.is_contiguous(memory_format=torch.channels_last)
    assert w_packed16.dtype == torch.float16 and w_packed16.is_contiguous() and w_packed16.shape == (9, Cout, Cin)
    if residual is not None:
        assert residual.shape == (B, Cout, H, W) and residual.dtype == torch.float32
        residual = residual.contiguous(memory_format=torch.channels_last)
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=x16.device, memory_format=torch.channels_last)
    rc = lib.b200vton_conv3x3_nhwc_f16in_f32(_p(x16), B, H, W, Cin, _p(w_packed16), Cout, _p(bias), _p(residual), _p(out),
                                             _stream())
    _check(rc, "b200vton_conv3x3_nhwc_f16in_f32")
    return out


def groupnorm_f32_nhwc(x, gamma, beta, eps, silu, out_half=False):
    """x: logical [B,C,H,W] fp32 in channels_last memory (= dense NHWC); returns the same layout, fp32 or (out_half) fp16."""
    lib = load()
    B, C, H, W = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous(memory_format=torch.channels_last)
    key = (x.device, torch.cuda.current_stream().cuda_stream)
    ws = _gn32_ws.get(key)
    need = 64 * max(B, 1184)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.float64, device=x.device)
        _gn32_ws[key] = ws
    out = torch.empty(x.shape, dtype=torch.float16 if out_half else torch.float32, device=x.device,
                      memory_format=torch.channels_last)
    rc = lib.b200vton_groupnorm_nhwc_f32(_p(x), B, H * W, C, _p(gamma), _p(beta), float(eps), int(silu), _p(ws),
                                         ws.numel(), _p(out), int(out_half), _stream())
    _check(rc, "b200vton_groupnorm_nhwc_f32")
    return out


def cross_attention(q, kt, vt, ki=None, vi=None, heads=None, scale=None, ip_scale=1.0, out=None):
    """Text (+ IP-Adapter image token) cross-attention in one launch. q: [B,Nq,*]; kt/vt: [B,Nt<=80,*]; ki/vi:
    [B,Ni<=16,*] or None. 3-D views with contiguous last dim (slices of fused [K|V] buffers are fine)."""
    lib = load()
    B, Nq = q.shape[0], q.shape[1]
    H = heads
    Nt = kt.shape[1]
    assert q.stride(2) == 1 and kt.stride(2) == 1 and vt.stride() == kt.stride() and kt.shape[0] == B
    assert q.stride(0) == Nq * q.stride(1) and kt.stride(0) == Nt * kt.stride(1)
    if scale is None:
        scale = 64 ** -0.5
    if out is None:
        out = torch.empty(B, Nq, H * 64, dtype=torch.float16, device=q.device)
    assert out.stride(2) == 1 and out.stride(0) == Nq * out.stride(1)
    Ni, ldi = 0, 0
    if ki is not None:
        Ni, ldi = ki.shape[1], ki.stride(1)
        assert ki.stride(2) == 1 and vi.stride() == ki.stride() and ki.shape[0] == B and ki.stride(0) == Ni * ldi
    rc = lib.b200vton_cross_attention(_p(q), q.stride(1), _p(kt), _p(vt), kt.stride(1), Nt, _p(ki), _p(vi), ldi, Ni,
                                      _p(out), out.stride(1), B, H, Nq, float(scale), float(ip_scale), _stream())
    _check(rc, "b200vton_cross_attention")
    return out


_gn_ws = {}


GN_BARRIER_DOUBLES = 4096      # 8 bytes of barrier state per sample, up to 4096 samples (include/b200vton.h)


def _stats_ws(device, B):
    """GroupNorm workspace: max(B,296)*64 doubles of partial sums followed by the per-sample barrier state, which must be
    ZERO before first use (the kernel leaves it reusable), hence torch.zeros."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _gn_ws.get(key)
    if ws is None or ws.numel() < max(B, 296) * 64 + GN_BARRIER_DOUBLES:
        ws = torch.zeros(max(B, 296) * 64 + GN_BARRIER_DOUBLES, dtype=torch.float64, device=device)
        _gn_ws[key] = ws
    return ws


def groupnorm(x0, gamma, beta, eps, silu, x1=None, out=None, ws=None):
    """x0: [B,HW,C0] (or [B,H,W,C0]) contiguous, optional x1 [B,HW,C1]: GroupNorm(32) over the channel concat."""
    lib = load()
    B = x0.shape[0]
    C0 = x0.shape[-1]
    HW = x0.numel() // (B * C0)
    C1 = x1.shape[-1] if x1 is not None else 0
    assert x0.is_contiguous() and (x1 is None or x1.is_contiguous())
    if out is None:
        out = torch.empty(x0.shape[:-1] + (C0 + C1,), dtype=torch.float16, device=x0.device)
    if ws is None:
        ws = _stats_ws(x0.device, B)
    rc = lib.b200vton_groupnorm(_p(x0), C0, _p(x1), C1, B, HW, _p(gamma), _p(beta), float(eps), int(silu), _p(ws),
                                _p(out), _stream())
    _check(rc, "b200vton_groupnorm")
    return out


def layernorm(x, gamma, beta, eps=1e-5, out=None):
    lib = load()
    C = x.shape[-1]
    x2 = x.reshape(-1, C)
    assert x2.stride(1) == 1
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    o2 = out.reshape(-1, C)
    rc = lib.b200vton_layernorm(_p(x2), x2.stride(0), x2.shape[0], C, _p(gamma), _p(beta), float(eps), _p(o2),
                                o2.stride(0), _stream())
    _check(rc, "b200vton_layernorm")
    return out


def nchw_to_nhwc(src, dst, c_off=0):
    """dst[s,y,x,c_off+c] = src[s % Bs, c, y, x]; dst: [Bd,H,W,ldc] contiguous."""
    lib = load()
    Bs, Cs, H, W = src.shape
    assert src.is_contiguous() and dst.is_contiguous()
    rc = lib.b200vton_nchw_to_nhwc(_p(src), Bs, Cs, H, W, _p(dst), dst.shape[0], dst.shape[-1], c_off, _stream())
    _check(rc, "b200vton_nchw_to_nhwc")
    return dst


def nchw_to_nhwc_scaled(src, dst, scale, c_off=0):
    """dst[s,y,x,c_off+c] = fp16(src[s % Bs, c, y, x] * scale[0]); scale: fp32 CUDA tensor (one element read)."""
    lib = load()
    Bs, Cs, H, W = src.shape
    assert src.is_contiguous() and dst.is_contiguous()
    assert scale.dtype == torch.float32 and scale.is_cuda and scale.numel() >= 1
    rc = lib.b200vton_nchw_to_nhwc_scaled(_p(src), Bs, Cs, H, W, _p(scale), _p(dst), dst.shape[0], dst.shape[-1], c_off,
                                          _stream())
    _check(rc, "b200vton_nchw_to_nhwc_scaled")
    return dst


def nhwc_to_nchw(src, C, out=None):
    lib = load()
    B, H, W, ldc = src.shape
    if out is None:
        out = torch.empty((B, C, H, W), dtype=torch.float16, device=src.device)
    rc = lib.b200vton_nhwc_to_nchw(_p(src), B, C, H, W, ldc, _p(out), _stream())
    _check(rc, "b200vton_nhwc_to_nchw")
    return out


def upsample2x(x, out=None):
    lib = load()
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, 2 * H, 2 * W, C), dtype=torch.float16, device=x.device)
    rc = lib.b200vton_upsample2x_nhwc(_p(x), B, H, W, C, _p(out), _stream())
    _check(rc, "b200vton_upsample2x_nhwc")
    return out


def im2col3x3_s2(x, out=None):
    lib = load()
    B, H, W, C = x.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if out is None:
        out = torch.empty((B * Ho * Wo, 9 * C), dtype=torch.float16, device=x.device)
    rc = lib.b200vton_im2col3x3_s2_nhwc(_p(x), B, H, W, C, _p(out), _stream())
    _check(rc, "b200vton_im2col3x3_s2_nhwc")
    return out


def timestep_embedding(values, dim, rows_repeat=1, out=None):
    """values: fp32 CUDA tensor [n]; returns [n*rows_repeat, dim] fp16 ([cos|sin])."""
    lib = load()
    assert values.dtype == torch.float32 and values.is_cuda
    n = values.numel()
    if out is None:
        out = torch.empty((n * rows_repeat, dim), dtype=torch.float16, device=values.device)
    rc = lib.b200vton_timestep_embedding(_p(values), n, dim, rows_repeat, _p(out), _stream())
    _check(rc, "b200vton_timestep_embedding")
    return out


def skinny_linear(x, w, bias=None, in_silu=False, out_silu=False, addend=None, out=None):
    lib = load()
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float16, device=x.device)
    rc = lib.b200vton_skinny_linear(_p(x), x.stride(0), M, K, _p(w), w.stride(0), N, _p(bias), int(in_silu),
                                    int(out_silu), _p(addend), addend.stride(0) if addend is not None else 0, _p(out),
                                    out.stride(0), _stream())
    _check(rc, "b200vton_skinny_linear")
    return out


def cfg_ddpm_step(eps, latents, noise, coef, do_cfg=True, out=None):
    """eps: [2B,H,W,ldc] NHWC (or [B,...] without CFG); latents/noise: [B,C,H,W]; coef: 6 fp32 on device."""
    lib = load()
    B, C, H, W = latents.shape
    if out is None:
        out = torch.empty_like(latents)
    rc = lib.b200vton_cfg_ddpm_step(_p(eps), eps.shape[-1], B, C, H, W, _p(latents), _p(noise), _p(coef), int(do_cfg),
                                    _p(out), _stream())
    _check(rc, "b200vton_cfg_ddpm_step")
    return out


SCHED_FAMILIES = {"ddim": 0, "euler": 1, "euler_ancestral": 2, "dpmsolver++": 3}


def cfg_sched_step(eps, latents, noise, hist, coef, family, do_cfg=True, out=None):
    """Fused CFG + scheduler update (csrc/sched.cu). eps: [2B,H,W,ldc] NHWC (or [B,...] without CFG); latents / noise /
    hist: [B,C,H,W] fp16 (noise / hist may be None where the family does not read them; hist is updated in place);
    coef: 8 fp32 on device; family: a key of SCHED_FAMILIES."""
    lib = load()
    B, C, H, W = latents.shape
    if out is None:
        out = torch.empty_like(latents)
    rc = lib.b200vton_cfg_sched_step(_p(eps), eps.shape[-1], B, C, H, W, _p(latents), _p(noise), _p(hist), _p(coef),
                                     SCHED_FAMILIES[family], int(do_cfg), _p(out), _stream())
    _check(rc, "b200vton_cfg_sched_step")
    return out


def preprocess_inpaint(image, mask, vae_scale=8):
    """image [B,3,H,W] fp32 CUDA in [0,1] (or already [-1,1]), mask [B,1|3,H,W] fp32 -> (init_image, mask_bin, masked_image,
    mask_latent fp16 [B,1,H/s,W/s]); one launch, no host sync."""
    lib = load()
    B, _, H, W = image.shape
    assert image.is_cuda and image.dtype == torch.float32 and mask.dtype == torch.float32 and mask.shape[0] == B
    assert mask.shape[-2:] == image.shape[-2:] and image.is_contiguous() and mask.is_contiguous()
    img_min = image.amin().reshape(1)
    init = torch.empty_like(image)
    masked = torch.empty_like(image)
    mbin = torch.empty((B, 1, H, W), dtype=torch.float32, device=image.device)
    mlat = torch.empty((B, 1, H // vae_scale, W // vae_scale), dtype=torch.float16, device=image.device)
    rc = lib.b200vton_preprocess_inpaint(_p(image), _p(mask), mask.shape[1], _p(img_min), B, H, W, vae_scale, _p(init),
                                         _p(mbin), _p(masked), _p(mlat), _stream())
    _check(rc, "b200vton_preprocess_inpaint")
    return init, mbin, masked, mlat


def postprocess_image(x, want_pt=True, want_u8=False):
    """x: logical [B,3,H,W] fp32 CUDA, contiguous either as NCHW or as channels_last (NHWC memory). Returns
    (fp32 NCHW in [0,1] or None, uint8 NHWC or None)."""
    lib = load()
    B, C, H, W = x.shape
    assert C == 3 and x.is_cuda and x.dtype == torch.float32
    nhwc = 0
    if not x.is_contiguous():
        if x.is_contiguous(memory_format=torch.channels_last):
            nhwc = 1
        else:
            x = x.contiguous()
    pt = torch.empty((B, 3, H, W), dtype=torch.float32, device=x.device) if want_pt else None
    u8 = torch.empty((B, H, W, 3), dtype=torch.uint8, device=x.device) if want_u8 else None
    rc = lib.b200vton_postprocess_image(_p(x), nhwc, B, H, W, _p(pt), _p(u8), _stream())
    _check(rc, "b200vton_postprocess_image")
    return pt, u8
