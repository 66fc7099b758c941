"""ctypes binding of the C-ABI kernel library (``libpfd_b200.so``, see ``include/pfd_b200.h``).

This is the *only* way compute reaches the GPU in this package: there is no torch / CPU fallback.
If the shared library is missing or a call fails, a ``RuntimeError`` is raised.

Tensors are torch CUDA fp16 tensors used purely as device-memory handles (``data_ptr()``); the
stream is torch's current stream so calls can be captured into CUDA graphs.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_void_p
from typing import Optional, Sequence, Tuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# PFD_B200_LIB: load another build of the same ABI (A/B runs of compile-time variants); default = the in-tree library
LIB_PATH = os.environ.get("PFD_B200_LIB") or os.path.join(_HERE, "libpfd_b200.so")

PFD_MAX_SEG = 3
ACT_NONE, ACT_SILU, ACT_GELU, ACT_RELU, ACT_GEGLU = 0, 1, 2, 3, 4

EXPORTS = [
    "pfd_version", "pfd_last_error", "pfd_launch_count", "pfd_set_option", "pfd_gemm_f16", "pfd_groupnorm_f16",
    "pfd_layernorm_f16", "pfd_softmax_f16", "pfd_timestep_embedding_f16", "pfd_upsample2x_f16",
    "pfd_nchw_to_nhwc_f16", "pfd_nhwc_to_nchw_f16", "pfd_im2col3x3_f16", "pfd_axpby_f16",
    "pfd_add_rowvec_f16", "pfd_ddim_step_f16", "pfd_window_gather_f16", "pfd_window_scatter_f16",
    "pfd_patch_merge_gather_f16", "pfd_patchify_f16", "pfd_flash_attn_f16",
    "pfd_flash_attn_strided_f16", "pfd_ddim_begin_step", "pfd_vae_posterior_f16",
    "pfd_canny_workspace_bytes", "pfd_canny_f32", "pfd_image_u8_roundtrip_f32", "pfd_hed_input_f16",
    "pfd_maxpool2x2_f16", "pfd_hed_project_f32", "pfd_hed_fuse_f32",
]
PFD_HED_MAPS = 5


class GemmDesc(ctypes.Structure):
    """Mirror of ``pfd_gemm_desc`` (include/pfd_b200.h)."""
    _fields_ = [
        ("nseg", c_int32),
        ("taps", c_int32 * PFD_MAX_SEG),
        ("a_c", c_int32 * PFD_MAX_SEG),
        ("a_ptr", c_void_p * PFD_MAX_SEG),
        ("a_sx", c_int64 * PFD_MAX_SEG),
        ("a_sy", c_int64 * PFD_MAX_SEG),
        ("a_sn", c_int64 * PFD_MAX_SEG),
        ("in_w", c_int32), ("in_h", c_int32),
        ("stride", c_int32),
        ("W", c_int32), ("H", c_int32), ("NB", c_int32),
        ("b_ptr", c_void_p),
        ("N", c_int32),
        ("K", c_int64),
        ("b_batch_stride", c_int64),
        ("alpha", c_float),
        ("act", c_int32),
        ("bias", c_void_p),
        ("rowadd", c_void_p),
        ("rowadd_ld", c_int64),
        ("residual", c_void_p),
        ("out", c_void_p),
        ("so_n1", c_int64), ("so_n0", c_int64), ("so_y", c_int64), ("so_x", c_int64),
        ("so_c1", c_int64), ("so_c0", c_int64),
        ("ndiv", c_int32), ("cdiv", c_int32),
        ("bn_force", c_int32),
        ("tap_off", c_int32),
        ("stream", c_void_p),
    ]


_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once). Raises if it has not been built (``__graft_entry__.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU/PyTorch fallback for the pfd_b200 kernels)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.pfd_version.restype = c_int32
    lib.pfd_last_error.restype = c_char_p
    lib.pfd_launch_count.restype = c_int64
    lib.pfd_set_option.argtypes = [c_char_p, c_int32]
    lib.pfd_gemm_f16.argtypes = [POINTER(GemmDesc)]
    lib.pfd_groupnorm_f16.argtypes = [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int64, c_int32,
                                      c_void_p, c_void_p, c_float, c_int32, c_void_p, c_void_p, c_int32, c_void_p]
    lib.pfd_layernorm_f16.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_float,
                                      c_void_p, c_void_p]
    lib.pfd_softmax_f16.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_int64, c_float, c_void_p,
                                    c_int32, c_void_p, c_int32, c_void_p]
    lib.pfd_timestep_embedding_f16.argtypes = [c_void_p, c_int32, c_int32, c_float, c_void_p, c_void_p]
    lib.pfd_upsample2x_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    lib.pfd_nchw_to_nhwc_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                         c_float, c_float, c_void_p, c_void_p]
    lib.pfd_vae_posterior_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_float,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.pfd_nhwc_to_nchw_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_float,
                                         c_float, c_float, c_float, c_void_p, c_void_p]
    lib.pfd_im2col3x3_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                      c_void_p, c_void_p]
    lib.pfd_axpby_f16.argtypes = [c_void_p, c_float, c_void_p, c_float, c_int64, c_void_p, c_void_p]
    lib.pfd_add_rowvec_f16.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]
    lib.pfd_ddim_step_f16.argtypes = [c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.pfd_window_gather_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                          c_void_p, c_void_p]
    lib.pfd_window_scatter_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                           c_void_p, c_void_p, c_void_p]
    lib.pfd_patch_merge_gather_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                               c_void_p]
    lib.pfd_patchify_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                     c_void_p, c_void_p]
    if True:
        lib.pfd_flash_attn_f16.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                           c_int32, c_int32, c_int32, c_int32, c_int32, c_float,
                                           c_int64, c_int64, c_int64, c_int32, c_void_p]
    lib.pfd_flash_attn_strided_f16.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                               c_int32, c_int32, POINTER(c_int64), POINTER(c_int64),
                                               POINTER(c_int64), c_float, c_int64, c_int64, c_void_p]
    lib.pfd_ddim_begin_step.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_void_p]
    lib.pfd_canny_workspace_bytes.argtypes = [c_int32, c_int32, c_int32]
    lib.pfd_canny_workspace_bytes.restype = c_int64
    lib.pfd_canny_f32.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                  POINTER(c_int32), c_void_p]
    lib.pfd_image_u8_roundtrip_f32.argtypes = [c_void_p, c_int32, c_int64, c_void_p, c_void_p]
    lib.pfd_hed_input_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_float, c_void_p,
                                      c_void_p]
    lib.pfd_maxpool2x2_f16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    lib.pfd_hed_project_f32.argtypes = [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_float, c_void_p, c_void_p]
    lib.pfd_hed_fuse_f32.argtypes = [POINTER(c_void_p), POINTER(c_int32), POINTER(c_int32), c_int32, c_int32, c_int32,
                                     c_void_p, c_void_p, c_void_p]
    for name in EXPORTS:
        if hasattr(lib, name) and name not in ("pfd_version", "pfd_last_error", "pfd_launch_count",
                                               "pfd_canny_workspace_bytes"):
            getattr(lib, name).restype = c_int32
    _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pfd_last_error()
        raise RuntimeError(f"{what} failed: {msg.decode() if msg else rc}")


def set_env_option(name: Optional[str], value) -> None:
    """Library tuning switch (pfd_set_option); name=None resets every switch to its default."""
    _check(load().pfd_set_option(None if name is None else name.encode(), 0 if value is None else int(value)),
           "pfd_set_option")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


_replayed = 0


def note_replay(n: int) -> None:
    """Account for kernels re-launched by a CUDA-graph replay (they bypass the library's counter)."""
    global _replayed
    _replayed += int(n)


def launch_count() -> int:
    """Kernels launched by this library in this process (direct launches + graph-replayed ones)."""
    return int(load().pfd_launch_count()) + _replayed


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    return t.data_ptr()


def _chk16(t: torch.Tensor, name: str) -> None:
    if t.dtype != torch.float16 or not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA fp16 tensor, got {t.dtype} on {t.device}")


# --------------------------------------------------------------------------------------------
# GEMM family
# --------------------------------------------------------------------------------------------
def gemm_raw(segs: Sequence[Tuple[torch.Tensor, int, int, Tuple[int, int, int]]], *, in_w: int,
             in_h: int, stride: int, W: int, H: int, NB: int, w: torch.Tensor, N: int, K: int,
             b_batch_stride: int = 0, alpha: float = 1.0, act: int = ACT_NONE,
             bias: Optional[torch.Tensor] = None, rowadd: Optional[torch.Tensor] = None,
             residual: Optional[torch.Tensor] = None, out: torch.Tensor,
             so: Tuple[int, int, int, int, int, int], ndiv: int = 1, cdiv: int = 0,
             bn_force: int = 0, tap_off: int = 0) -> None:
    """Lowest-level call: ``segs`` is a list of (tensor, taps, channels, (sx, sy, sn))."""
    d = GemmDesc()
    d.nseg = len(segs)
    for i, (t, taps, c, (sx, sy, sn)) in enumerate(segs):
        _chk16(t, f"A[{i}]")
        d.taps[i] = taps
        d.a_c[i] = c
        d.a_ptr[i] = t.data_ptr()
        d.a_sx[i], d.a_sy[i], d.a_sn[i] = sx, sy, sn
    d.in_w, d.in_h, d.stride = in_w, in_h, stride
    d.W, d.H, d.NB = W, H, NB
    _chk16(w, "B")
    d.b_ptr = w.data_ptr()
    d.N, d.K, d.b_batch_stride = N, K, b_batch_stride
    d.alpha, d.act = alpha, act
    d.bias = _p(bias)
    d.rowadd = _p(rowadd)
    d.rowadd_ld = rowadd.stride(0) if rowadd is not None else 0
    d.residual = _p(residual)
    d.out = out.data_ptr()
    d.so_n1, d.so_n0, d.so_y, d.so_x, d.so_c1, d.so_c0 = so
    d.ndiv, d.cdiv = ndiv, cdiv
    d.bn_force = bn_force
    d.tap_off = tap_off
    d.stream = stream_ptr()
    _check(load().pfd_gemm_f16(ctypes.byref(d)), "pfd_gemm_f16")


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = ACT_NONE,
           residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
           alpha: float = 1.0, x2: Optional[torch.Tensor] = None, bn_force: int = 0) -> torch.Tensor:
    """out[M, N] = act(alpha * [x | x2] @ w^T + bias) + residual.  x: [M, K1] (row pitch = stride(0)),
    optional x2: [M, K2]; w: [N, K1+K2] (GEGLU: tile-packed, output has N/2 columns)."""
    M, K1 = x.shape
    N = w.shape[0]
    n_out = N // 2 if act == ACT_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=x.device, dtype=torch.float16)
    segs = [(x, 1, K1, (x.stride(0), x.stride(0) * M, x.stride(0) * M))]
    if x2 is not None:
        segs.append((x2, 1, x2.shape[1], (x2.stride(0), x2.stride(0) * M, x2.stride(0) * M)))
    ldo = out.stride(0)
    gemm_raw(segs, in_w=M, in_h=1, stride=1, W=M, H=1, NB=1, w=w, N=N, K=w.stride(0), alpha=alpha,
             act=act, bias=bias, residual=residual, out=out, so=(0, 0, 0, ldo, 0, 1), bn_force=bn_force)
    return out


def geglu_tile(n2: int) -> int:
    """N-tile width used for a GEGLU projection with 2*inner = n2 output features."""
    for bn in (160, 256, 128, 192, 64):
        if n2 % bn == 0:
            return bn
    raise RuntimeError(f"GEGLU width {n2} is not divisible by any supported N tile")


def pack_geglu(w: torch.Tensor, b: Optional[torch.Tensor]):
    """Re-order GEGLU.proj rows (attention.py:47-51: first half = value, second half = gate) so every
    N tile holds [value(bn/2) | gate(bn/2)] for the same output columns. Returns (w, b, bn)."""
    n2 = w.shape[0]
    inner = n2 // 2
    bn = geglu_tile(n2)
    h = bn // 2
    idx = torch.arange(n2, device=w.device).reshape(n2 // bn, 2, h)
    tile = torch.arange(n2 // bn, device=w.device).reshape(-1, 1)
    j = torch.arange(h, device=w.device).reshape(1, -1)
    src = torch.stack([tile * h + j, inner + tile * h + j], dim=1).reshape(-1)
    wp = w.index_select(0, src).contiguous()
    bp = b.index_select(0, src).contiguous() if b is not None else None
    return wp, bp, bn


def conv3x3(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, stride: int = 1,
            rowadd: Optional[torch.Tensor] = None, act: int = ACT_NONE,
            residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
            skip: Sequence[torch.Tensor] = (), tap_off: int = 0) -> torch.Tensor:
    """3x3 / pad 1 convolution on channel-last x [NB, H, W, C] with packed weights
    w [Cout, 9*C (+ sum of skip channels)] (k = tap*C + c, then the 1x1 skip-segment channels).
    ``skip`` tensors (same raster, stride 1 only) are extra 1x1 K-segments accumulated into the same
    output — used to fuse ResBlock.skip_connection(x) (openaimodel.py:240,274) into out_layers' conv."""
    NB, H, W, C = x.shape
    # padding (1 - tap_off) on the top/left, 1 on the bottom/right: tap_off = 1 is F.pad(x, (0,1,0,1)) + padding 0
    Ho, Wo = (H - 1 - tap_off) // stride + 1, (W - 1 - tap_off) // stride + 1
    N = w.shape[0]
    if out is None:
        out = torch.empty((NB, Ho, Wo, N), device=x.device, dtype=torch.float16)
    segs = [(x, 9, C, (x.stride(2), x.stride(1), x.stride(0)))]
    for s in skip:
        segs.append((s, 1, s.shape[3], (s.stride(2), s.stride(1), s.stride(0))))
    gemm_raw(segs, in_w=W, in_h=H, stride=stride, W=Wo, H=Ho, NB=NB, w=w, N=N, K=w.stride(0), act=act,
             bias=bias, rowadd=rowadd, residual=residual, out=out,
             so=(out.stride(0), 0, out.stride(1), out.stride(2), 0, 1), tap_off=tap_off)
    return out


def conv1x1(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *, act: int = ACT_NONE,
            residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
            x2: Optional[torch.Tensor] = None) -> torch.Tensor:
    """1x1 conv on channel-last tensors == linear over flattened pixels."""
    NB, H, W, C = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((NB, H, W, N), device=x.device, dtype=torch.float16)
    r = residual.reshape(NB * H * W, -1) if residual is not None else None
    linear(x.reshape(NB * H * W, C), w, bias, act=act, residual=r, out=out.reshape(NB * H * W, N),
           x2=None if x2 is None else x2.reshape(NB * H * W, -1))
    return out


def bmm_nt(a: torch.Tensor, b: torch.Tensor, *, out: torch.Tensor, so, ndiv: int = 1, cdiv: int = 0,
           alpha: float = 1.0) -> None:
    """Batched out[b] = a[b] @ b[b]^T.  a: [B, M, K] contiguous-in-K, b: [B, N, K]; generic out strides."""
    B, M, K = a.shape
    N = b.shape[1]
    gemm_raw([(a, 1, K, (a.stride(1), a.stride(1) * M, a.stride(0)))], in_w=M, in_h=1, stride=1, W=M,
             H=1, NB=B, w=b, N=N, K=b.stride(1), b_batch_stride=b.stride(0), alpha=alpha, out=out,
             so=so, ndiv=ndiv, cdiv=cdiv)


# --------------------------------------------------------------------------------------------
# normalisation / softmax / misc
# --------------------------------------------------------------------------------------------
# GroupNorm statistics scratch: a ring of pre-zeroed slots per (device, stream).  `gn_reset()` zeroes the
# whole ring with ONE memset (called at the start of every network evaluation); each groupnorm() call then
# takes the next slot without a memset of its own.  If the ring is exhausted the call zeroes a fallback slot itself.
_GN_SLOT_BYTES = 64 * 32 * 16 + 256    # up to 64 images x 32 groups x (sum, sumsq) fp64 (+ spare)
_GN_SLOTS = 256
_gn_rings = {}


def _gn_ring():
    key = (torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    ring = _gn_rings.get(key)
    if ring is None:
        buf = torch.zeros(_GN_SLOT_BYTES * (_GN_SLOTS + 1), device="cuda", dtype=torch.uint8)   # + 1 fallback slot
        ring = {"buf": buf, "next": _GN_SLOTS}      # exhausted until the first gn_reset()
        _gn_rings[key] = ring
    return ring


def gn_reset() -> None:
    """Zero all GroupNorm scratch slots of the current stream (one memset) and rewind the ring."""
    ring = _gn_ring()
    ring["buf"].zero_()
    ring["next"] = 0


def groupnorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, *, silu: bool,
              x2: Optional[torch.Tensor] = None, groups: int = 32,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(+SiLU) over channel-last x [NB, H, W, C1] (optionally concatenated with x2 [.., C2])."""
    NB, H, W, C1 = x.shape
    C2 = x2.shape[3] if x2 is not None else 0
    if out is None:
        out = torch.empty((NB, H, W, C1 + C2), device=x.device, dtype=torch.float16)
    ring = _gn_ring()
    need = NB * groups * 16 + NB * 4
    if ring["next"] < _GN_SLOTS and need <= _GN_SLOT_BYTES:
        ws_ptr, zero = ring["buf"].data_ptr() + ring["next"] * _GN_SLOT_BYTES, 0
        ring["next"] += 1
    else:
        if need > _GN_SLOT_BYTES:
            raise RuntimeError("groupnorm: batch too large for the statistics scratch")
        ws_ptr, zero = ring["buf"].data_ptr() + _GN_SLOTS * _GN_SLOT_BYTES, 1    # shared fallback slot, zeroed per call
        ring["next"] = _GN_SLOTS
    _check(load().pfd_groupnorm_f16(x.data_ptr(), C1, _p(x2), C2, NB, H * W, groups, gamma.data_ptr(),
                                    beta.data_ptr(), eps, int(silu), out.data_ptr(), ws_ptr, zero, stream_ptr()),
           "pfd_groupnorm_f16")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, *,
              residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    C = x.shape[-1]
    rows = x.numel() // C
    if out is None:
        out = torch.empty_like(x)
    _check(load().pfd_layernorm_f16(x.data_ptr(), _p(residual), rows, C, gamma.data_ptr(), beta.data_ptr(),
                                    eps, out.data_ptr(), stream_ptr()), "pfd_layernorm_f16")
    return out


def softmax_(s: torch.Tensor, scale: float, *, bias: Optional[torch.Tensor] = None, nheads: int = 1,
             mask: Optional[torch.Tensor] = None, nwin: int = 1) -> torch.Tensor:
    """In-place row softmax over s [batch, rows, cols] (see pfd_softmax_f16)."""
    batch, rows, cols = s.shape
    _check(load().pfd_softmax_f16(s.data_ptr(), batch, rows, cols, s.stride(1), scale, _p(bias), nheads,
                                  _p(mask), nwin, stream_ptr()), "pfd_softmax_f16")
    return s


def timestep_embedding(t: torch.Tensor, dim: int, max_period: float = 10000.0) -> torch.Tensor:
    out = torch.empty((t.shape[0], dim), device=t.device, dtype=torch.float16)
    _check(load().pfd_timestep_embedding_f16(t.data_ptr(), t.shape[0], dim, max_period, out.data_ptr(),
                                             stream_ptr()), "pfd_timestep_embedding_f16")
    return out


def upsample2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    NB, H, W, C = x.shape
    if out is None:
        out = torch.empty((NB, 2 * H, 2 * W, C), device=x.device, dtype=torch.float16)
    _check(load().pfd_upsample2x_f16(x.data_ptr(), NB, H, W, C, out.data_ptr(), stream_ptr()),
           "pfd_upsample2x_f16")
    return out


def nchw_to_nhwc(x: torch.Tensor, cpad: Optional[int] = None, out: Optional[torch.Tensor] = None, *,
                 mul: float = 1.0, add: float = 0.0) -> torch.Tensor:
    NB, C, H, W = x.shape
    cpad = cpad or C
    x = x.contiguous()
    if out is None:
        out = torch.empty((NB, H, W, cpad), device=x.device, dtype=torch.float16)
    if x.dtype not in (torch.float16, torch.float32):
        raise RuntimeError(f"nchw_to_nhwc: unsupported dtype {x.dtype}")
    _check(load().pfd_nchw_to_nhwc_f16(x.data_ptr(), int(x.dtype == torch.float32), NB, C, H, W, cpad, mul, add,
                                       out.data_ptr(), stream_ptr()), "pfd_nchw_to_nhwc_f16")
    return out


def nhwc_to_nchw(x: torch.Tensor, C: Optional[int] = None, *, mul: float = 1.0, add: float = 0.0,
                 lo: float = -65504.0, hi: float = 65504.0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    NB, H, W, Cpad = x.shape
    C = C or Cpad
    if out is None:
        out = torch.empty((NB, C, H, W), device=x.device, dtype=torch.float16)
    _check(load().pfd_nhwc_to_nchw_f16(x.data_ptr(), NB, C, H, W, Cpad, mul, add, lo, hi, out.data_ptr(),
                                       stream_ptr()), "pfd_nhwc_to_nchw_f16")
    return out


def im2col3x3(x: torch.Tensor, kpad: int, stride: int = 1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    NB, H, W, C = x.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((NB, Ho, Wo, kpad), device=x.device, dtype=torch.float16)
    _check(load().pfd_im2col3x3_f16(x.data_ptr(), NB, H, W, C, stride, kpad, out.data_ptr(), stream_ptr()),
           "pfd_im2col3x3_f16")
    return out


def axpby(a: torch.Tensor, sa: float, b: Optional[torch.Tensor] = None, sb: float = 0.0,
          out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(a)
    _check(load().pfd_axpby_f16(a.data_ptr(), sa, _p(b), sb, a.numel(), out.data_ptr(), stream_ptr()),
           "pfd_axpby_f16")
    return out


def add_rowvec(a: torch.Tensor, row: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    C = a.shape[-1]
    if out is None:
        out = torch.empty_like(a)
    _check(load().pfd_add_rowvec_f16(a.data_ptr(), row.data_ptr(), a.numel() // C, C, out.data_ptr(),
                                     stream_ptr()), "pfd_add_rowvec_f16")
    return out


def ddim_step(eps: torch.Tensor, x: torch.Tensor, guidance: float, coef: torch.Tensor,
              step: Optional[torch.Tensor], x_prev: torch.Tensor, pred_x0: Optional[torch.Tensor], *,
              noise: Optional[torch.Tensor] = None, temperature: float = 1.0,
              log_tab: Optional[torch.Tensor] = None, log_xt: Optional[torch.Tensor] = None,
              log_x0: Optional[torch.Tensor] = None) -> None:
    """Fused CFG combine + DDIM update (see pfd_ddim_step_f16); eps holds [uncond | cond] halves."""
    _check(load().pfd_ddim_step_f16(eps.data_ptr(), x.data_ptr(), x.numel(), guidance, coef.data_ptr(),
                                    _p(step), x_prev.data_ptr(), _p(pred_x0), _p(noise), float(temperature),
                                    _p(log_tab), _p(log_xt), _p(log_x0), stream_ptr()),
           "pfd_ddim_step_f16")


def ddim_begin_step(step: torch.Tensor, ttab: torch.Tensor, t_out: torch.Tensor) -> None:
    """Device-side loop header: step -= 1; t_out[:] = ttab[step] (see pfd_ddim_begin_step)."""
    if step.dtype != torch.int32 or ttab.dtype != torch.int64 or t_out.dtype != torch.int64:
        raise RuntimeError("ddim_begin_step: step int32, ttab / t_out int64 expected")
    _check(load().pfd_ddim_begin_step(step.data_ptr(), ttab.data_ptr(), t_out.data_ptr(), t_out.numel(),
                                      stream_ptr()), "pfd_ddim_begin_step")


def vae_posterior(moments: torch.Tensor, zc: int, *, noise: Optional[torch.Tensor] = None, scale: float = 1.0,
                  want=("mean", "logvar", "std", "sample")):
    """moments: channel-last [B,H,W,cpad] fp16 -> dict of NCHW fp16 [B,zc,H,W] tensors (pfd_vae_posterior_f16)."""
    B, H, W, cpad = moments.shape
    outs = {k: torch.empty((B, zc, H, W), device=moments.device, dtype=torch.float16) for k in want}
    if noise is not None and (noise.dtype != torch.float32 or not noise.is_contiguous()):
        noise = noise.to(torch.float32).contiguous()
    _check(load().pfd_vae_posterior_f16(moments.data_ptr(), B, zc, H, W, cpad, _p(noise), scale,
                                        _p(outs.get("mean")), _p(outs.get("logvar")), _p(outs.get("std")),
                                        _p(outs.get("sample")), stream_ptr()), "pfd_vae_posterior_f16")
    return outs


def canny(x: torch.Tensor, low: int = 100, high: int = 200) -> Tuple[torch.Tensor, int]:
    """NCHW [B,3,H,W] image in [0,1] (fp16/fp32) -> (float32 [B,3,H,W] edge map, hysteresis sweeps).  Bit-exact
    cv2.Canny(ToPILImage(x), low, high) (pfd_canny_f32); synchronises the stream."""
    if x.dim() != 4 or x.shape[1] != 3 or not x.is_cuda or x.dtype not in (torch.float16, torch.float32):
        raise RuntimeError(f"canny: expected a CUDA fp16/fp32 [B,3,H,W] image, got {tuple(x.shape)} {x.dtype} {x.device}")
    x = x.contiguous()
    B, _, H, W = x.shape
    ws = torch.empty(int(load().pfd_canny_workspace_bytes(B, H, W)), device=x.device, dtype=torch.uint8)
    out = torch.empty((B, 3, H, W), device=x.device, dtype=torch.float32)
    sweeps = c_int32(0)
    _check(load().pfd_canny_f32(x.data_ptr(), int(x.dtype == torch.float32), B, H, W, int(low), int(high),
                                ws.data_ptr(), out.data_ptr(), ctypes.byref(sweeps), stream_ptr()), "pfd_canny_f32")
    return out, int(sweeps.value)


def image_u8_roundtrip(x: torch.Tensor) -> torch.Tensor:
    """ToTensor(ToPILImage(x)) = floor(x*255)/255 as float32 (pfd_image_u8_roundtrip_f32)."""
    if not x.is_cuda or x.dtype not in (torch.float16, torch.float32):
        raise RuntimeError("image_u8_roundtrip: expected a CUDA fp16/fp32 tensor")
    x = x.contiguous()
    out = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    _check(load().pfd_image_u8_roundtrip_f32(x.data_ptr(), int(x.dtype == torch.float32), x.numel(), out.data_ptr(),
                                             stream_ptr()), "pfd_image_u8_roundtrip_f32")
    return out


def hed_input(x: torch.Tensor, norm: torch.Tensor, scale: float) -> torch.Tensor:
    """NCHW [B,3,H,W] image in [0,1] (fp16/fp32) -> channel-last fp16 [B,H,W,3] = (floor(x*255) - norm[c]) * scale
    (pfd_hed_input_f16); norm: CUDA fp32 [3]."""
    if x.dim() != 4 or x.shape[1] != 3 or not x.is_cuda or x.dtype not in (torch.float16, torch.float32):
        raise RuntimeError(f"hed_input: expected a CUDA fp16/fp32 [B,3,H,W] image, got {tuple(x.shape)} {x.dtype} {x.device}")
    if norm.dtype != torch.float32 or norm.numel() != 3 or not norm.is_cuda:
        raise RuntimeError("hed_input: norm must be a CUDA fp32 tensor of 3 values")
    x, norm = x.contiguous(), norm.contiguous()
    B, _, H, W = x.shape
    out = torch.empty((B, H, W, 3), device=x.device, dtype=torch.float16)
    _check(load().pfd_hed_input_f16(x.data_ptr(), int(x.dtype == torch.float32), B, H, W, norm.data_ptr(),
                                    float(scale), out.data_ptr(), stream_ptr()), "pfd_hed_input_f16")
    return out


def maxpool2x2(x: torch.Tensor) -> torch.Tensor:
    """2x2 / stride-2 max-pool (floor) of channel-last fp16 [NB,H,W,C] -> [NB,H/2,W/2,C] (pfd_maxpool2x2_f16)."""
    _chk16(x, "maxpool2x2")
    x = x.contiguous()
    NB, H, W, C = x.shape
    out = torch.empty((NB, H // 2, W // 2, C), device=x.device, dtype=torch.float16)
    _check(load().pfd_maxpool2x2_f16(x.data_ptr(), NB, H, W, C, out.data_ptr(), stream_ptr()), "pfd_maxpool2x2_f16")
    return out


def hed_project(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, inv_scale: float = 1.0) -> torch.Tensor:
    """1x1 conv to one channel with fp32 accumulation: channel-last fp16 [NB,H,W,C] -> fp32 [NB,H,W] =
    dot(x, w) * inv_scale + b (pfd_hed_project_f32); w: CUDA fp32 [C], b: CUDA fp32 [1]."""
    _chk16(x, "hed_project")
    x = x.contiguous()
    NB, H, W, C = x.shape
    if w.dtype != torch.float32 or b.dtype != torch.float32 or w.numel() != C or b.numel() != 1 or not w.is_cuda \
            or not b.is_cuda:
        raise RuntimeError(f"hed_project: expected CUDA fp32 w [{C}] and b [1]")
    out = torch.empty((NB, H, W), device=x.device, dtype=torch.float32)
    _check(load().pfd_hed_project_f32(x.data_ptr(), NB * H * W, C, w.contiguous().data_ptr(), b.data_ptr(),
                                      float(inv_scale), out.data_ptr(), stream_ptr()), "pfd_hed_project_f32")
    return out


def hed_fuse(maps: Sequence[torch.Tensor], H: int, W: int,
             nonfinite: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Five fp32 logit maps [B,h_k,w_k] -> (float32 [B,3,H,W] edge map, CUDA int32 [1] count of non-finite mean
    logits) (pfd_hed_fuse_f32: cv2 INTER_LINEAR resize, mean, sigmoid, uint8 truncation)."""
    if len(maps) != PFD_HED_MAPS:
        raise RuntimeError(f"hed_fuse: expected {PFD_HED_MAPS} maps, got {len(maps)}")
    B = maps[0].shape[0]
    for m in maps:
        if m.dtype != torch.float32 or m.dim() != 3 or m.shape[0] != B or not m.is_cuda or not m.is_contiguous():
            raise RuntimeError(f"hed_fuse: expected contiguous CUDA fp32 [B,h,w] maps, got {tuple(m.shape)} {m.dtype}")
    out = torch.empty((B, 3, H, W), device=maps[0].device, dtype=torch.float32)
    if nonfinite is None:
        nonfinite = torch.empty(1, device=maps[0].device, dtype=torch.int32)
    ptrs = (c_void_p * PFD_HED_MAPS)(*[m.data_ptr() for m in maps])
    hs = (c_int32 * PFD_HED_MAPS)(*[m.shape[1] for m in maps])
    ws = (c_int32 * PFD_HED_MAPS)(*[m.shape[2] for m in maps])
    _check(load().pfd_hed_fuse_f32(ptrs, hs, ws, B, H, W, out.data_ptr(), nonfinite.data_ptr(), stream_ptr()),
           "pfd_hed_fuse_f32")
    return out, nonfinite


def window_gather(x: torch.Tensor, ws: int, shift: int) -> torch.Tensor:
    B, H, W, C = x.shape
    Hp, Wp = -(-H // ws) * ws, -(-W // ws) * ws
    out = torch.empty((B * (Hp // ws) * (Wp // ws), ws * ws, C), device=x.device, dtype=torch.float16)
    _check(load().pfd_window_gather_f16(x.data_ptr(), B, H, W, C, ws, shift, out.data_ptr(), stream_ptr()),
           "pfd_window_gather_f16")
    return out


def window_scatter(win: torch.Tensor, B: int, H: int, W: int, ws: int, shift: int,
                   residual: Optional[torch.Tensor]) -> torch.Tensor:
    C = win.shape[-1]
    out = torch.empty((B, H, W, C), device=win.device, dtype=torch.float16)
    _check(load().pfd_window_scatter_f16(win.data_ptr(), B, H, W, C, ws, shift, _p(residual),
                                         out.data_ptr(), stream_ptr()), "pfd_window_scatter_f16")
    return out


def patch_merge_gather(x: torch.Tensor) -> torch.Tensor:
    B, H, W, C = x.shape
    out = torch.empty((B, (H + 1) // 2, (W + 1) // 2, 4 * C), device=x.device, dtype=torch.float16)
    _check(load().pfd_patch_merge_gather_f16(x.data_ptr(), B, H, W, C, out.data_ptr(), stream_ptr()),
           "pfd_patch_merge_gather_f16")
    return out


def patchify(img: torch.Tensor, P: int, kpad: int) -> torch.Tensor:
    """NCHW image (fp16/fp32) -> [B, ceil(H/P), ceil(W/P), kpad] patch rows (see pfd_patchify_f16)."""
    B, C, H, W = img.shape
    img = img.contiguous()
    if img.dtype not in (torch.float16, torch.float32):
        img = img.to(torch.float16)
    out = torch.empty((B, -(-H // P), -(-W // P), kpad), device=img.device, dtype=torch.float16)
    _check(load().pfd_patchify_f16(img.data_ptr(), int(img.dtype == torch.float32), B, C, H, W, P, kpad,
                                   out.data_ptr(), stream_ptr()), "pfd_patchify_f16")
    return out


def flash_attn(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, *, B: int, heads: int, Nq: int, Nk: int,
               scale: float, out: torch.Tensor) -> torch.Tensor:
    """Fused attention (see pfd_flash_attn_f16): q [BH, Nqp, d], k [BH, Nkp, d], vt [BH, d, Nkp] ->
    out [B, Nq, heads*d]."""
    d = q.shape[2]
    _check(load().pfd_flash_attn_f16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), out.data_ptr(), B, heads, Nq, Nk,
                                     d, q.shape[1], k.shape[1], scale, vt.shape[2], out.stride(0), out.stride(1),
                                     0, stream_ptr()), "pfd_flash_attn_f16")
    return out


def flash_attn_strided(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, *, Nq: int, Nk: int, scale: float,
                       out: torch.Tensor) -> torch.Tensor:
    """pfd_flash_attn_strided_f16: q, k strided views [B, heads, N(p), d]; vt strided view [B, heads, d, Nk(p)]
    (rows contiguous); out [B, Nq, heads*d]."""
    B, heads, _, d = q.shape
    st = lambda t: (c_int64 * 3)(t.stride(0), t.stride(1), t.stride(2))
    _check(load().pfd_flash_attn_strided_f16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), out.data_ptr(), B, heads, Nq,
                                             Nk, d, st(q), st(k), st(vt), scale, out.stride(0), out.stride(1),
                                             stream_ptr()), "pfd_flash_attn_strided_f16")
    return out
