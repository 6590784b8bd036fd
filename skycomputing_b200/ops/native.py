"""Tensor-level wrappers of the sm_100a kernel library (``skycomputing_b200._cuda``).

Every function validates dtype / layout in Python, then hands raw device pointers and the current
CUDA stream to the C++ launcher (which is torch-free, see csrc/bindings_cuda.cpp).  Outputs are
pre-allocated by the caller or allocated here through torch's caching allocator, so everything is
CUDA-graph capturable.

These wrappers FAIL LOUDLY when the extension is missing on a GPU machine: there is no silent
PyTorch fallback on the hot path (the eager oracle lives in ``skycomputing_b200.models`` and is
selected explicitly with ``backend="torch"``).
"""
from __future__ import annotations

from typing import Optional

import torch

_cuda = None
_import_error: Optional[BaseException] = None
try:  # the .so is built in-tree by skycomputing_b200._build / __graft_entry__.build()
    from .. import _cuda as _cuda_mod  # type: ignore

    _cuda = _cuda_mod
except Exception as e:  # pragma: no cover - exercised only when the build is missing
    _import_error = e

ACT_NONE, ACT_GELU, ACT_DGELU_MUL_AUX, ACT_TANH = 0, 1, 2, 3


def available() -> bool:
    """True iff the native extension is importable AND a CUDA device is present."""
    return _cuda is not None and torch.cuda.is_available()


# ---- launch accounting (bench.py reports how many of OUR kernels ran in the timed region) ----
_KERNELS_PER_CALL = {
    "gemm": 1, "layernorm_fwd": 1, "layernorm_bwd": 1, "ln_param_grad": 1, "colsum": 1, "dgelu_mul": 1,
    "attention_fwd": 1, "attention_bwd": 1, "embed_fwd": 1, "embed_bwd": 1,
    "small_linear_fwd": 1, "small_linear_bwd": 2, "softmax_ce": 1, "sgd_multi": 1, "adam_multi": 1,
    "cast_f32_to_bf16": 1, "cast_bf16_to_f32": 1, "advance_counter": 1, "advance_epoch": 1,
    "signal_flags": 1, "wait_flags": 1, "spin_ns": 1, "record_time": 1, "spin_factor": 1,
    "peer_copy_signal": 1,
}
_launches = [0]
_counting_proxy = None


class _CountingExt:
    """Attribute proxy of the extension module that counts kernel launches per call."""

    def __init__(self, mod):
        self._mod = mod
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            target = getattr(self._mod, name)
            n = _KERNELS_PER_CALL.get(name, 0)
            if n and callable(target):
                def fn(*a, __t=target, __n=n, **k):
                    _launches[0] += __n
                    return __t(*a, **k)
            else:
                fn = target
            self._cache[name] = fn
        return fn


def enable_launch_counter() -> None:
    global _counting_proxy
    if _counting_proxy is None and _cuda is not None:
        _counting_proxy = _CountingExt(_cuda)


def reset_launch_counter() -> None:
    _launches[0] = 0


def launch_count() -> int:
    return _launches[0]


def ext():
    if _counting_proxy is not None:
        return _counting_proxy
    if _cuda is None:
        raise RuntimeError(
            "skycomputing_b200._cuda is not built/importable "
            f"({_import_error!r}); run `python -m skycomputing_b200._build` "
            "(or __graft_entry__.build()) first"
        )
    return _cuda


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


def _check(t: torch.Tensor, dtype: torch.dtype, name: str) -> None:
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() >= 1 and t.stride(-1) != 1:
        raise ValueError(f"{name} must have a unit inner stride")


class RngState:
    """Device-resident dropout RNG state {seed, step}; ``advance()`` is a captured kernel."""

    def __init__(self, seed: int, device: torch.device | str = "cuda"):
        # int64 storage, interpreted as uint64 on the device
        self.state = torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64,
                                  device=device)

    @property
    def ptr(self) -> int:
        return self.state.data_ptr()

    def advance(self, inc: int = 1) -> None:
        ext().advance_counter(self.state.data_ptr() + 8, inc, _stream())


def gemm(
    a: torch.Tensor,
    b: torch.Tensor,
    *,
    a_mn: bool = False,
    b_mn: bool = False,
    out: Optional[torch.Tensor] = None,
    out_dtype: torch.dtype = torch.bfloat16,
    accumulate: bool = False,
    bias: Optional[torch.Tensor] = None,
    aux: Optional[torch.Tensor] = None,
    act: int = ACT_NONE,
    add_aux: bool = False,
    out2: Optional[torch.Tensor] = None,
    dropout_p: float = 0.0,
    rng: Optional[RngState] = None,
    rng_stream: int = 0,
    out_ptr: int = 0,
    out_ld: int = 0,
    signal_flags: int = 0,
    wait_flags: int = 0,
    wait_epoch: int = 0,
    wait_mult: int = 0,
    error_flag: int = 0,
    block_n: int = 0,
    pair: int = -1,
    stream_k: int = -1,
    max_ctas: int = 0,
    debug: int = 0,
) -> Optional[torch.Tensor]:
    """out[M,N] = epilogue(sum_k A[m,k] B[n,k]) on the tcgen05 kernel.

    ``a``: [M,K] (or [K,M] when ``a_mn``); ``b``: [N,K] (or [K,N] when ``b_mn``), both bf16 with
    unit inner stride.  ``out_ptr``/``out_ld`` redirect the store to a raw (peer) pointer.
    """
    _check(a, torch.bfloat16, "a")
    _check(b, torch.bfloat16, "b")
    if a.dim() != 2 or b.dim() != 2:
        raise ValueError("gemm operands must be 2-D")
    if a_mn:
        K, M = a.shape
    else:
        M, K = a.shape
    if b_mn:
        Kb, N = b.shape
    else:
        N, Kb = b.shape
    if K != Kb:
        raise ValueError(f"inner dimensions differ: {K} vs {Kb}")
    out_f32 = out_dtype == torch.float32 if out is None else out.dtype == torch.float32
    if out_ptr:
        o_ptr, ldo = out_ptr, out_ld
    else:
        if out is None:
            out = torch.empty((M, N), dtype=out_dtype, device=a.device)
        _check(out, torch.float32 if out_f32 else torch.bfloat16, "out")
        if tuple(out.shape) != (M, N):
            raise ValueError(f"out has shape {tuple(out.shape)}, expected {(M, N)}")
        o_ptr, ldo = out.data_ptr(), out.stride(0)
    if bias is not None:
        _check(bias, torch.float32, "bias")
    if aux is not None:
        _check(aux, torch.bfloat16, "aux")
    if out2 is not None:
        _check(out2, torch.bfloat16, "out2")
    ext().gemm(
        A=a.data_ptr(), B=b.data_ptr(), M=M, N=N, K=K, lda=a.stride(0), ldb=b.stride(0),
        a_mn=a_mn, b_mn=b_mn, out=o_ptr, ldo=ldo, out_f32=out_f32, accumulate=accumulate,
        out2=_ptr(out2), ldo2=0 if out2 is None else out2.stride(0), bias=_ptr(bias),
        aux=_ptr(aux), ldaux=0 if aux is None else aux.stride(0), act=act, add_aux=add_aux,
        dropout_p=float(dropout_p), rng_state=0 if rng is None else rng.ptr,
        rng_stream=rng_stream, signal_flags=signal_flags, wait_flags=wait_flags,
        wait_epoch=wait_epoch, wait_mult=wait_mult, error_flag=error_flag, block_n=block_n, pair=pair, stream_k=stream_k,
        max_ctas=max_ctas, debug=debug, stream=_stream(),
    )
    return out


def _fuse_ln_mode() -> str:
    import os

    return os.environ.get("SKY_FUSE_LN", "1")


def gemm_ln_supported(M: int, N: int) -> bool:
    """Should ``dense + LayerNorm`` of this output shape run as the one-kernel GEMM + LayerNorm
    epilogue?  Default: where it is faster than GEMM + standalone LayerNorm (csrc: gemm_ln_block_n);
    ``SKY_FUSE_LN=force``: wherever the kernel can run; ``SKY_FUSE_LN=0``: never."""
    mode = _fuse_ln_mode()
    if mode == "0":
        return False
    return ext().gemm_ln_block_n(int(M), int(N), mode == "force") != 0


def gemm_ln_tiles_per_panel(M: int, N: int) -> int:
    """Flag signals per 128-row panel when the fused kernel writes a stage boundary."""
    return ext().gemm_ln_tiles_per_panel(int(M), int(N), _fuse_ln_mode() == "force")


def gemm_ln(a: torch.Tensor, b: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *,
            eps: float = 1e-12, bias: Optional[torch.Tensor] = None,
            residual: Optional[torch.Tensor] = None, dropout_p: float = 0.0,
            rng: Optional[RngState] = None, rng_stream: int = 0, save_z: bool = True,
            y_ptr: int = 0, y_ld: int = 0, signal_flags: int = 0, wait_flags: int = 0,
            wait_epoch: int = 0, wait_mult: int = 0, error_flag: int = 0, block_n: int = 0):
    """y = LayerNorm(dropout(a b^T + bias) + residual) * gamma + beta in ONE tcgen05 kernel
    (cluster-wide row statistics through DSMEM, see csrc/kernels/gemm_sm100.cu).

    Returns ``(y, z, mean, rstd)``: ``z`` is the bf16 pre-LayerNorm sum saved for backward (None
    when ``save_z`` is False), ``y`` is None when ``y_ptr`` redirects the store to raw (peer)
    memory; ``signal_flags`` then receives ``gemm_ln_tiles_per_panel`` signals per 128-row panel."""
    _check(a, torch.bfloat16, "a")
    _check(b, torch.bfloat16, "b")
    _check(gamma, torch.float32, "gamma")
    _check(beta, torch.float32, "beta")
    M, K = a.shape
    N, Kb = b.shape
    if K != Kb:
        raise ValueError(f"inner dimensions differ: {K} vs {Kb}")
    if bias is not None:
        _check(bias, torch.float32, "bias")
    if residual is not None:
        _check(residual, torch.bfloat16, "residual")
    dev = a.device
    y = None
    if y_ptr:
        o_ptr, ldo = y_ptr, (y_ld or N)
    else:
        y = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
        o_ptr, ldo = y.data_ptr(), N
    z = torch.empty((M, N), dtype=torch.bfloat16, device=dev) if save_z else None
    mean = torch.empty(M, dtype=torch.float32, device=dev)
    rstd = torch.empty(M, dtype=torch.float32, device=dev)
    ext().gemm(
        A=a.data_ptr(), B=b.data_ptr(), M=M, N=N, K=K, lda=a.stride(0), ldb=b.stride(0),
        out=o_ptr, ldo=ldo, out2=_ptr(z), ldo2=0 if z is None else N, bias=_ptr(bias),
        aux=_ptr(residual), ldaux=0 if residual is None else residual.stride(0),
        add_aux=residual is not None, dropout_p=float(dropout_p),
        rng_state=0 if rng is None else rng.ptr, rng_stream=rng_stream,
        signal_flags=signal_flags, wait_flags=wait_flags, wait_epoch=wait_epoch,
        wait_mult=wait_mult, error_flag=error_flag, block_n=block_n,
        ln_gamma=gamma.data_ptr(), ln_beta=beta.data_ptr(), ln_mean=mean.data_ptr(),
        ln_rstd=rstd.data_ptr(), ln_eps=float(eps), stream=_stream(),
    )
    return y, z, mean, rstd


def layernorm_fwd(z, gamma, beta, eps: float = 1e-12, *, y=None, wait_flags: int = 0,
                  wait_epoch: int = 0, wait_mult: int = 0, error_flag: int = 0):
    _check(z, torch.bfloat16, "z")
    M, H = z.shape
    if not z.is_contiguous():
        raise ValueError("z must be contiguous")
    y = torch.empty_like(z) if y is None else y
    mean = torch.empty(M, dtype=torch.float32, device=z.device)
    rstd = torch.empty(M, dtype=torch.float32, device=z.device)
    ext().layernorm_fwd(z=z.data_ptr(), y=y.data_ptr(), mean=mean.data_ptr(), rstd=rstd.data_ptr(),
                        gamma=gamma.data_ptr(), beta=beta.data_ptr(), M=M, H=H, eps=eps,
                        wait_flags=wait_flags, wait_epoch=wait_epoch, wait_mult=wait_mult,
                        error_flag=error_flag, stream=_stream())
    return y, mean, rstd


def layernorm_bwd(dy, z, mean, rstd, gamma, dgamma, dbeta, *, dropout_p: float = 0.0,
                  rng: Optional[RngState] = None, rng_stream: int = 0, wait_flags: int = 0,
                  wait_epoch: int = 0, wait_mult: int = 0, error_flag: int = 0):
    """Returns (dz, dz_dropped or None); dgamma/dbeta (fp32) are accumulated in place, or left to a
    later `ln_param_grad` call when passed as None."""
    _check(dy, torch.bfloat16, "dy")
    _check(z, torch.bfloat16, "z")
    M, H = z.shape
    dz = torch.empty_like(z)
    dzd = torch.empty_like(z) if dropout_p > 0 else None
    ext().layernorm_bwd(dy=dy.data_ptr(), z=z.data_ptr(), mean=mean.data_ptr(),
                        rstd=rstd.data_ptr(), gamma=gamma.data_ptr(), dz=dz.data_ptr(),
                        dz_dropped=_ptr(dzd), dgamma=_ptr(dgamma), dbeta=_ptr(dbeta),
                        M=M, H=H, dropout_p=float(dropout_p),
                        rng_state=0 if rng is None else rng.ptr, rng_stream=rng_stream,
                        wait_flags=wait_flags, wait_epoch=wait_epoch, wait_mult=wait_mult,
                        error_flag=error_flag, stream=_stream())
    return dz, dzd


def ln_param_grad(dy, z, mean, rstd, dgamma, dbeta, x2=None, out2=None) -> None:
    """dgamma += sum_rows dy * xhat, dbeta += sum_rows dy (the second half of layernorm_bwd);
    optionally also out2 += column sums of x2 ([M,H] bf16): the bias gradient of the dense layer
    in front of the LayerNorm, fused to save a launch."""
    M, H = z.shape
    if x2 is not None:
        _check(x2, torch.bfloat16, "x2")
        if tuple(x2.shape) != (M, H) or not x2.is_contiguous():
            raise ValueError("x2 must be a contiguous [M,H] tensor")
    ext().ln_param_grad(dy=dy.data_ptr(), z=z.data_ptr(), mean=mean.data_ptr(), rstd=rstd.data_ptr(),
                        dgamma=dgamma.data_ptr(), dbeta=dbeta.data_ptr(), M=M, H=H, x2=_ptr(x2),
                        out2=_ptr(out2), stream=_stream())


def colsum_(x: torch.Tensor, out: torch.Tensor) -> None:
    """out[n] += sum_m x[m, n]  (x bf16, out fp32)."""
    _check(x, torch.bfloat16, "x")
    _check(out, torch.float32, "out")
    M, N = x.shape
    ext().colsum(x=x.data_ptr(), M=M, N=N, ldx=x.stride(0), out=out.data_ptr(), stream=_stream())


def attention_supported(S: int, head_dim: int) -> bool:
    """Shapes the tcgen05 attention kernels run: any sequence length that is a multiple of 8 and
    any head size that is a multiple of 8 from 8 to 128.  Pure Python (the same rule as the C++
    ``attention_supported``), so CPU-only callers can ask without loading the extension."""
    return S > 0 and S % 8 == 0 and head_dim % 8 == 0 and 8 <= head_dim <= 128


def attention_fwd(qkv, mask, B: int, S: int, heads: int, *, dropout_p: float = 0.0,
                  rng: Optional[RngState] = None, rng_stream: int = 0):
    _check(qkv, torch.bfloat16, "qkv")
    H = qkv.shape[1] // 3
    d = H // heads
    ctx = torch.empty((B * S, H), dtype=torch.bfloat16, device=qkv.device)
    lse = torch.empty((B * heads * S,), dtype=torch.float32, device=qkv.device)
    ext().attention_fwd(qkv=qkv.data_ptr(), mask=_ptr(mask), ctx=ctx.data_ptr(),
                        lse=lse.data_ptr(), B=B, S=S, heads=heads, head_dim=d,
                        scale=1.0 / (d ** 0.5), dropout_p=float(dropout_p),
                        rng_state=0 if rng is None else rng.ptr, rng_stream=rng_stream,
                        stream=_stream())
    return ctx, lse


def attention_bwd(qkv, mask, ctx, lse, dctx, B: int, S: int, heads: int, *,
                  dropout_p: float = 0.0, rng: Optional[RngState] = None, rng_stream: int = 0):
    _check(dctx, torch.bfloat16, "dctx")
    if not dctx.is_contiguous():
        dctx = dctx.contiguous()
    H = qkv.shape[1] // 3
    d = H // heads
    dqkv = torch.empty_like(qkv)
    ext().attention_bwd(qkv=qkv.data_ptr(), mask=_ptr(mask), ctx=ctx.data_ptr(),
                        lse=lse.data_ptr(), dctx=dctx.data_ptr(), dqkv=dqkv.data_ptr(), B=B, S=S,
                        heads=heads, head_dim=d, scale=1.0 / (d ** 0.5),
                        dropout_p=float(dropout_p), rng_state=0 if rng is None else rng.ptr,
                        rng_stream=rng_stream, stream=_stream())
    return dqkv


def cast_f32_to_bf16_(src: torch.Tensor, dst: torch.Tensor) -> None:
    ext().cast_f32_to_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream())


def softmax_ce(logits: torch.Tensor, labels: torch.Tensor, grad_scale: float = 1.0,
               loss_acc: Optional[torch.Tensor] = None):
    """Mean cross entropy and d(loss * grad_scale)/dlogits; ``loss_acc[0] += loss * grad_scale``
    when given (the step loss of a micro-batched step, accumulated without extra launches)."""
    _check(logits, torch.float32, "logits")
    M, C = logits.shape
    loss = torch.empty(1, dtype=torch.float32, device=logits.device)
    dlogits = torch.empty_like(logits)
    ext().softmax_ce(logits=logits.data_ptr(), labels=labels.data_ptr(), loss=loss.data_ptr(),
                     dlogits=dlogits.data_ptr(), M=M, C=C, grad_scale=grad_scale,
                     loss_acc=_ptr(loss_acc), stream=_stream())
    return loss, dlogits
