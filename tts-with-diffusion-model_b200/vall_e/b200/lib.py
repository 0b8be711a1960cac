"""ctypes binding of libvalle_b200.so (C ABI declared in include/vb200.h).

There is no fallback: if the library is missing or a call fails, this raises.  Tensors are
passed as raw device pointers; every call runs on torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("VB200_LIB", _HERE / "libvalle_b200.so"))   # override: bring-up experiments only

OK = 0
F32, BF16, F16 = 0, 1, 2
EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESIDUAL = 0, 1, 2, 3
ABSORBING, UNIFORM = 0, 1
NOISE_PHILOX, NOISE_UNIFORMS, NOISE_GREEDY = 0, 1, 2
U_ROW0, U_TTXT, U_TPROM, U_TRESP, U_TXT0, U_PROM0, U_RESP0, U_GID, U_STRIDE = range(9)
(TAB_ONE_KEEP, TAB_ONE_OFF, TAB_ONE_ABSORB, TAB_ONE_BOTH, TAB_CUM_KEEP, TAB_CUM_OFF, TAB_CUM_ABSORB,
 TAB_CUM_BOTH, TAB_LOG_KEEP, TAB_LOG_OFF, TAB_LOG_ABSORB, TAB_LOG_BOTH, TAB_STRIDE) = range(13)

_DTYPES = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}

_p, _i32, _i64, _u64, _f = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float

# name -> argtypes; must list every symbol include/vb200.h declares (tests check this)
PROTOTYPES = {
    "vb200_last_error": ([], C.c_char_p),
    "vb200_version": ([], C.c_int),
    "vb200_device_sms": ([], C.c_int),
    "vb200_embed_gather": ([_p] * 13 + [_i32] * 4 + [_p], C.c_int),
    "vb200_adaln": ([_p, C.c_int] + [_p] * 4 + [_i32, _i32, _f, _f, _f, _p], C.c_int),
    "vb200_layernorm": ([_p, C.c_int] + [_p] * 3 + [_i32, _i32, _f, _p], C.c_int),
    "vb200_gather_rows_bf16": ([_p, C.c_int, _p, _p, _i32, _i32, _p], C.c_int),
    "vb200_gemm_bf16": ([_p, C.c_int, _p, C.c_int, _p, _p, _p, _i32, _i32, _i32, C.c_int, _p], C.c_int),
    "vb200_gemm_bf16_simt": ([_p, C.c_int, _p, C.c_int, _p, _p, _p, _i32, _i32, _i32, C.c_int, _p], C.c_int),
    "vb200_flash_attn_varlen": ([_p, _p, _p, _i32, _i32, _i32, _i32, _f, _p], C.c_int),
    "vb200_attn_varlen_simt": ([_p, _p, _p, _i32, _i32, _i32, _i32, _f, _p], C.c_int),
    "vb200_q_sample": ([_p] * 6 + [_i32, _i32, _i32, C.c_int, _p], C.c_int),
    "vb200_q_sample_dense": ([_p] * 6 + [_i32, _i32, _i32, _p], C.c_int),
    "vb200_posterior_sample_from_logits": (
        [_p, _p, _p, C.c_int, _i64, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, C.c_int, C.c_int, _p, _u64, _p],
        C.c_int),
    "vb200_head_posterior_sample": (
        [_p, _p, C.c_int, _p, C.c_int, _p, _p, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _i32, C.c_int, C.c_int, _p, _u64,
         _p],
        C.c_int),
    "vb200_posterior_sample_from_logits_known": (
        [_p, _p, _p, C.c_int, _i64, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, C.c_int, C.c_int, _p, _u64, _p, _p],
        C.c_int),
    "vb200_head_posterior_sample_known": (
        [_p, _p, C.c_int, _p, C.c_int, _p, _p, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _i32, C.c_int, C.c_int, _p, _u64,
         _p, _p],
        C.c_int),
    "vb200_q_sample_philox": ([_p] * 5 + [_i32, _i32, _i32, C.c_int, _u64, _p], C.c_int),
    "vb200_head_fused": ([_i32, _i32, C.c_int], C.c_int),
    "vb200_head_ce_loss": ([_p, _p, C.c_int, _p, _p, _p, _i32, _i32, _i32, _i32, _p], C.c_int),
    "vb200_workspace_bytes": ([_i64, _i64, _i32, _i32, C.c_int, C.POINTER(C.c_int64)], C.c_int64),
    "vb200_step_timesteps": ([_p, _i32, _i32, _p], C.c_int),
    "vb200_step_timesteps_to": ([_p, _i32, _p, _i32, _p], C.c_int),
    "vb200_codes_to_bqt": ([_p, _p, _p, _i32, _i32, _i32, _i64, _p], C.c_int),
}

_lib = None


class VB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Loads the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VB200Error(
            f"{LIB_PATH} is missing: build it with `python tts-with-diffusion-model_b200/build.py` "
            "(the CUDA library is the only implementation of the hot path; there is no fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (argtypes, restype) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def last_error() -> str:
    return load().vb200_last_error().decode("utf-8", "replace")


def _check(rc: int, what: str) -> None:
    if rc != OK:
        raise VB200Error(f"{what} failed with status {rc}: {last_error()}")


# Devices of the tensors handed to the call being assembled.  Every wrapper below builds its argument
# list as ``fn(ptr(a), ptr(b), ..., stream())``: Python evaluates the arguments left to right, so by the
# time ``stream()`` runs, ``ptr`` has seen every tensor of the call.
_call_devices: set = set()


def ptr(t: torch.Tensor | None):
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        _call_devices.clear()
        raise VB200Error("vb200 kernels take CUDA tensors only (no CPU fallback)" if not t.is_cuda
                         else "vb200 kernels take contiguous tensors")
    _call_devices.add(t.device.index)
    return t.data_ptr()


def stream():
    """The launch stream: torch's current stream ON THE DEVICE THE TENSORS LIVE ON.  The library launches on
    the current CUDA device (kernel attributes, SM count and the stream all belong to it), so tensors on
    another device would be dereferenced from the wrong GPU — refused here instead (callers switch with
    ``torch.cuda.device``; the engine and the model classes do)."""
    devs = set(_call_devices)
    _call_devices.clear()
    cur = torch.cuda.current_device()
    if len(devs) > 1:
        raise VB200Error(f"tensors of one call live on different devices: cuda:{sorted(devs)}")
    if devs and devs != {cur}:
        raise VB200Error(f"tensors live on cuda:{devs.pop()} but the current CUDA device is cuda:{cur}; "
                         "wrap the call in `with torch.cuda.device(...)`")
    return torch.cuda.current_stream(cur).cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    return _DTYPES[dt]


def act_code(t: torch.Tensor) -> int:
    """dtype code of a 16-bit activation tensor (bf16 or fp16)."""
    if t.dtype not in (torch.bfloat16, torch.float16):
        raise VB200Error(f"16-bit activations must be bf16 or fp16, got {t.dtype}")
    return _DTYPES[t.dtype]


# ------------------------------------------------------------------ thin typed wrappers
def embed_gather(x_out, text_w, prom_w, resp_w, sep, time_w, pe, text_ids, prom_ids, resp_ids, utt,
                 row_utt, t_utt, K, resp_levels_in):
    M, d = x_out.shape
    _check(load().vb200_embed_gather(ptr(x_out), ptr(text_w), ptr(prom_w), ptr(resp_w), ptr(sep),
                                     ptr(time_w), ptr(pe), ptr(text_ids), ptr(prom_ids), ptr(resp_ids),
                                     ptr(utt), ptr(row_utt), ptr(t_utt), M, d, K, resp_levels_in,
                                     stream()), "vb200_embed_gather")


def adaln(out, x, table, level_utt, row_utt, eps=1e-5, k=0.1, c=2.0):
    M, d = x.shape
    _check(load().vb200_adaln(ptr(out), act_code(out), ptr(x), ptr(table), ptr(level_utt), ptr(row_utt), M, d, eps,
                              k, c, stream()), "vb200_adaln")


def layernorm(out, x, weight, bias, eps=1e-5):
    M, d = x.shape
    _check(load().vb200_layernorm(ptr(out), act_code(out), ptr(x), ptr(weight), ptr(bias), M, d, eps, stream()),
           "vb200_layernorm")


def gather_rows_bf16(out, x, row_index):
    n, d = out.shape
    _check(load().vb200_gather_rows_bf16(ptr(out), act_code(out), ptr(x), ptr(row_index), n, d, stream()),
           "vb200_gather_rows_bf16")


def codes_to_bqt(out, codes, utt, pad=0):
    """packed int32 codes (sum t'', l) -> int64 (B, l, T_max) for the EnCodec decoder (emb/qnt.py:32-49)."""
    B, n_levels, T_max = out.shape
    assert out.dtype == torch.int64 and codes.dtype == torch.int32 and out.is_contiguous() and codes.is_contiguous()
    _check(load().vb200_codes_to_bqt(ptr(out), ptr(codes), ptr(utt), B, n_levels, T_max, int(pad), stream()),
           "vb200_codes_to_bqt")


def gemm_bf16(out, A, W, bias=None, residual=None, epi=EPI_NONE, simt=False):
    M, K = A.shape
    N = W.shape[0]
    assert W.shape[1] == K and tuple(out.shape) == (M, N), (A.shape, W.shape, out.shape)
    assert A.dtype in (torch.bfloat16, torch.float16) and W.dtype == A.dtype, (A.dtype, W.dtype)
    fn = load().vb200_gemm_bf16_simt if simt else load().vb200_gemm_bf16
    _check(fn(ptr(out), dtype_code(out.dtype), ptr(A), act_code(A), ptr(W), ptr(bias), ptr(residual), M, N, K, epi,
              stream()), "vb200_gemm_bf16")


def flash_attn_varlen(out, qkv, cu_rows, max_T, n_heads, scale, variant="tmem"):
    M = qkv.shape[0]
    B = cu_rows.numel() - 1
    fn = {"tmem": load().vb200_flash_attn_varlen, "simt": load().vb200_attn_varlen_simt}[variant]
    _check(fn(ptr(out), ptr(qkv), ptr(cu_rows), B, max_T, M, n_heads, scale, stream()),
           f"vb200_flash_attn_varlen[{variant}]")


def q_sample(x_out, x0, t_tok, mask, uniforms, table, K, transition):
    n = x0.numel()
    _check(load().vb200_q_sample(ptr(x_out), ptr(x0), ptr(t_tok), ptr(mask), ptr(uniforms), ptr(table), n, K,
                                 table.shape[0], transition, stream()), "vb200_q_sample")


def q_sample_dense(x_out, x0, t_tok, mask, uniforms, log_qbar):
    """q_sample against the caller's dense fp16 (S, K, K) log(Qbar_t + eps) (bit-exact for any table)."""
    S, K, _ = log_qbar.shape
    assert log_qbar.dtype == torch.float16
    _check(load().vb200_q_sample_dense(ptr(x_out), ptr(x0), ptr(t_tok), ptr(mask), ptr(uniforms), ptr(log_qbar),
                                       x0.numel(), K, S, stream()), "vb200_q_sample_dense")


def posterior_sample_from_logits(x_out, post_out, logits, ld_logits, x_t, row_utt, t_utt, utt, table,
                                 n_rows, n_levels, K, transition, noise, uniforms=None, seed=0, known=None):
    """``known``: int32 (n_rows, n_levels), -1 = draw as usual, k in [0, K) = the token's x0 is k (the ``_known``
    entry point); None calls the plain one."""
    if known is None:
        _check(load().vb200_posterior_sample_from_logits(
            ptr(x_out), ptr(post_out), ptr(logits), dtype_code(logits.dtype), ld_logits, ptr(x_t),
            ptr(row_utt), ptr(t_utt), ptr(utt), ptr(table), n_rows, n_levels, K, table.shape[0], transition,
            noise, ptr(uniforms), seed, stream()), "vb200_posterior_sample_from_logits")
        return
    _check(load().vb200_posterior_sample_from_logits_known(
        ptr(x_out), ptr(post_out), ptr(logits), dtype_code(logits.dtype), ld_logits, ptr(x_t),
        ptr(row_utt), ptr(t_utt), ptr(utt), ptr(table), n_rows, n_levels, K, table.shape[0], transition,
        noise, ptr(uniforms), seed, ptr(known), stream()), "vb200_posterior_sample_from_logits_known")


def head_posterior_sample(x_out, logits, head_in, W, bias, x_t, row_utt, t_utt, utt, table, n_levels, K,
                          transition, noise, uniforms=None, seed=0, known=None):
    """classifier + reverse step in one C call: one kernel (reverse step as the GEMM epilogue) when
    head_fused(), else GEMM into the caller's `logits` scratch (required then) + standalone kernel.
    ``known`` as in posterior_sample_from_logits."""
    n_rows, d = head_in.shape
    ldt = dtype_code(logits.dtype) if logits is not None else dtype_code(torch.float16)
    if known is None:
        _check(load().vb200_head_posterior_sample(
            ptr(x_out), ptr(logits), ldt, ptr(head_in), act_code(head_in), ptr(W), ptr(bias), n_rows, d,
            n_levels, K, ptr(x_t), ptr(row_utt), ptr(t_utt), ptr(utt), ptr(table), table.shape[0], transition,
            noise, ptr(uniforms), seed, stream()), "vb200_head_posterior_sample")
        return
    _check(load().vb200_head_posterior_sample_known(
        ptr(x_out), ptr(logits), ldt, ptr(head_in), act_code(head_in), ptr(W), ptr(bias), n_rows, d,
        n_levels, K, ptr(x_t), ptr(row_utt), ptr(t_utt), ptr(utt), ptr(table), table.shape[0], transition,
        noise, ptr(uniforms), seed, ptr(known), stream()), "vb200_head_posterior_sample_known")


def q_sample_philox(x_out, x0, t_tok, mask, table, K, transition, seed=0):
    """x_t ~ q(x_t | x_0) with in-kernel Philox noise, O(1) per token."""
    _check(load().vb200_q_sample_philox(ptr(x_out), ptr(x0), ptr(t_tok), ptr(mask), ptr(table), x0.numel(), K,
                                        table.shape[0], transition, seed, stream()), "vb200_q_sample_philox")


def head_ce_loss(loss, head_in, W, bias, targets, n_levels, K):
    """loss[r, l] = -log softmax(head_in[r] W_l^T + b_l)[targets[r, l]] as the classifier GEMM's epilogue."""
    n_rows, d = head_in.shape
    _check(load().vb200_head_ce_loss(ptr(loss), ptr(head_in), act_code(head_in), ptr(W), ptr(bias), ptr(targets),
                                     n_rows, d, n_levels, K, stream()), "vb200_head_ce_loss")


def head_fused(d, K, noise) -> bool:
    """Whether head_posterior_sample runs as one kernel (else GEMM + standalone reverse step); host-only."""
    return bool(load().vb200_head_fused(d, K, noise))


WS_FIELDS = ("x", "h", "qkv", "att", "ff", "head_in", "logits")


def workspace_bytes(M, M_resp, d, n_out, logits_dtype):
    """(total, sizes[7]) of the scratch one denoiser forward needs, in WS_FIELDS order (host-only call)."""
    sizes = (C.c_int64 * 7)()
    total = load().vb200_workspace_bytes(M, M_resp, d, n_out, dtype_code(logits_dtype), sizes)
    if total < 0:
        raise VB200Error(f"vb200_workspace_bytes failed with status {total}: {last_error()}")
    return int(total), [int(v) for v in sizes]


def step_timesteps(t_utt, delta):
    _check(load().vb200_step_timesteps(ptr(t_utt), t_utt.numel(), delta, stream()), "vb200_step_timesteps")


def step_timesteps_to(t_utt, next_t):
    """t_utt[b] = next_t[t_utt[b]] on device; next_t int32 (S,) (d3pm.successors)."""
    _check(load().vb200_step_timesteps_to(ptr(t_utt), t_utt.numel(), ptr(next_t),
                                          next_t.numel() if next_t is not None else 0, stream()),
           "vb200_step_timesteps_to")
