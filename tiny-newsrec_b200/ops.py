"""Tensor-level wrappers over the C ABI (include/tinyrec.h).

Every function takes CUDA torch tensors, checks dtype / layout, and enqueues the
kernel on torch's current stream.  Torch is used only for device memory and
streams.  No function here has a non-CUDA path.
"""
import ctypes

import torch

from . import _lib
from ._lib import ACT_DGELU, ACT_GELU, ACT_GELU_DAUX, ACT_MULAUX, ACT_NONE, ACT_TANH, BF16, F32, Dropout, GemmArgs  # noqa: F401

_bf16 = torch.bfloat16
_f32 = torch.float32


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t, dtype, name):
    if t.dtype != dtype or not t.is_cuda:
        raise _lib.TinyRecError(f"{name}: expected CUDA {dtype}, got {t.dtype} on {t.device}")
    return t


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def make_drop(seed_tensor, site, p):
    """tnr_dropout for dropout tensor ``site``; ``seed_tensor`` is a 1-element CUDA int64 tensor
    (the kernels read the seed from device memory).  Returns None when p == 0."""
    if seed_tensor is None or not p > 0.0:
        return None
    d = Dropout()
    d.seed, d.site, d.p = seed_tensor.data_ptr(), int(site), float(p)
    return d


def _dp(d):
    return ctypes.byref(d) if d is not None else None


def dropout_mask(drop, n, device):
    """keep flags (uint8 [n]) of dropout tensor ``drop`` by linear element index (tests)."""
    keep = torch.empty(n, device=device, dtype=torch.uint8)
    lib = _ready(keep)
    _lib.check(lib.tnr_dropout_mask(_dp(drop), n, _ptr(keep), _stream()), "tnr_dropout_mask")
    return keep


class _Stats:
    """Launch accounting for bench.py: ``launches`` counts kernels of libtinyrec enqueued;
    when ``gemm_events`` is a list every tnr_gemm_bf16 launch is bracketed by CUDA events on the
    launching stream and (flops, start, stop) is appended (roofline measurement); when
    ``op_events`` is a list every op wrapper of this module is bracketed the same way and
    (name, tag, start, stop) appended (tools/step_profile.py)."""
    launches = 0
    gemm_events = None
    op_events = None


stats = _Stats()

# Bumped whenever a kernel of this library rewrites parameters in place through raw pointers (the fused Adam, eager
# or inside a replayed graph): torch's ``_version`` counters do not see those writes, so derived copies that are
# cached per parameter (the packed TF32 W1 of the scoring kernels) key on this as well.
param_generation = 0


def bump_param_generation():
    global param_generation
    param_generation += 1


def _timed(fn):
    """Per-op CUDA-event bracketing, active only while ``stats.op_events`` is a list."""
    import functools

    @functools.wraps(fn)
    def wrap(*a, **k):
        if stats.op_events is None:
            return fn(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn(*a, **k)
        e1.record()
        tag = ""
        if fn.__name__ == "gemm":
            A, Bm = a[0], a[1]
            M, K = (A.shape[1], A.shape[0]) if k.get("a_t") else (A.shape[0], A.shape[1])
            N = Bm.shape[1] if k.get("b_t") else Bm.shape[0]
            tag = f"{M}x{N}x{K}" + ("/wgrad" if k.get("a_t") else "/dgrad" if k.get("b_t") else "") + \
                  {ACT_NONE: "", ACT_GELU: "+gelu", ACT_TANH: "+tanh", ACT_DGELU: "+dgelu", ACT_GELU_DAUX: "+gelu",
                   ACT_MULAUX: "+mulaux"}[k.get("act", ACT_NONE)] + \
                  ("+aux" if k.get("aux") is not None and k.get("act") in (ACT_GELU, ACT_GELU_DAUX) else "") + \
                  ("+res" if k.get("residual") is not None else "") + ("+bias" if k.get("bias") is not None else "")
        stats.op_events.append((fn.__name__, tag, e0, e1))
        return r
    return wrap


def _ready(t, kernels=1):
    _lib.require_device(t.device.index)
    stats.launches += kernels
    return _lib.load()


@_timed
def gemm(a, b, out, *, a_t=False, b_t=False, bias=None, residual=None, act=ACT_NONE, aux=None,
         split_k=1, accumulate=False, drop=None, colsum=None):
    """out[M,N] = epilogue(A[M,K] @ B[N,K]^T).

    a: bf16 [M,K] (or [K,M] when ``a_t``); b: bf16 [N,K] (or [K,N] when ``b_t``); 2-D, unit
    inner stride.  out: bf16 or fp32 [M,N].  See tnr_gemm_bf16 in include/tinyrec.h.
    """
    lib = _ready(a)
    _chk(a, _bf16, "gemm.a"); _chk(b, _bf16, "gemm.b")
    if a.stride(1) != 1 or b.stride(1) != 1 or out.stride(1) != 1:
        raise _lib.TinyRecError("gemm: operands must have unit inner stride")
    M, K = (a.shape[1], a.shape[0]) if a_t else (a.shape[0], a.shape[1])
    N, Kb = (b.shape[1], b.shape[0]) if b_t else (b.shape[0], b.shape[1])
    if K != Kb or out.shape[0] != M or out.shape[1] != N:
        raise _lib.TinyRecError(f"gemm: shape mismatch A{tuple(a.shape)} B{tuple(b.shape)} C{tuple(out.shape)} "
                                f"a_t={a_t} b_t={b_t}")
    g = GemmArgs()
    g.M, g.N, g.K = M, N, K
    g.A, g.lda, g.a_mn_major = a.data_ptr(), a.stride(0), int(a_t)
    g.B, g.ldb, g.b_mn_major = b.data_ptr(), b.stride(0), int(b_t)
    g.C, g.ldc = out.data_ptr(), out.stride(0)
    if out.dtype == _bf16:
        g.c_dtype = BF16
    elif out.dtype == _f32:
        g.c_dtype = F32
    else:
        raise _lib.TinyRecError("gemm: out must be bf16 or fp32")
    g.bias = _chk(bias, _f32, "gemm.bias").data_ptr() if bias is not None else None
    if residual is not None:
        _chk(residual, _bf16, "gemm.residual")
        g.residual, g.ldr = residual.data_ptr(), residual.stride(0)
    g.act = act
    if aux is not None:
        _chk(aux, _bf16, "gemm.aux")
        g.aux, g.ldaux = aux.data_ptr(), aux.stride(0)
    g.split_k = split_k
    g.accumulate = int(accumulate)
    if drop is not None:
        g.drop = ctypes.pointer(drop)
    if colsum is not None:
        g.colsum = _chk(colsum, _f32, "gemm.colsum").data_ptr()
    if stats.gemm_events is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(lib.tnr_gemm_bf16(ctypes.byref(g), _stream()), "tnr_gemm_bf16")
        e1.record()
        stats.gemm_events.append((2.0 * M * N * K, e0, e1))
        return out
    _lib.check(lib.tnr_gemm_bf16(ctypes.byref(g), _stream()), "tnr_gemm_bf16")
    return out


@_timed
def embed_ln(x, L, word, pos, type0, gamma, beta, eps, out, drop=None):
    """x: int64 [n, 2L] (ids | mask) -> out bf16 [n*L, E]."""
    lib = _ready(x)
    _chk(x, torch.int64, "embed_ln.x")
    n = x.shape[0]
    E = word.shape[1]
    wd = BF16 if word.dtype == _bf16 else F32
    _lib.check(lib.tnr_embed_ln_fwd(_ptr(x), x.stride(0), n, L, word.shape[0], _ptr(word), wd,
                                    _ptr(_chk(pos, _f32, "pos")), _ptr(_chk(type0, _f32, "type0")),
                                    _ptr(_chk(gamma, _f32, "gamma")), _ptr(_chk(beta, _f32, "beta")),
                                    eps, E, _ptr(_chk(out, _bf16, "out")), _dp(drop), _stream()), "tnr_embed_ln_fwd")
    return out


@_timed
def layernorm_fwd(x, gamma, beta, eps, out):
    lib = _ready(x)
    rows, E = x.shape
    _lib.check(lib.tnr_layernorm_fwd(_ptr(_chk(x, _bf16, "ln.x")), rows, E, _ptr(gamma), _ptr(beta), eps,
                                     _ptr(_chk(out, _bf16, "ln.out")), _stream()), "tnr_layernorm_fwd")
    return out


@_timed
def layernorm_bwd(dy, x, gamma, eps, dx, dgamma, dbeta, dx_drop=None, drop=None, dsum=None):
    lib = _ready(x)
    rows, E = x.shape
    _lib.check(lib.tnr_layernorm_bwd(_ptr(_chk(dy, _bf16, "ln.dy")), _ptr(_chk(x, _bf16, "ln.x")), rows, E,
                                     _ptr(gamma), eps, _ptr(_chk(dx, _bf16, "ln.dx")),
                                     _ptr(_chk(dgamma, _f32, "dgamma")), _ptr(_chk(dbeta, _f32, "dbeta")),
                                     _ptr(dx_drop), _ptr(dsum), _dp(drop), _stream()), "tnr_layernorm_bwd")
    return dx


@_timed
def colsum(x, out):
    lib = _ready(x)
    _lib.check(lib.tnr_colsum_bf16(_ptr(_chk(x, _bf16, "colsum.x")), x.shape[0], x.shape[1], x.stride(0),
                                   _ptr(_chk(out, _f32, "colsum.out")), _stream()), "tnr_colsum_bf16")
    return out


def _chk_relbias(relpos, A, L):
    _chk(relpos, _f32, "relpos")
    if tuple(relpos.shape) != (A, 2 * L - 1) or not relpos.is_contiguous():
        raise _lib.TinyRecError(f"attention: rel-pos bias must be contiguous fp32 [A, 2L-1] = [{A}, {2 * L - 1}], "
                                f"got {tuple(relpos.shape)}")


@_timed
def attn_fwd(qkv, x, L, relpos, ctx, A, drop=None):
    """qkv bf16 [n*L, 3E]; x int64 [n, 2L] (mask = columns L..2L); relpos fp32 [A, 2L-1] (bias of key j for
    query i at index (j - i) + L - 1).  L <= 32: one warp per (news, head); 32 < L <= 512: streamed-KV kernel."""
    lib = _ready(qkv)
    n = x.shape[0]
    E = qkv.shape[1] // 3
    mask_ptr = ctypes.c_void_p(x.data_ptr() + 8 * L)
    _chk_relbias(relpos, A, L)
    _lib.check(lib.tnr_attn_relpos_fwd(_ptr(_chk(qkv, _bf16, "attn.qkv")), mask_ptr, x.stride(0),
                                       _ptr(_chk(relpos, _f32, "relpos")), _ptr(_chk(ctx, _bf16, "ctx")),
                                       n, L, A, E, _dp(drop), _stream()), "tnr_attn_relpos_fwd")
    return ctx


_attn_ws = {}


@_timed
def attn_bwd(qkv, x, L, relpos, dctx, dqkv, A, drop=None, dbias=None, workspace=None):
    """dqkv from dctx; ``dbias`` fp32 [3E] (optional) += column sums of dqkv (the [bq|bk|bv] gradient).
    L > 32 needs ``workspace`` fp32 [2 * n * A * L] (row statistics between the two kernels); one cached per
    (device, size) is used when none is passed."""
    n = x.shape[0]
    lib = _ready(qkv, 1 if L <= 32 else 2)
    E = qkv.shape[1] // 3
    mask_ptr = ctypes.c_void_p(x.data_ptr() + 8 * L)
    _chk_relbias(relpos, A, L)
    if L > 32 and workspace is None:
        key = (qkv.device, 2 * n * A * L)
        workspace = _attn_ws.get(key)
        if workspace is None:
            _attn_ws.clear()
            workspace = _attn_ws[key] = torch.empty(2 * n * A * L, device=qkv.device, dtype=_f32)
    if workspace is not None:
        _chk(workspace, _f32, "attn.workspace")
        if workspace.numel() < 2 * n * A * L:
            raise _lib.TinyRecError("attn_bwd: workspace too small")
    _lib.check(lib.tnr_attn_relpos_bwd(_ptr(_chk(qkv, _bf16, "attn.qkv")), mask_ptr, x.stride(0),
                                       _ptr(relpos), _ptr(_chk(dctx, _bf16, "dctx")),
                                       _ptr(_chk(dqkv, _bf16, "dqkv")), _ptr(dbias), _ptr(workspace), n, L, A, E, _dp(drop),
                                       _stream()),
               "tnr_attn_relpos_bwd")
    return dqkv


@_timed
def attnpool_fwd(x, e, Q, w2, b2, mask, out, a_out, n, S):
    """x bf16 [n*S, C]; e bf16 [n*S, ldq]; out bf16 [n, C]; a_out fp32 [n, S]."""
    lib = _ready(x)
    C = x.shape[1]
    _lib.check(lib.tnr_attnpool_fwd(_ptr(_chk(x, _bf16, "pool.x")), _ptr(_chk(e, _bf16, "pool.e")), e.stride(0), Q,
                                    _ptr(_chk(w2, _f32, "w2")), _ptr(_chk(b2, _f32, "b2")), _ptr(mask),
                                    _ptr(_chk(out, _bf16, "pool.out")), _ptr(_chk(a_out, _f32, "a_out")),
                                    n, S, C, _stream()), "tnr_attnpool_fwd")
    return out


@_timed
def attnpool_bwd(x, e, Q, w2, a_in, dout, dx, du, dw2, db2, n, S):
    lib = _ready(x)
    C = x.shape[1]
    _lib.check(lib.tnr_attnpool_bwd(_ptr(x), _ptr(e), e.stride(0), Q, _ptr(w2), _ptr(_chk(a_in, _f32, "a_in")),
                                    _ptr(_chk(dout, _f32, "dout")), _ptr(_chk(dx, _bf16, "dx")),
                                    _ptr(_chk(du, _bf16, "du")), _ptr(_chk(dw2, _f32, "dw2")),
                                    _ptr(_chk(db2, _f32, "db2")), n, S, C, _stream()), "tnr_attnpool_bwd")


# ---- fp32 inference path of the news encoder (tnr_split_bf16x3 + the four fp32 row / attention kernels) ----------
@_timed
def split_bf16x3(x, out, weight=False, gelu=False):
    """x fp32 [rows, K] (unit inner stride) -> out bf16 [rows, 3K] contiguous: [hi | lo | hi] for an activation,
    [hi | hi | lo] for a weight (``weight``); ``gelu`` applies the exact erf-GELU first."""
    lib = _ready(x)
    _chk(x, _f32, "split.x"); _chk(out, _bf16, "split.out")
    rows, K = x.shape
    if x.stride(1) != 1 or tuple(out.shape) != (rows, 3 * K) or not out.is_contiguous():
        raise _lib.TinyRecError(f"split_bf16x3: x {tuple(x.shape)} -> out must be contiguous [{rows}, {3 * K}], "
                                f"got {tuple(out.shape)}")
    _lib.check(lib.tnr_split_bf16x3(_ptr(x), rows, K, x.stride(0), _lib.SPLIT_WEIGHT if weight else _lib.SPLIT_ACT,
                                    int(bool(gelu)), _ptr(out), _stream()), "tnr_split_bf16x3")
    return out


def _chk_rows_f32(name, *ts):
    for t in ts:
        _chk(t, _f32, name)
        if not t.is_contiguous():
            raise _lib.TinyRecError(f"{name}: fp32 operands must be contiguous")


@_timed
def embed_ln_f32(x, L, word, pos, type0, gamma, beta, eps, out):
    """x: int64 [n, 2L] (ids | mask), fp32 word table [vocab, E] -> out fp32 [n*L, E]."""
    lib = _ready(x)
    _chk(x, torch.int64, "embed_ln_f32.x")
    _chk_rows_f32("embed_ln_f32", word, pos, type0, gamma, beta, out)
    n, E = x.shape[0], word.shape[1]
    if tuple(out.shape) != (n * L, E) or x.stride(1) != 1:
        raise _lib.TinyRecError("embed_ln_f32: shape / layout mismatch")
    _lib.check(lib.tnr_embed_ln_fwd_f32(_ptr(x), x.stride(0), n, L, word.shape[0], _ptr(word), _ptr(pos), _ptr(type0),
                                        _ptr(gamma), _ptr(beta), eps, E, _ptr(out), _stream()), "tnr_embed_ln_fwd_f32")
    return out


@_timed
def add_layernorm_f32(x, residual, gamma, beta, eps, out):
    """out = LayerNorm(x + residual), fp32 [rows, E]."""
    lib = _ready(x)
    _chk_rows_f32("add_layernorm_f32", x, residual, gamma, beta, out)
    rows, E = x.shape
    if residual.shape != x.shape or out.shape != x.shape:
        raise _lib.TinyRecError("add_layernorm_f32: shape mismatch")
    _lib.check(lib.tnr_add_layernorm_f32(_ptr(x), _ptr(residual), rows, E, _ptr(gamma), _ptr(beta), eps, _ptr(out),
                                         _stream()), "tnr_add_layernorm_f32")
    return out


@_timed
def attn_fwd_f32(qkv, x, L, relpos, ctx, A):
    """qkv fp32 [n*L, 3E]; x int64 [n, 2L] (mask = columns L..2L); relpos fp32 [A, 2L-1] -> ctx fp32 [n*L, E]."""
    lib = _ready(qkv)
    n = x.shape[0]
    E = qkv.shape[1] // 3
    _chk_rows_f32("attn_fwd_f32", qkv, ctx)
    _chk(x, torch.int64, "attn_fwd_f32.x")
    _chk_relbias(relpos, A, L)
    if qkv.shape[0] != n * L or tuple(ctx.shape) != (n * L, E) or x.stride(1) != 1:
        raise _lib.TinyRecError("attn_fwd_f32: shape / layout mismatch")
    mask_ptr = ctypes.c_void_p(x.data_ptr() + 8 * L)
    _lib.check(lib.tnr_attn_relpos_fwd_f32(_ptr(qkv), mask_ptr, x.stride(0), _ptr(relpos), _ptr(ctx), n, L, A, E,
                                           _stream()), "tnr_attn_relpos_fwd_f32")
    return ctx


@_timed
def attnpool_fwd_f32(x, u, Q, w2, b2, out, n, S):
    """x fp32 [n*S, C]; u fp32 [n*S, ldq] (fc1 pre-activation, bias included) -> out fp32 [n, C]."""
    lib = _ready(x)
    _chk_rows_f32("attnpool_fwd_f32", x, w2, b2, out)
    _chk(u, _f32, "attnpool_fwd_f32.u")
    C = x.shape[1]
    if u.stride(1) != 1 or x.shape[0] != n * S or u.shape[0] != n * S or u.shape[1] < Q or tuple(out.shape) != (n, C):
        raise _lib.TinyRecError("attnpool_fwd_f32: shape / layout mismatch")
    _lib.check(lib.tnr_attnpool_fwd_f32(_ptr(x), _ptr(u), u.stride(0), Q, _ptr(w2), _ptr(b2), _ptr(out), n, S, C,
                                        _stream()), "tnr_attnpool_fwd_f32")
    return out


@_timed
def cast_f32_bf16(x, y):
    lib = _ready(x)
    _lib.check(lib.tnr_cast_f32_bf16(_ptr(_chk(x, _f32, "cast.x")), _ptr(_chk(y, _bf16, "cast.y")), x.numel(),
                                     _stream()), "tnr_cast_f32_bf16")
    return y


@_timed
def user_encoder_fwd(vecs, mask, pad_doc, W1, b1, w2, b2, use_mask, user, a_out, e_out, B, H, *, fp32=False):
    """vecs fp32 [B*H, D] (contiguous rows), mask fp32 [B, H] -> user [B, D], a [B, H], e [B, H, Q].
    ``fp32``: the fc1 contraction to fp32 accuracy (3xTF32, tnr_user_encoder_fwd_f32) instead of TF32."""
    lib = _ready(vecs)
    D, Q = W1.shape[1], W1.shape[0]
    for t, nm in ((vecs, "vecs"), (mask, "mask"), (pad_doc, "pad_doc"), (W1, "W1"), (b1, "b1"), (w2, "w2"), (b2, "b2"),
                  (user, "user"), (a_out, "a")):
        _chk(t, _f32, "user_encoder." + nm)
    name = "tnr_user_encoder_fwd_f32" if fp32 else "tnr_user_encoder_fwd"
    _lib.check(getattr(lib, name)(_ptr(vecs), _ptr(mask), _ptr(pad_doc), _ptr(W1), _ptr(b1), _ptr(w2), _ptr(b2),
                                  int(use_mask), _ptr(user), _ptr(a_out), _ptr(e_out), B, H, D, Q, _stream()), name)
    return user


@_timed
def user_encoder_fwd_gather(table, idx, mask, pad_doc, W1, b1, w2, b2, use_mask, user, a_out=None, *, fp32=False):
    """user[b] = user_encoder(table[idx[b, :]], mask[b]) with the row gather fused into the kernel.
    table fp32 [n_rows, D], idx int32 [B, H], mask fp32 [B, H] -> user fp32 [B, D].  ``fp32`` as in user_encoder_fwd."""
    lib = _ready(table)
    B, H = idx.shape
    D, Q = W1.shape[1], W1.shape[0]
    for t, nm in ((table, "table"), (mask, "mask"), (pad_doc, "pad_doc"), (W1, "W1"), (b1, "b1"), (w2, "w2"), (b2, "b2"),
                  (user, "user")):
        _chk(t, _f32, "user_encoder_gather." + nm)
    _chk(idx, torch.int32, "user_encoder_gather.idx")
    if table.shape[1] != D or not table.is_contiguous() or not idx.is_contiguous() or tuple(mask.shape) != (B, H):
        raise _lib.TinyRecError("user_encoder_fwd_gather: shape / layout mismatch")
    name = "tnr_user_encoder_fwd_gather_f32" if fp32 else "tnr_user_encoder_fwd_gather"
    _lib.check(getattr(lib, name)(_ptr(table), table.shape[0], _ptr(idx), _ptr(mask), _ptr(pad_doc), _ptr(W1), _ptr(b1),
                                  _ptr(w2), _ptr(b2), int(use_mask), _ptr(user), _ptr(a_out), B, H, D, Q, _stream()), name)
    return user


MAX_HISTORY = 512          # longest user history (user_log_length) the user-encoder and NRMS kernels take


def check_history_length(H):
    """Reject a history length the user-encoder kernels cannot take, before anything is staged or launched."""
    if not 1 <= H <= MAX_HISTORY:
        raise _lib.TinyRecError(f"user_log_length={H} is not supported (1..{MAX_HISTORY})")


def user_encoder_score_supported(B, H, D, Q):
    """Shapes the flat scoring path takes (tnr_user_encoder_score); small batches stay on the per-impression kernel."""
    return B >= 64 and H <= MAX_HISTORY and D % 32 == 0 and D <= 256 and Q <= 208


def user_encoder_pack_w1(W1, pad_doc, b1, w2, packed=None):
    """att_fc1.weight fp32 [Q, D] (+ pad_doc [D], att_fc1.bias [Q], att_fc2.weight [Q]) -> the packed image
    tnr_user_encoder_score reads: W1 TF32-rounded in the swizzled shared-memory layout, W1 pad_doc, the pad_doc logit."""
    lib = _ready(W1, 2)
    Q, D = W1.shape
    n = int(lib.tnr_user_encoder_packed_w1_floats(D))
    if packed is None or packed.numel() != n:
        packed = torch.empty(n, device=W1.device, dtype=_f32)
    for t, nm in ((W1, "W1"), (pad_doc, "pad_doc"), (b1, "b1"), (w2, "w2")):
        _chk(t, _f32, "pack_w1." + nm)
    _lib.check(lib.tnr_user_encoder_pack_w1(_ptr(W1.contiguous()), _ptr(pad_doc.contiguous()), _ptr(b1.contiguous()),
                                            _ptr(w2.contiguous()), _ptr(packed), D, Q, _stream()),
               "tnr_user_encoder_pack_w1")
    return packed


_score_ws = {}


@_timed
def user_encoder_score(vecs, idx, mask, pad_doc, w1_packed, Q, b1, w2, b2, use_mask, user, a_out, B, H):
    """Scoring path: vecs fp32 [B*H, D] (idx None) or the [N, D] table with idx int32 [B, H]; mask fp32 [B, H]
    -> user fp32 [B, D], a_out fp32 [B, H]."""
    lib = _ready(vecs, 3)
    D = vecs.shape[1]
    for t, nm in ((vecs, "vecs"), (mask, "mask"), (pad_doc, "pad_doc"), (w1_packed, "w1_packed"), (b1, "b1"), (w2, "w2"),
                  (b2, "b2"), (user, "user"), (a_out, "a")):
        _chk(t, _f32, "user_encoder_score." + nm)
    if idx is not None:
        _chk(idx, torch.int32, "user_encoder_score.idx")
        if tuple(idx.shape) != (B, H) or not idx.is_contiguous():
            raise _lib.TinyRecError("user_encoder_score: idx must be contiguous int32 [B, H]")
    elif vecs.shape[0] != B * H:
        raise _lib.TinyRecError("user_encoder_score: vecs must be [B*H, D]")
    if not vecs.is_contiguous() or tuple(mask.shape) != (B, H) or a_out.numel() != B * H or user.numel() != B * D:
        raise _lib.TinyRecError("user_encoder_score: shape / layout mismatch")
    nbytes = int(lib.tnr_user_encoder_score_ws_bytes(B, H))
    key = (vecs.device, nbytes)
    ws = _score_ws.get(key)
    if ws is None:
        _score_ws.clear()
        ws = _score_ws[key] = torch.empty(nbytes, device=vecs.device, dtype=torch.uint8)
    _lib.check(lib.tnr_user_encoder_score(_ptr(vecs), vecs.shape[0], _ptr(idx), _ptr(mask), _ptr(pad_doc), _ptr(w1_packed),
                                          _ptr(b1), _ptr(w2), _ptr(b2), int(use_mask), _ptr(user), _ptr(a_out), _ptr(ws),
                                          B, H, D, Q, _stream()), "tnr_user_encoder_score")
    return user


@_timed
def user_encoder_fwd_multi(encoders, mask, use_mask, B, H):
    """One launch for several user encoders sharing ``mask``.  ``encoders``: list of dicts with
    vecs [B*H, D], pad_doc [D], W1 [Q, D], b1 [Q], w2 [Q], b2 [1], user [B, D], a [B, H], e [B, H, Q] | None."""
    lib = _ready(mask, 1)
    n = len(encoders)
    arr = (_lib.UserEncoderIO * n)()
    D, Q = encoders[0]["W1"].shape[1], encoders[0]["W1"].shape[0]
    for io, enc in zip(arr, encoders):
        for k in ("vecs", "pad_doc", "W1", "b1", "w2", "b2", "user", "a"):
            _chk(enc[k], _f32, "user_encoder." + k)
        if tuple(enc["W1"].shape) != (Q, D) or not enc["W1"].is_contiguous():
            raise _lib.TinyRecError("user_encoder_fwd_multi: all encoders must share [Q, D] contiguous fc1 weights")
        io.vecs, io.pad_doc, io.W1, io.b1 = enc["vecs"].data_ptr(), enc["pad_doc"].data_ptr(), enc["W1"].data_ptr(), enc["b1"].data_ptr()
        io.w2, io.b2, io.user, io.a_out = enc["w2"].data_ptr(), enc["b2"].data_ptr(), enc["user"].data_ptr(), enc["a"].data_ptr()
        io.e_out = enc["e"].data_ptr() if enc.get("e") is not None else None
    _lib.check(lib.tnr_user_encoder_fwd_multi(arr, n, _ptr(_chk(mask, _f32, "user_encoder.mask")), int(use_mask), B, H, D, Q,
                                              _stream()), "tnr_user_encoder_fwd_multi")


@_timed
def user_encoder_bwd(vecs, mask, pad_doc, W1, w2, use_mask, a_in, e_in, d_user, d_vecs, dpad, dW1, db1, dw2, db2, scratch, B, H):
    lib = _ready(vecs, 2)
    D, Q = W1.shape[1], W1.shape[0]
    for t, nm in ((d_user, "d_user"), (d_vecs, "d_vecs"), (dpad, "dpad"), (dW1, "dW1"), (db1, "db1"), (dw2, "dw2"),
                  (db2, "db2"), (a_in, "a"), (e_in, "e"), (scratch, "scratch")):
        _chk(t, _f32, "user_encoder_bwd." + nm)
    if scratch.numel() < B * H * (Q + D):
        raise _lib.TinyRecError("user_encoder_bwd: scratch too small")
    _lib.check(lib.tnr_user_encoder_bwd(_ptr(vecs), _ptr(mask), _ptr(pad_doc), _ptr(W1), _ptr(w2), int(use_mask),
                                        _ptr(a_in), _ptr(e_in), _ptr(d_user), _ptr(d_vecs), _ptr(dpad), _ptr(dW1),
                                        _ptr(db1), _ptr(dw2), _ptr(db2), _ptr(scratch), B, H, D, Q, _stream()),
               "tnr_user_encoder_bwd")


@_timed
def kd_loss(s_news, s_user, label, T_ext, TP_ext, M, B, H, K, D, temperature, coef, want_grad, score_out, losses,
            d_news, d_user, G_ext):
    lib = _ready(s_news)
    _chk(label, torch.int64, "kd_loss.label")
    for t, nm in ((s_news, "s_news"), (s_user, "s_user"), (score_out, "score"), (losses, "losses")):
        _chk(t, _f32, "kd_loss." + nm)
    if losses.numel() < 4 + 4 * B + 1:
        raise _lib.TinyRecError("kd_loss: losses must hold 4 + 4B + 1 floats (zero-initialised once)")
    _lib.check(lib.tnr_kd_loss_fwdbwd(_ptr(s_news), _ptr(s_user), _ptr(label), _ptr(T_ext), _ptr(TP_ext), M, B, H, K, D,
                                      float(temperature), float(coef), int(want_grad), _ptr(score_out), _ptr(losses),
                                      _ptr(d_news), _ptr(d_user), _ptr(G_ext), _stream()), "tnr_kd_loss_fwdbwd")


@_timed
def sgemm_nt(A, Bm, bias, C, M, N, K, batch, sA, sB, sbias, sC, *, fp32=False):
    """C[b][M,N] = A[b][M,K] . B[b][N,K]^T + bias[b][N] on the TF32 tensor path; ``fp32``: to fp32 accuracy (3xTF32)."""
    lib = _ready(A)
    name = "tnr_sgemm_nt_f32" if fp32 else "tnr_sgemm_nt"
    _lib.check(getattr(lib, name)(_ptr(_chk(A, _f32, "sgemm.A")), _ptr(_chk(Bm, _f32, "sgemm.B")), _ptr(bias),
                                  _ptr(_chk(C, _f32, "sgemm.C")), M, N, K, batch, sA, sB, sbias, sC, _stream()), name)


@_timed
def sgemm_tn_acc(A, Bm, C, cbias, R, N1, N2, batch, sA, sB, sC, sbias):
    lib = _ready(A)
    _lib.check(lib.tnr_sgemm_tn_acc(_ptr(_chk(A, _f32, "sgemm.A")), _ptr(_chk(Bm, _f32, "sgemm.B")),
                                    _ptr(_chk(C, _f32, "sgemm.C")), _ptr(cbias), R, N1, N2, batch, sA, sB, sC, sbias,
                                    _stream()), "tnr_sgemm_tn_acc")


@_timed
def sgemm_nn(A, Bm, C, M, N, K, parts=1, sA=0, sB=0):
    """C[M,N] = sum_p A[p][M,K] . B[p][K,N]   (fp32, TF32 tensor path)."""
    lib = _ready(A)
    _lib.check(lib.tnr_sgemm_nn(_ptr(_chk(A, _f32, "sgemm_nn.A")), _ptr(_chk(Bm, _f32, "sgemm_nn.B")),
                                _ptr(_chk(C, _f32, "sgemm_nn.C")), M, N, K, parts, sA, sB, _stream()), "tnr_sgemm_nn")


# ---- NRMS user encoder (model_bert.py:37-100) ------------------------------------------------------
@_timed
def nrms_blend_fwd(vecs, mask, pad_doc, out):
    """out = vecs * m + pad_doc * (1 - m);  vecs / out fp32 [R, D], mask fp32 [R]."""
    lib = _ready(vecs)
    R, D = vecs.shape
    for t, nm in ((vecs, "vecs"), (mask, "mask"), (pad_doc, "pad_doc"), (out, "out")):
        _chk(t, _f32, "nrms_blend_fwd." + nm)
    if mask.numel() != R or pad_doc.numel() != D or not vecs.is_contiguous() or not out.is_contiguous():
        raise _lib.TinyRecError("nrms_blend_fwd: shape / layout mismatch")
    _lib.check(lib.tnr_nrms_blend_fwd(_ptr(vecs), _ptr(mask), _ptr(pad_doc), _ptr(out), R, D, _stream()), "tnr_nrms_blend_fwd")
    return out


@_timed
def nrms_blend_bwd(d_blend, mask, d_vecs, dpad):
    """d_vecs += d_blend * m, dpad += sum_r d_blend (1 - m);  mask None: d_vecs += d_blend."""
    lib = _ready(d_blend)
    R, D = d_blend.shape
    for t, nm in ((d_blend, "d_blend"), (d_vecs, "d_vecs")):
        _chk(t, _f32, "nrms_blend_bwd." + nm)
    if not d_blend.is_contiguous() or not d_vecs.is_contiguous() or d_vecs.numel() != R * D:
        raise _lib.TinyRecError("nrms_blend_bwd: shape / layout mismatch")
    _lib.check(lib.tnr_nrms_blend_bwd(_ptr(d_blend), _ptr(mask), _ptr(d_vecs), _ptr(dpad), R, D, _stream()), "tnr_nrms_blend_bwd")


def _nrms_planes(qkv, B, H):
    _chk(qkv, _f32, "nrms.qkv")
    if qkv.dim() != 3 or qkv.shape[0] != 3 or qkv.shape[1] != B * H or qkv.shape[2] % 16 or not qkv.is_contiguous():
        raise _lib.TinyRecError(f"nrms: qkv must be contiguous fp32 [3, B*H, n_heads*16], got {tuple(qkv.shape)}")
    return qkv.shape[2] // 16


@_timed
def nrms_attn_fwd(qkv, mask, ctx, B, H):
    """qkv fp32 [3, B*H, Dh] planes, mask fp32 [B, H] or None -> ctx fp32 [B*H, Dh]."""
    lib = _ready(qkv)
    heads = _nrms_planes(qkv, B, H)
    _chk(ctx, _f32, "nrms.ctx")
    _lib.check(lib.tnr_nrms_attn_fwd(_ptr(qkv[0]), _ptr(qkv[1]), _ptr(qkv[2]), _ptr(mask), _ptr(ctx), B, H, heads, _stream()),
               "tnr_nrms_attn_fwd")
    return ctx


@_timed
def nrms_attn_bwd(qkv, mask, d_ctx, dqkv, B, H):
    lib = _ready(qkv)
    heads = _nrms_planes(qkv, B, H)
    _nrms_planes(dqkv, B, H)
    _chk(d_ctx, _f32, "nrms.d_ctx")
    _lib.check(lib.tnr_nrms_attn_bwd(_ptr(qkv[0]), _ptr(qkv[1]), _ptr(qkv[2]), _ptr(mask), _ptr(d_ctx), _ptr(dqkv[0]),
                                     _ptr(dqkv[1]), _ptr(dqkv[2]), B, H, heads, _stream()), "tnr_nrms_attn_bwd")


@_timed
def adam_amsgrad(p, g, m, v, vmax, shadow, lr, beta1, beta2, eps, step, grad_scale=1.0):
    lib = _ready(p)
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v")) + (((vmax, "vmax"),) if vmax is not None else ()):
        _chk(t, _f32, "adam." + nm)
    _lib.check(lib.tnr_adam_amsgrad(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(vmax), _ptr(shadow), p.numel(), lr, beta1,
                                    beta2, eps, step, grad_scale, _stream()), "tnr_adam_amsgrad")


@_timed
def adam_amsgrad_devstep(p, g, m, v, vmax, shadow, lr, beta1, beta2, eps, step_dev, bc_ws, grad_scale=1.0, advance=True):
    """Adam(amsgrad) with the step counter on the device (int32 [1]): graph-capturable.  ``advance`` increments the
    counter and refreshes the bias corrections first; a second range of the same step passes ``advance=False``."""
    lib = _ready(p, 2 if advance else 1)
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v"), (bc_ws, "bc_ws")) + (((vmax, "vmax"),) if vmax is not None else ()):
        _chk(t, _f32, "adam." + nm)
    _chk(step_dev, torch.int32, "adam.step_dev")
    _lib.check(lib.tnr_adam_amsgrad_devstep(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(vmax), _ptr(shadow), p.numel(), lr, beta1,
                                            beta2, eps, _ptr(step_dev), _ptr(bc_ws), grad_scale, int(bool(advance)),
                                            _stream()),
               "tnr_adam_amsgrad_devstep")


def host_copy(dst, src, n_threads=4):
    """dst: CPU tensor (pinned staging) <- src: C-contiguous numpy array of the same dtype, element for element into
    dst's first src.size elements; the bytes are split over ``n_threads`` host threads (tnr_host_copy_mt; the GIL is
    released for the call)."""
    import numpy as np
    src = np.ascontiguousarray(src)
    nbytes = src.size * src.itemsize
    if dst.is_cuda or not dst.is_contiguous() or dst.numel() * dst.element_size() < nbytes or dst.element_size() != src.itemsize:
        raise _lib.TinyRecError("host_copy: dst must be a contiguous CPU tensor of the source's element size, large enough")
    _lib.check(_lib.load().tnr_host_copy_mt(ctypes.c_void_p(dst.data_ptr()), ctypes.c_void_p(src.ctypes.data), nbytes,
                                            int(n_threads)), "tnr_host_copy_mt")
    return dst


def allreduce_p2p(ptrs_dev, multicast_ptr, flags_dev, rank, world, off, n, n_ctas):
    """In-place sum all-reduce of floats [off, off + n) of a symmetric fp32 buffer over NVLink peer memory
    (tnr_allreduce_p2p); ``ptrs_dev`` / ``flags_dev`` are device addresses of the per-rank pointer tables,
    ``multicast_ptr`` the NVLS multicast address of the buffer (0: peer loads / stores)."""
    lib = _lib.load()
    stats.launches += 1
    _lib.check(lib.tnr_allreduce_p2p(ctypes.c_void_p(int(ptrs_dev)), ctypes.c_void_p(int(multicast_ptr) or None),
                                     ctypes.c_void_p(int(flags_dev)), int(rank), int(world), int(off), int(n), int(n_ctas),
                                     _stream()), "tnr_allreduce_p2p")


def set_sm_reserve(n_sms, device=None):
    """SMs the persistent GEMM grids leave free on ``device`` from now on (0 = all SMs): tnr_set_sm_reserve."""
    lib = _lib.load()
    if device is not None and torch.cuda.current_device() != torch.device(device).index:
        with torch.cuda.device(device):
            _lib.check(lib.tnr_set_sm_reserve(int(n_sms)), "tnr_set_sm_reserve")
        return
    _lib.check(lib.tnr_set_sm_reserve(int(n_sms)), "tnr_set_sm_reserve")


@_timed
def gather_rows_i32_i64(table, idx, out):
    """out int64 [n, W] = table int32 [N, W][idx int32 [n]]"""
    lib = _ready(table)
    _chk(table, torch.int32, "gather.table"); _chk(idx, torch.int32, "gather.idx"); _chk(out, torch.int64, "gather.out")
    _lib.check(lib.tnr_gather_rows_i32_i64(_ptr(table), table.shape[0], _ptr(idx), idx.numel(), table.shape[1], _ptr(out),
                                           _stream()), "tnr_gather_rows_i32_i64")
    return out


@_timed
def train_batch_gather(news, teacher_tables, hist_idx, cand_idx, tokens_out, teacher_out):
    """One launch: tokens_out int64 [n_hist + n_cand, W] = news[idx] and teacher_out[i][r, :] = teacher_tables[i][idx[r]]
    for idx = [hist_idx | cand_idx] (tnr_train_batch_gather).  teacher_out: tensors [n_hist + n_cand (+ extra), D]."""
    lib = _ready(news)
    _chk(news, torch.int32, "batch_gather.news"); _chk(hist_idx, torch.int32, "batch_gather.hist_idx")
    _chk(cand_idx, torch.int32, "batch_gather.cand_idx"); _chk(tokens_out, torch.int64, "batch_gather.tokens")
    M = len(teacher_tables)
    nh, nc, W = hist_idx.numel(), cand_idx.numel(), news.shape[1]
    if tokens_out.numel() != (nh + nc) * W or not tokens_out.is_contiguous() or len(teacher_out) != M:
        raise _lib.TinyRecError("train_batch_gather: shape / layout mismatch")
    D = teacher_tables[0].shape[1] if M else 4
    tabs = (ctypes.c_void_p * max(M, 1))()
    outs = (ctypes.c_void_p * max(M, 1))()
    ld = D
    for i in range(M):
        _chk(teacher_tables[i], _f32, "batch_gather.teacher"); _chk(teacher_out[i], _f32, "batch_gather.teacher_out")
        if teacher_tables[i].shape[1] != D or teacher_out[i].shape[-1] != D or teacher_out[i].stride(-1) != 1:
            raise _lib.TinyRecError("train_batch_gather: teacher tables / outputs must share the row width")
        tabs[i], outs[i] = teacher_tables[i].data_ptr(), teacher_out[i].data_ptr()
        ld = teacher_out[i].stride(-2)
    _lib.check(lib.tnr_train_batch_gather(_ptr(news), news.shape[0], W, tabs, outs, M, D, ld, _ptr(hist_idx), nh, _ptr(cand_idx), nc,
                                          _ptr(tokens_out), _stream()), "tnr_train_batch_gather")


@_timed
def gather_rows_f32(table, idx, out, out_ld=None):
    lib = _ready(table)
    _chk(table, _f32, "gather.table"); _chk(idx, torch.int32, "gather.idx"); _chk(out, _f32, "gather.out")
    D = table.shape[1]
    _lib.check(lib.tnr_gather_rows_f32(_ptr(table), table.shape[0], _ptr(idx), idx.numel(), D, _ptr(out),
                                       D if out_ld is None else out_ld, _stream()), "tnr_gather_rows_f32")
    return out


_eval_ws = {}


@_timed
def eval_metrics(table, user, ptr, cand, label, max_c, per_imp, sums=None, score_out=None):
    """table fp32 [N, D]; user fp32 [n_imp, D]; ptr int64 [n_imp+1]; cand int32 [nnz]; label int8 [nnz];
    ``score_out`` fp32 [nnz] receives the dot scores (a cached workspace is used when None)."""
    lib = _ready(table, 3 if sums is not None else 2)
    _chk(table, _f32, "eval.table"); _chk(user, _f32, "eval.user"); _chk(ptr, torch.int64, "eval.ptr")
    _chk(cand, torch.int32, "eval.cand"); _chk(label, torch.int8, "eval.label"); _chk(per_imp, torch.float64, "eval.per_imp")
    n_imp = ptr.numel() - 1
    nnz = cand.numel()
    if label.numel() != nnz or user.shape[0] < n_imp or per_imp.numel() < 5 * n_imp or not table.is_contiguous():
        raise _lib.TinyRecError("eval_metrics: shape / layout mismatch")
    if score_out is None:
        key = table.device
        score_out = _eval_ws.get(key)
        if score_out is None or score_out.numel() < nnz:
            score_out = _eval_ws[key] = torch.empty(max(nnz, 1 << 16), device=table.device, dtype=_f32)
    else:
        _chk(score_out, _f32, "eval.score_out")
        if score_out.numel() < nnz:
            raise _lib.TinyRecError("eval_metrics: score_out must hold nnz floats")
    _lib.check(lib.tnr_eval_metrics(_ptr(table), table.shape[0], _ptr(user), _ptr(ptr), _ptr(cand), _ptr(label), n_imp, nnz,
                                    table.shape[1], int(max_c), _ptr(per_imp), _ptr(sums), _ptr(score_out), _stream()),
               "tnr_eval_metrics")
    return per_imp


@_timed
def doc_sim(table, pairs, sum_out):
    """sum_out (fp64 [1]) += sum of cos(table[i], table[j]) over the int32 [P, 2] pairs with i != j."""
    lib = _ready(table)
    _chk(table, _f32, "doc_sim.table")
    _chk(pairs, torch.int32, "doc_sim.pairs")
    _chk(sum_out, torch.float64, "doc_sim.sum")
    if pairs.dim() != 2 or pairs.shape[1] != 2 or not pairs.is_contiguous() or not table.is_contiguous():
        raise _lib.TinyRecError("doc_sim: pairs must be contiguous int32 [P, 2]")
    _lib.check(lib.tnr_doc_sim(_ptr(table), table.shape[0], _ptr(pairs), pairs.shape[0], table.shape[1], _ptr(sum_out),
                               _stream()), "tnr_doc_sim")
    return sum_out
