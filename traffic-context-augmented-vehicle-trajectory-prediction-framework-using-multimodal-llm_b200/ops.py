"""Thin torch-tensor front end of the C ABI in include/tcavp.h.

torch is used for device memory and streams only: every function here hands raw device pointers to
libtcavp.so and raises TcavpError on a non-zero return code.  Nothing falls back to torch math."""
import ctypes
import os as _os
from ctypes import POINTER, Structure, byref, c_float, c_int, c_longlong, c_uint32, c_void_p

import torch

from . import lib as _lib

F32, BF16, E4M3 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_SWIGLU, ACT_SWIGLU_BWD, ACT_GELU_TANH = 0, 1, 2, 3, 4
_DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float8_e4m3fn: E4M3}


class GemmArgs(Structure):
    _fields_ = [("M", c_int), ("N", c_int), ("K", c_int),
                ("A", c_void_p), ("lda", c_int),
                ("W", c_void_p), ("ldw", c_int),
                ("in_dtype", c_int),
                ("out", c_void_p), ("ldo", c_int), ("out_dtype", c_int),
                ("bias", c_void_p),
                ("residual", c_void_p), ("ldr", c_int), ("res_dtype", c_int),
                ("act", c_int),
                ("remap_gi", c_int), ("remap_go", c_int), ("remap_off", c_int),
                ("rope_cos_sin", c_void_p), ("rope_L", c_int), ("rope_dh", c_int), ("rope_cols", c_int),
                ("row_scale", c_void_p),
                ("sumsq_out", c_void_p), ("row_sumsq", c_void_p), ("sumsq_inv_cols", c_float), ("sumsq_eps", c_float),
                ("aux_out", c_void_p), ("ld_aux", c_int),
                ("col_scale", c_void_p)]


class AttnArgs(Structure):
    _fields_ = [("B", c_int), ("H", c_int), ("Hkv", c_int), ("Tq", c_int), ("Tk", c_int), ("dh", c_int),
                ("q", c_void_p), ("q_sb", c_longlong), ("q_st", c_longlong),
                ("k", c_void_p), ("k_sb", c_longlong), ("k_st", c_longlong),
                ("v", c_void_p), ("v_sb", c_longlong), ("v_st", c_longlong),
                ("out", c_void_p), ("o_sb", c_longlong), ("o_st", c_longlong),
                ("dtype", c_int), ("scale", c_float), ("causal", c_int), ("key_mask", c_void_p),
                ("drop_seed", c_void_p), ("drop_site", c_uint32), ("drop_thresh", c_uint32), ("drop_scale", c_float)]


class Drop:
    """One dropout site of a train-mode pass: (device seed tensor uint32[2], site id, p).  The mask is a pure function of
    (seed, site, element index) — include/tcavp.h: tcavp_dropout — so the backward pass re-creates it from the same Drop."""
    __slots__ = ("seed", "site", "p", "thresh", "scale")

    def __init__(self, seed, site, p):
        if seed.dtype != torch.int32 or seed.numel() != 2 or not seed.is_cuda:
            raise TypeError("Drop: seed must be a CUDA int32[2] tensor (base seed, step counter)")
        if not 0.0 <= p < 1.0:
            raise ValueError(f"dropout p = {p}")
        self.seed, self.site, self.p = seed, int(site), float(p)
        self.thresh = drop_threshold(p)
        self.scale = 1.0 / (1.0 - p)


def drop_threshold(p):
    """uint32 threshold of the mask function: an element is kept when its 32-bit hash >= thresh, P(drop) = thresh / 2^32."""
    return min(max(int(round(float(p) * 4294967296.0)), 0), 4294967295)


def _set_drop(a, drop):
    if drop is not None and drop.thresh:
        a.drop_seed, a.drop_site, a.drop_thresh, a.drop_scale = drop.seed.data_ptr(), drop.site, drop.thresh, drop.scale


_PROF = None


class LaunchProfiler:
    """Times every libtcavp launch with CUDA events on the launching stream (bench.py's roofline numbers).
    Events are recorded around each launch inside the timed region; nothing synchronises until summary()."""

    def __init__(self):
        self.rec = []

    def __enter__(self):
        global _PROF
        _PROF = self
        return self

    def __exit__(self, *a):
        global _PROF
        _PROF = None

    def add(self, kernel, flops, nbytes, e0, e1):
        self.rec.append((kernel, flops, nbytes, e0, e1))

    def summary(self):
        torch.cuda.synchronize()
        groups, base = {}, {}
        for kernel, flops, nbytes, e0, e1 in self.rec:
            ms = e0.elapsed_time(e1)
            for key, table in ((kernel, groups), (kernel.split("[")[0], base)):
                g = table.setdefault(key, dict(kernel=key, launches=0, time_ms=0.0, flops=0.0, bytes=0.0))
                g["launches"] += 1
                g["time_ms"] += ms
                g["flops"] += flops
                g["bytes"] += nbytes
        for g in list(groups.values()) + list(base.values()):
            g["avg_ms"] = g["time_ms"] / max(g["launches"], 1)
            g["tflops"] = g["flops"] / (g["time_ms"] * 1e-3) / 1e12 if g["time_ms"] > 0 else 0.0
            g["gbs"] = g["bytes"] / (g["time_ms"] * 1e-3) / 1e9 if g["time_ms"] > 0 else 0.0
        order = sorted(groups.values(), key=lambda g: -g["time_ms"])
        total = sum(g["time_ms"] for g in order) or 1.0
        brief = [dict(kernel=g["kernel"], launches=g["launches"], time_ms=round(g["time_ms"], 3), share=round(g["time_ms"] / total, 4),
                      tflops=round(g["tflops"], 1), gbs=round(g["gbs"], 1)) for g in order]
        dominant = max(base.values(), key=lambda g: g["time_ms"]) if base else None
        return {"dominant": dominant, "groups": brief}


class _Timed:
    """Records one launch with the active LaunchProfiler.  `kernel` is the label, or, for entry points where the library picks the
    kernel, a function of last_kernel() that returns (label, nbytes), called only while a profiler is active; None records nothing."""
    __slots__ = ("kernel", "flops", "nbytes", "e0")

    def __init__(self, kernel, flops=0.0, nbytes=0.0):
        self.kernel, self.flops, self.nbytes = kernel, flops, nbytes

    def __enter__(self):
        if _PROF is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *a):
        if _PROF is not None and self.kernel is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            kernel, nbytes = (self.kernel, self.nbytes) if isinstance(self.kernel, str) else self.kernel(last_kernel())
            _PROF.add(kernel, self.flops, nbytes, self.e0, e1)


def _nb(*ts):
    return float(sum(t.numel() * t.element_size() for t in ts if t is not None))


def dt(t):
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype}") from None


def _p(t):
    return None if t is None else c_void_p(t.data_ptr())


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.TcavpError("tcavp ops need CUDA tensors (there is no CPU fallback)")


# Long contractions (K >= 2048: down_proj, every 7B-class projection, the dX GEMMs of the fine-tune step) have two tcgen05 kernels: the
# 512 x 256 "wide" CTA-pair tile and the double-buffered 256 x 256 pair tile.  Which one wins is a property of the board, not of the shape:
# wide is 6-15 % ahead on some B200s, the pair tile 6-12 % ahead on others of the same pool and power cap (profiles/wide_vs_pair_r02y.txt).
# So the first long-K GEMM of a process times both for ~0.1 s each on this GPU and keeps the faster (TCAVP_GEMM_WIDE_K pins it instead).
_ROUTE = {"wide_k": None, "tuned": None}


def _long_k_gemm(M, N, K):
    """True for the bf16 problems tcavp_gemm sends to the wide kernel when the threshold allows it: a long contraction and at least
    four waves of 512 x 256 tiles on 148 SMs.  Must match the condition in tcavp_gemm (gemm.cu): it is the only routing decision
    this module repeats, to run autotune_gemm_route() before the first such GEMM."""
    return N > 128 and K >= 2048 and M >= 8192 and ((M + 511) // 512) * ((N + 255) // 256) >= 4 * 74


def autotune_gemm_route(budget_ms=120.0):
    """Sets the wide-kernel routing threshold of tcavp_gemm from a sustained A/B on the current device; returns the decision dict."""
    lib = _lib.load()
    env = _os.environ.get("TCAVP_GEMM_WIDE_K")
    if env is not None or torch.cuda.is_current_stream_capturing():
        if _ROUTE["wide_k"] is None:
            _ROUTE["wide_k"] = int(lib.tcavp_gemm_wide_min_k(-1))
            _ROUTE["tuned"] = {"source": "TCAVP_GEMM_WIDE_K" if env is not None else "default (stream capture in progress)"}
        return _ROUTE["tuned"]
    global _PROF
    prof, _PROF = _PROF, None              # the probe launches are not part of any profiled step
    launches0 = launch_count()
    try:
        dev = torch.cuda.current_device()
        gen = torch.Generator(device="cuda").manual_seed(1)
        shapes = [(32768, 768, 3072), (16384, 4096, 4096)]
        ms = {2048: 0.0, 0: 0.0}
        bufs = []
        for (M, N, K) in shapes:
            a = (torch.randn(M, K, device="cuda", generator=gen) * 0.5).bfloat16()
            w = (torch.randn(N, K, device="cuda", generator=gen) * 0.05).bfloat16()
            bufs.append((a, w, torch.empty(M, N, device="cuda", dtype=torch.bfloat16)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for rnd in range(2):               # A-B-A-B: clock drift of the warming GPU hits both variants alike
            for wk in (2048, 0):
                lib.tcavp_gemm_wide_min_k(wk)
                for (a, w, o) in bufs:
                    g = GemmArgs()
                    g.M, g.N, g.K = a.shape[0], w.shape[0], a.shape[1]
                    g.A, g.lda, g.W, g.ldw, g.in_dtype = a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), BF16
                    g.out, g.ldo, g.out_dtype, g.act = o.data_ptr(), o.stride(0), BF16, ACT_NONE
                    _lib.check(lib.tcavp_gemm(byref(g), _stream()), "tcavp_gemm")
                    e0.record()
                    _lib.check(lib.tcavp_gemm(byref(g), _stream()), "tcavp_gemm")
                    e1.record()
                    e1.synchronize()
                    n = max(3, min(400, int(budget_ms / 2 / max(e0.elapsed_time(e1), 1e-3))))
                    e0.record()
                    for _ in range(n):
                        lib.tcavp_gemm(byref(g), _stream())
                    e1.record()
                    e1.synchronize()
                    ms[wk] += e0.elapsed_time(e1) / n
        wide_k = 2048 if ms[2048] <= ms[0] else 0
        lib.tcavp_gemm_wide_min_k(wide_k)
        _ROUTE["wide_k"] = wide_k
        _ROUTE["tuned"] = {"source": "autotune", "device": dev, "wide_ms": round(ms[2048], 4), "pair_ms": round(ms[0], 4),
                           "long_k_kernel": "gemm_tc_wide_kernel" if wide_k else "gemm_tc_pair_kernel", "probe_launches": launch_count() - launches0}
    finally:
        _PROF = prof
    return _ROUTE["tuned"]


def gemm(a, w, out, *, M=None, N=None, K=None, lda=None, ldw=None, ldo=None, bias=None, residual=None, ldr=None,
         act=ACT_NONE, remap=(0, 0, 0), rope=None, row_scale=None, aux_out=None, sumsq_out=None, row_sumsq=None, col_scale=None):
    """out = act(a @ w.T + bias) + residual.  a: [M, >=K] row-major (lda = a.stride(0)), w: [N, >=K].
    float8_e4m3fn operands need `col_scale` (fp32 [N], the weight rows' dequantisation factors) and usually `row_scale` (the activation
    rows' factors from quant_e4m3_rows): out = act(acc * row_scale[m] * col_scale[n] + bias) + residual."""
    _need_cuda(a, w, out, bias, residual, col_scale)
    g = GemmArgs()
    g.M = a.shape[0] if M is None else M
    g.N = w.shape[0] if N is None else N
    g.K = a.shape[1] if K is None else K
    g.A, g.lda = a.data_ptr(), (a.stride(0) if lda is None else lda)
    g.W, g.ldw = w.data_ptr(), (w.stride(0) if ldw is None else ldw)
    if a.dtype != w.dtype:
        raise TypeError(f"gemm: a is {a.dtype}, w is {w.dtype}")
    g.in_dtype = dt(a)
    g.out, g.ldo, g.out_dtype = out.data_ptr(), (out.stride(0) if ldo is None else ldo), dt(out)
    g.bias = None if bias is None else bias.data_ptr()
    if bias is not None and bias.dtype != torch.float32:
        raise TypeError("gemm: bias must be fp32")
    if residual is not None:
        g.residual, g.ldr, g.res_dtype = residual.data_ptr(), (residual.stride(0) if ldr is None else ldr), dt(residual)
    g.act = act
    g.remap_gi, g.remap_go, g.remap_off = remap
    if row_scale is not None:
        if row_scale.dtype != torch.float32:
            raise TypeError("gemm: row_scale must be fp32")
        g.row_scale = row_scale.data_ptr()
    if sumsq_out is not None:   # += per-row sum of squares of the final output (int64 Q44.20 [rows], zeroed by the caller)
        if sumsq_out.dtype != torch.int64:
            raise TypeError("gemm: sumsq_out must be int64 (64-bit fixed point, 20 fractional bits)")
        g.sumsq_out = sumsq_out.data_ptr()
    if row_sumsq is not None:   # (tensor int64 Q44.20 [M], columns, eps): row factor rsqrt(sumsq / columns + eps)
        t, ncols, eps = row_sumsq
        if t.dtype != torch.int64:
            raise TypeError("gemm: row_sumsq must be int64 (64-bit fixed point, 20 fractional bits)")
        g.row_sumsq, g.sumsq_inv_cols, g.sumsq_eps = t.data_ptr(), 1.0 / ncols, eps
    if aux_out is not None:  # SwiGLU: raw gate/up accumulators (bf16, interleaved) for the backward pass
        if aux_out.dtype != torch.bfloat16:
            raise TypeError("gemm: aux_out must be bf16")
        g.aux_out, g.ld_aux = aux_out.data_ptr(), aux_out.stride(0)
    if rope is not None:     # (table, L, dh, cols)
        g.rope_cos_sin, g.rope_L, g.rope_dh, g.rope_cols = rope[0].data_ptr(), rope[1], rope[2], rope[3]
    if col_scale is not None:
        if col_scale.dtype != torch.float32:
            raise TypeError("gemm: col_scale must be fp32")
        g.col_scale = col_scale.data_ptr()
    if g.in_dtype == BF16 and _ROUTE["wide_k"] is None and _long_k_gemm(g.M, g.N, g.K):
        autotune_gemm_route()
    esz = a.element_size()
    nbytes = float(g.M * g.K * esz + g.N * g.K * esz + g.M * g.N * out.element_size())

    def label(kern):
        if kern == "gemm_simt_kernel":
            return kern, nbytes
        # small-M pair launches (the Q-Former's 16 query rows per scene) are reported apart from the token-stream launches of the same [N, K]
        m = "M%d," % g.M if kern.startswith("gemm_tc_pair_kernel") and g.M < 32768 else ""
        return "%s[%sN%d,K%d]" % (kern, m, g.N, g.K), nbytes

    with _Timed(label if g.M > 0 else None, 2.0 * g.M * g.N * g.K):      # M = 0: tcavp_gemm checks the arguments and launches nothing
        _lib.check(_lib.load().tcavp_gemm(byref(g), _stream()), "tcavp_gemm")
    return out


def attention(q, k, v, out, *, B, H, Hkv, Tq, Tk, dh, q_strides, k_strides, v_strides, o_strides, scale, causal=False,
              key_mask=None, drop=None):
    """q/k/v/out are tensors whose data_ptr() is element (0,0,0,0); *_strides = (batch stride, time stride) in elements."""
    _need_cuda(q, k, v, out, key_mask)
    a = AttnArgs()
    a.B, a.H, a.Hkv, a.Tq, a.Tk, a.dh = B, H, Hkv, Tq, Tk, dh
    a.q, (a.q_sb, a.q_st) = q.data_ptr(), q_strides
    a.k, (a.k_sb, a.k_st) = k.data_ptr(), k_strides
    a.v, (a.v_sb, a.v_st) = v.data_ptr(), v_strides
    a.out, (a.o_sb, a.o_st) = out.data_ptr(), o_strides
    a.dtype, a.scale, a.causal = dt(q), scale, int(causal)
    if key_mask is not None:
        if key_mask.dtype != torch.int32:
            raise TypeError("attention: key_mask must be int32")
        a.key_mask = key_mask.data_ptr()
    _set_drop(a, drop)
    fl = 4.0 * B * H * Tq * Tk * dh * (0.5 if causal else 1.0)

    def label(kern):
        # algorithmic bytes: q read + out written + k and v read once (ONE pass when the keys are the values: attn_xt_kernel)
        nbytes = q.element_size() * B * dh * (2.0 * H * Tq + (1.0 if kern == "attn_xt_kernel" else 2.0) * Hkv * Tk)
        if kern == "attn_tm_kernel":
            return f"{kern}[dh{dh},L{Tq}]", nbytes
        return (kern if kern == "attn_x_kernel" else f"{kern}[dh{dh},q{Tq},k{Tk}]"), nbytes

    with _Timed(label if B > 0 and Tq > 0 else None, fl):      # an empty problem launches nothing
        _lib.check(_lib.load().tcavp_attention(byref(a), _stream()), "tcavp_attention")
    return out


def layernorm(x, w, b, out, *, residual=None, eps=1e-5, remap=(0, 0, 0), rowvec=None, rows=None, cols=None):
    _need_cuda(x, w, b, out, residual, rowvec)
    rows = x.numel() // x.shape[-1] if rows is None else rows
    cols = x.shape[-1] if cols is None else cols
    with _Timed("layernorm_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size() + (residual.element_size() if residual is not None else 0)))):
        _lib.check(_lib.load().tcavp_layernorm(_p(x), _p(residual), _p(w), _p(b), _p(out), rows, cols, c_float(eps), dt(x), dt(out),
                                           remap[0], remap[1], remap[2], _p(rowvec), _stream()), "tcavp_layernorm")
    return out


def layernorm_strided(x, w, b, out, *, rows, cols, eps=1e-5, ldx=None, ldo=None):
    """LayerNorm (no residual) with row strides: `out` may be the leading columns of a wider buffer."""
    _need_cuda(x, w, b, out)
    with _Timed("layernorm_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size()))):
        _lib.check(_lib.load().tcavp_layernorm_strided(_p(x), cols if ldx is None else ldx, _p(w), _p(b), _p(out), cols if ldo is None else ldo, rows, cols,
                                                       c_float(eps), dt(x), dt(out), _stream()), "tcavp_layernorm_strided")
    return out


def rmsnorm(x, w, out, *, eps, rows=None, cols=None, ldi=None, ldo=None):
    _need_cuda(x, w, out)
    rows = x.numel() // x.shape[-1] if rows is None else rows
    cols = x.shape[-1] if cols is None else cols
    ldo = cols if ldo is None else ldo
    ldi = cols if ldi is None else ldi
    with _Timed("rmsnorm_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size()))):
        _lib.check(_lib.load().tcavp_rmsnorm(_p(x), ldi, _p(w), _p(out), rows, cols, ldo, c_float(eps), dt(x), dt(out), _stream()),
                   "tcavp_rmsnorm")
    return out


def row_rstd(x, out, *, rows, cols, ldx, eps):
    _need_cuda(x, out)
    with _Timed("row_rstd_kernel", 0.0, float(rows * cols * x.element_size())):
        _lib.check(_lib.load().tcavp_row_rstd(_p(x), ldx, rows, cols, c_float(eps), dt(x), _p(out), _stream()), "tcavp_row_rstd")
    return out


def rope_table(L, dh, theta, device, layout=0):
    """cos / sin table for positions [0, L).  `theta`: the rope base (plain rope, HF:86-88 inv_freq evaluated on the host exactly as
    transformers does) or a precomputed fp32 inv_freq[dh/2] tensor (config.rope_inv_freq: llama3 frequency scaling)."""
    if torch.is_tensor(theta):
        if theta.numel() != dh // 2:
            raise ValueError(f"rope_table: inv_freq has {theta.numel()} entries, head_dim {dh} needs {dh // 2}")
        inv = theta.to(device=device, dtype=torch.float32).contiguous()
    else:
        inv = (1.0 / (theta ** (torch.arange(0, dh, 2, dtype=torch.int64).float() / dh))).to(device)
    t = torch.empty((L, dh // 2, 2) if layout == 0 else (dh // 4, L, 4), dtype=torch.float32, device=device)
    with _Timed("rope_table_kernel"):
        _lib.check(_lib.load().tcavp_rope_table(_p(t), _p(inv), L, dh, layout, _stream()), "tcavp_rope_table")
    return t


def rope_(qkv, *, rows, L, ld, n_q_heads, n_k_heads, dh, table):
    _need_cuda(qkv, table)
    with _Timed("rope_kernel"):
        _lib.check(_lib.load().tcavp_rope(_p(qkv), rows, L, ld, n_q_heads, n_k_heads, dh, _p(table), dt(qkv), _stream()), "tcavp_rope")
    return qkv


def embed_text(ids, attn_mask, embed, text_mod, fused, mask_out, *, B, L_text, n_img, H):
    _need_cuda(ids, attn_mask, embed, text_mod, fused, mask_out)
    if ids.dtype != torch.int64 or (attn_mask is not None and attn_mask.dtype != torch.int64):
        raise TypeError("embed_text: ids / attention_mask must be int64")
    with _Timed("embed_text_kernel", 0.0, float(B * L_text * (H * (embed.element_size() + fused.element_size()) + 16))):
        _lib.check(_lib.load().tcavp_embed_text(_p(ids), _p(attn_mask), _p(embed), dt(embed), _p(text_mod), _p(fused), dt(fused),
                                            _p(mask_out), B, L_text, n_img, H, embed.shape[0], _stream()), "tcavp_embed_text")


def add_rowvec(x, rowvec, out, *, rows, cols, remap=(0, 0, 0)):
    _need_cuda(x, rowvec, out)
    with _Timed("add_rowvec_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size()))):
        _lib.check(_lib.load().tcavp_add_rowvec(_p(x), _p(rowvec), _p(out), rows, cols, dt(x), dt(out), remap[0], remap[1], remap[2],
                                            _stream()), "tcavp_add_rowvec")
    return out


def cast(x, out, *, rows, cols, ldi=None, ldo=None, in_row_mod=0):
    _need_cuda(x, out)
    with _Timed("cast_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size()))):
        _lib.check(_lib.load().tcavp_cast(_p(x), cols if ldi is None else ldi, dt(x), _p(out), cols if ldo is None else ldo, dt(out),
                                      rows, cols, in_row_mod, _stream()), "tcavp_cast")
    return out


def split3(x, out, *, rows, cols):
    """fp32 [rows, cols] -> bf16 [rows, 3 * cols] = [hi | hi | lo] (see tcavp_split_bf16x3)."""
    _need_cuda(x, out)
    if x.dtype != torch.float32 or out.dtype != torch.bfloat16:
        raise TypeError("split3: fp32 in, bf16 out")
    with _Timed("split3_kernel", 0.0, float(rows * cols * (4 + 6))):
        _lib.check(_lib.load().tcavp_split_bf16x3(_p(x), x.stride(0), _p(out), out.stride(0), _ll(rows), cols, _stream()), "tcavp_split_bf16x3")
    return out


def poly_embed(polygon, lens, w, bias, pos, out, key_mask, *, B, P, D):
    _need_cuda(polygon, lens, w, bias, pos, out, key_mask)
    with _Timed("poly_embed_kernel", 0.0, float(B * P * (8 + 4 + D * out.element_size()))):
        _lib.check(_lib.load().tcavp_poly_embed(_p(polygon), _p(lens), _p(w), _p(bias), _p(pos), _p(out), dt(out), _p(key_mask), B, P, D,
                                            _stream()), "tcavp_poly_embed")


def masked_mean(x, lens, out, *, B, P, D):
    _need_cuda(x, lens, out)
    with _Timed("masked_mean_kernel", 0.0, float(B * P * D * x.element_size() + B * D * out.element_size())):
        _lib.check(_lib.load().tcavp_masked_mean(_p(x), dt(x), _p(lens), _p(out), dt(out), B, P, D, _stream()), "tcavp_masked_mean")
    return out


def ltsf_encode(x, wt, bt, we, be, pos, enc, *, B, F, C, T_in):
    _need_cuda(x, wt, bt, we, be, pos, enc)
    with _Timed("ltsf_encode_kernel", 0.0, float(B * F * T_in * 4 + B * T_in * C * enc.element_size())):
        _lib.check(_lib.load().tcavp_ltsf_encode(_p(x), _p(wt), _p(bt), _p(we), _p(be), _p(pos), _p(enc), dt(enc), B, F, C, T_in,
                                             _stream()), "tcavp_ltsf_encode")
    return enc


def nlinear_decode(enc, wd, bd, lane_adj, dec, *, B, C, T_in, T_out):
    _need_cuda(enc, wd, bd, lane_adj, dec)
    with _Timed("nlinear_decode_kernel", 0.0, float(B * T_in * C * enc.element_size() + B * T_out * C * (dec.element_size() + (lane_adj.element_size() if lane_adj is not None else 0)))):
        _lib.check(_lib.load().tcavp_nlinear_decode(_p(enc), dt(enc), _p(wd), _p(bd), _p(lane_adj), 0 if lane_adj is None else dt(lane_adj),
                                                _p(dec), dt(dec), B, C, T_in, T_out, _stream()), "tcavp_nlinear_decode")
    return dec


def fusion_head(fused, ln_w, ln_b, w1, b1, w2, b2, wo, bo, x, decoded, *, y=None, norm_stat=None, metrics=None, per_scene=None,
                B, C, T_in, T_out, tensor_cores=False):
    """`tensor_cores`: the split-bf16 mma.sync form (d_model 64; the bf16 compute mode) instead of the exact-fp32 FFMA kernel."""
    _need_cuda(fused, x, decoded, y, norm_stat, metrics, per_scene)
    tc = tensor_cores and C == 64
    fn = _lib.load().tcavp_fusion_head_tc if tc else _lib.load().tcavp_fusion_head
    with _Timed("fusion_head_tc_kernel" if tc else "fusion_head_kernel", 0.0,      # bandwidth-bound by design: reported against the HBM peak
                float(B * T_out * C * fused.element_size() + B * 2 * T_out * 4 * (2 if y is not None else 1) + B * (2 * T_in * 4 + 16))):
        _lib.check(fn(_p(fused), dt(fused), _p(ln_w), _p(ln_b), _p(w1), _p(b1), _p(w2), _p(b2), _p(wo), _p(bo),
                      _p(x), _p(decoded), _p(y), _p(norm_stat), _p(metrics), _p(per_scene), B, C, T_in, T_out,
                      _stream()), "tcavp_fusion_head")
    return decoded


def ffn64_ln(x, w1, b1, w2, b2, ln_w, ln_b, out, *, eps=1e-5):
    """out = LayerNorm(x + w2 relu(w1 x + b1) + b2) for d_model 64 in one tcgen05 kernel (tcavp_ffn64_ln); x, out bf16 [M, 64]."""
    _need_cuda(x, w1, b1, w2, b2, ln_w, ln_b, out)
    M, F = x.shape[0], w1.shape[0]
    if x.dtype != torch.bfloat16 or w1.dtype != torch.bfloat16 or w2.dtype != torch.bfloat16 or out.dtype != torch.bfloat16:
        raise TypeError("ffn64_ln: x, w1, w2, out must be bf16")
    if x.shape[1] != 64 or tuple(w1.shape) != (F, 64) or tuple(w2.shape) != (64, F) or not (x.is_contiguous() and w1.is_contiguous() and w2.is_contiguous() and out.is_contiguous()):
        raise ValueError("ffn64_ln: contiguous x [M, 64], w1 [F, 64], w2 [64, F]")
    with _Timed("ffn64_ln_kernel[F%d]" % F, 4.0 * M * 64 * F, float(2 * M * 64 * 2 + 2 * F * 64 * 2)):
        _lib.check(_lib.load().tcavp_ffn64_ln(_p(x), _p(w1), _p(b1), _p(w2), _p(b2), _p(ln_w), _p(ln_b), c_float(eps), _p(out), c_longlong(M), F,
                                              _stream()), "tcavp_ffn64_ln")
    return out


def traj_metrics(decoded, y, norm_stat, metrics, per_scene, *, B, T_out):
    _need_cuda(decoded, y, norm_stat, metrics, per_scene)
    with _Timed("traj_metrics_kernel", 0.0, float(B * 2 * T_out * 4 * 2 + B * 24)):
        _lib.check(_lib.load().tcavp_traj_metrics(_p(decoded), _p(y), _p(norm_stat), _p(metrics), _p(per_scene), B, T_out, _stream()),
               "tcavp_traj_metrics")


def best_of_k(candidates, y, norm_stat, per_scene, totals, *, B, K, T_out):
    """min over K candidates of ADE / FDE / RMSE per scene (+ batch sums); candidates (B, K, 2, T_out) fp32."""
    _need_cuda(candidates, y, norm_stat, per_scene, totals)
    with _Timed("best_of_k_kernel", 0.0, float(B * (K + 1) * 2 * T_out * 4)):
        _lib.check(_lib.load().tcavp_best_of_k(_p(candidates), _p(y), _p(norm_stat), _p(per_scene), _p(totals), B, K, T_out, _stream()),
                   "tcavp_best_of_k")
    return per_scene, totals


def dropout(x, out, drop, *, rows, cols, ldi=None, ldo=None, residual=None, ldr=None, accumulate=False, scale=None):
    """out = [out +] [residual +] (keep ? x * scale : 0) with the counter-based mask of `drop` (tcavp_dropout); scale defaults to
    1 / (1 - p); x is out is allowed.  The same call on a gradient is the backward pass."""
    _need_cuda(x, out, residual)
    with _Timed("dropout_kernel", 0.0, float(rows * cols * (x.element_size() + out.element_size() * (2 if accumulate else 1) +
                                                             (residual.element_size() if residual is not None else 0)))):
        _lib.check(_lib.load().tcavp_dropout(_p(x), cols if ldi is None else ldi, dt(x), _p(residual), (cols if ldr is None else ldr),
                                             0 if residual is None else dt(residual), _p(out), cols if ldo is None else ldo, dt(out),
                                             c_longlong(rows), cols, _p(drop.seed), c_uint32(drop.site), c_uint32(drop.thresh),
                                             c_float(drop.scale if scale is None else scale), int(accumulate), _stream()), "tcavp_dropout")
    return out


def _drop_arrays(drops):
    n = len(drops)
    if not 1 <= n <= 4 or any(d.seed.data_ptr() != drops[0].seed.data_ptr() for d in drops):
        raise ValueError("LoRA dropout: 1..4 targets sharing one device seed")
    return n, (c_uint32 * n)(*[d.site for d in drops]), (c_uint32 * n)(*[d.thresh for d in drops])


def lora_a_drop(x, a, out, drops, *, M, H, r, ldx=None, ldo=None):
    """out[:, :len(drops) * r] = sum_h keep_t(m H + h) x[m, h] a[j, h] (target t = j // r): peft's lora_A(dropout(x)) for every target in
    one pass over x (tcavp_lora_a_drop); `a` carries 1 / (1 - p)."""
    _need_cuda(x, a, out)
    n, sites, th = _drop_arrays(drops)
    with _Timed("lora_a_drop_kernel", 0.0, float(M * H * x.element_size())):
        _lib.check(_lib.load().tcavp_lora_a_drop(_p(x), x.stride(0) if ldx is None else ldx, _p(a), a.stride(0), _p(out), out.stride(0) if ldo is None else ldo,
                                                 c_longlong(M), H, r, n, _p(drops[0].seed), sites, th, _stream()), "tcavp_lora_a_drop")
    return out


def lora_dx_drop(dT, a, dx, drops, *, M, H, r, lddt=None, lddx=None):
    """dx[m, h] += sum_t keep_t(m H + h) (dT_t . a_t)[m, h] in place (tcavp_lora_dx_drop)."""
    _need_cuda(dT, a, dx)
    n, sites, th = _drop_arrays(drops)
    with _Timed("lora_dx_drop_kernel", 0.0, float(2 * M * H * dx.element_size())):
        _lib.check(_lib.load().tcavp_lora_dx_drop(_p(dT), dT.stride(0) if lddt is None else lddt, _p(a), a.stride(0), _p(dx), dx.stride(0) if lddx is None else lddx,
                                                  c_longlong(M), H, r, n, _p(drops[0].seed), sites, th, _stream()), "tcavp_lora_dx_drop")
    return dx


def lora_da_drop(x, dT, out, drops, *, M, H, r, ldx=None, lddt=None, row_scale=None):
    """out[h, j] += sum_m row_scale[m] keep_t(m H + h) x[m, h] dT[m, j] (fp32, zeroed by the caller; tcavp_lora_da_drop)."""
    _need_cuda(x, dT, out, row_scale)
    n, sites, th = _drop_arrays(drops)
    with _Timed("dw_tc_drop_kernel", 0.0, float(M * H * x.element_size())):
        _lib.check(_lib.load().tcavp_lora_da_drop(_p(x), x.stride(0) if ldx is None else ldx, _p(dT), dT.stride(0) if lddt is None else lddt, _p(row_scale),
                                                  _p(out), out.stride(0), c_longlong(M), H, r, n, _p(drops[0].seed), sites, th, _stream()), "tcavp_lora_da_drop")
    return out


def ce_loss(logits, targets, loss_sum, grad=None, *, scale=1.0):
    """loss_sum[0] += sum over rows of (logsumexp(row) - row[target]); grad (optional, bf16 / fp32 [rows, V]) = (softmax - onehot) * scale."""
    _need_cuda(logits, targets, loss_sum, grad)
    if logits.dtype != torch.float32 or targets.dtype != torch.int64 or loss_sum.dtype != torch.float32:
        raise TypeError("ce_loss: fp32 logits, int64 targets, fp32 loss_sum")
    rows, V = logits.shape
    if grad is not None and (grad.shape[0] != rows or grad.shape[1] < V):
        raise ValueError("ce_loss: grad must be [rows, >= V]")
    with _Timed("ce_loss_kernel", 0.0, float(rows * V * (4 + (grad.element_size() if grad is not None else 0)))):
        _lib.check(_lib.load().tcavp_ce_loss(_p(logits), c_longlong(logits.stride(0)), _p(targets), _p(loss_sum), _p(grad),
                                             c_longlong(grad.stride(0) if grad is not None else 0), dt(grad) if grad is not None else 0,
                                             c_longlong(rows), V, c_float(scale), _stream()), "tcavp_ce_loss")
    return loss_sum


def quant_e4m3_rows(x, q, f, *, rows=None, cols=None, ldi=None, ldo=None, rms_eps=None):
    """q = e4m3(x * 448 / amax(row)) (float8_e4m3fn [rows, >=cols]), f = amax / 448 per row (fp32 [rows]); with `rms_eps` the row's
    LlamaRMSNorm factor rsqrt(mean(x^2) + eps) is folded into f.  x: bf16 [rows, >=cols]."""
    _need_cuda(x, q, f)
    if x.dtype != torch.bfloat16 or q.dtype != torch.float8_e4m3fn or f.dtype != torch.float32:
        raise TypeError(f"quant_e4m3_rows: x bf16, q float8_e4m3fn, f fp32 (got {x.dtype}, {q.dtype}, {f.dtype})")
    rows = x.shape[0] if rows is None else rows
    cols = x.shape[1] if cols is None else cols
    with _Timed("quant_e4m3_kernel[%d]" % cols, 0.0, float(rows * (cols * 3 + 4))):
        _lib.check(_lib.load().tcavp_quant_e4m3_rows(_p(x), c_int(x.stride(0) if ldi is None else ldi), _p(q), c_int(q.stride(0) if ldo is None else ldo),
                                                     _p(f), c_int(rows), c_int(cols), c_int(0 if rms_eps is None else 1),
                                                     c_float(0.0 if rms_eps is None else rms_eps), _stream()), "tcavp_quant_e4m3_rows")
    return q, f


def launch_count():
    return int(_lib.load().tcavp_launch_count())


def last_kernel():
    """Name of the kernel the most recent op on this thread launched last (which variant a shape was routed to)."""
    return _lib.load().tcavp_last_kernel().decode()


def device_info():
    sm, maj, mnr = c_int(), c_int(), c_int()
    _lib.check(_lib.load().tcavp_device_info(byref(sm), byref(maj), byref(mnr)), "tcavp_device_info")
    return sm.value, maj.value, mnr.value


# --------------------------------------------------------------------------------------------------
# fine-tune step: backward kernels (include/tcavp.h, "fine-tune step")
# --------------------------------------------------------------------------------------------------
from ctypes import c_longlong as _ll  # noqa: E402


def _call(name, kernel, *args, flops=0.0, nbytes=0.0):
    with _Timed(kernel, flops, nbytes):
        _lib.check(getattr(_lib.load(), name)(*args, _stream()), name)


def transpose(x, out, *, rows, cols, ldi=None, ldo=None, batch=1, in_bstride=0, out_bstride=0):
    """out[b][c][r] = x[b][r][c]."""
    _need_cuda(x, out)
    _call("tcavp_transpose", "transpose_kernel", _p(x), _ll(in_bstride), cols if ldi is None else ldi, dt(x), _p(out), _ll(out_bstride),
          rows if ldo is None else ldo, dt(out), batch, rows, cols, nbytes=float(batch * rows * cols * (x.element_size() + out.element_size())))
    return out


def period_sum(x, out, *, rows, cols, period=1, ldx=None):
    """out[r % period][c] += x[r][c] (out fp32, accumulated)."""
    _need_cuda(x, out)
    if out.dtype != torch.float32:
        raise TypeError("period_sum: out must be fp32")
    _call("tcavp_period_sum", "period_sum_kernel", _p(x), cols if ldx is None else ldx, dt(x), _ll(rows), cols, period, _p(out))
    return out


def relu_bwd(dy, y, dx, *, rows, cols, lddy=None, ldy=None, lddx=None):
    _need_cuda(dy, y, dx)
    if not (dy.dtype == y.dtype == dx.dtype):
        raise TypeError("relu_bwd: dtype mismatch")
    _call("tcavp_relu_bwd", "relu_bwd_kernel", _p(dy), cols if lddy is None else lddy, _p(y), cols if ldy is None else ldy, _p(dx),
          cols if lddx is None else lddx, dt(dy), _ll(rows), cols)
    return dx


def axpby(a, out, *, rows, cols, alpha=1.0, b=None, beta=1.0, lda=None, ldb=None, ldo=None):
    _need_cuda(a, b, out)
    _call("tcavp_axpby", "axpby_kernel", _p(a), cols if lda is None else lda, dt(a), c_float(alpha), _p(b), cols if ldb is None else ldb,
          0 if b is None else dt(b), c_float(beta), _p(out), cols if ldo is None else ldo, dt(out), _ll(rows), cols)
    return out


def swiglu(gu, out, *, rows, I):
    _need_cuda(gu, out)
    _call("tcavp_swiglu", "swiglu_kernel", _p(gu), _p(out), dt(gu), _ll(rows), I)
    return out


def swiglu_bwd(dout, gu, dgu, *, rows, I):
    _need_cuda(dout, gu, dgu)
    _call("tcavp_swiglu_bwd", "swiglu_bwd_kernel", _p(dout), _p(gu), _p(dgu), dt(gu), _ll(rows), I)
    return dgu


def gelu_tanh(x, out, *, rows, cols, ldx=None, ldo=None):
    """out = gelu_new(x) (HF ACT2FN["gelu_new"], GPT-2 mlp.act) as a pass of its own (the fine-tune step keeps the pre-activation)."""
    _need_cuda(x, out)
    if x.dtype != out.dtype:
        raise TypeError("gelu_tanh: dtype mismatch")
    _call("tcavp_gelu_tanh", "gelu_new_kernel", _p(x), cols if ldx is None else ldx, _p(out), cols if ldo is None else ldo, dt(x), _ll(rows), cols)
    return out


def gelu_tanh_bwd(dy, x, dx, *, rows, cols, lddy=None, ldx=None, lddx=None):
    """dx = dy * gelu_new'(x) on the stored pre-activation x."""
    _need_cuda(dy, x, dx)
    if not (dy.dtype == x.dtype == dx.dtype):
        raise TypeError("gelu_tanh_bwd: dtype mismatch")
    _call("tcavp_gelu_tanh_bwd", "gelu_new_bwd_kernel", _p(dy), cols if lddy is None else lddy, _p(x), cols if ldx is None else ldx, _p(dx),
          cols if lddx is None else lddx, dt(x), _ll(rows), cols)
    return dx


def layernorm_bwd(dy, x, w, *, residual=None, eps=1e-5, dx=None, dw=None, db=None, rows=None, cols=None):
    _need_cuda(dy, x, w, residual, dx, dw, db)
    rows = x.numel() // x.shape[-1] if rows is None else rows
    cols = x.shape[-1] if cols is None else cols
    _call("tcavp_layernorm_bwd", "layernorm_bwd_kernel", _p(dy), dt(dy), _p(x), _p(residual), dt(x), _p(w), rows, cols, c_float(eps), _p(dx),
          0 if dx is None else dt(dx), _p(dw), _p(db))
    return dx


def layernorm_bwd_dx(dy, x, w, dx, *, rows, cols, eps=1e-5, add=None, lddy=None, ldx=None, ldadd=None, lddx=None):
    """dx = LayerNorm backward w.r.t. its input (frozen LayerNorm: no dw / db) [+ add]."""
    _need_cuda(dy, x, w, dx, add)
    if not (dy.dtype == x.dtype == dx.dtype) or (add is not None and add.dtype != x.dtype):
        raise TypeError("layernorm_bwd_dx: dtype mismatch")
    _call("tcavp_layernorm_bwd_dx", "layernorm_bwd_dx_kernel", _p(dy), cols if lddy is None else lddy, _p(x), cols if ldx is None else ldx, _p(w),
          _p(add), cols if ldadd is None else ldadd, _p(dx), cols if lddx is None else lddx, dt(x), rows, cols, c_float(eps),
          nbytes=float(rows * cols * x.element_size() * (4 if add is not None else 3)))
    return dx


def rmsnorm_bwd(dy, x, dx, *, rows, cols, eps, w=None, add=None, lddy=None, ldx=None, ldadd=None, lddx=None):
    _need_cuda(dy, x, dx, w, add)
    _call("tcavp_rmsnorm_bwd", "rmsnorm_bwd_kernel", _p(dy), cols if lddy is None else lddy, _p(x), cols if ldx is None else ldx, _p(w),
          _p(add), cols if ldadd is None else ldadd, _p(dx), cols if lddx is None else lddx, dt(x), rows, cols, c_float(eps))
    return dx


def rope_adjacent_(buf, *, rows, L, ld, cols, dh, table, inverse=False):
    _need_cuda(buf, table)
    _call("tcavp_rope_adjacent", "rope_adjacent_kernel", _p(buf), dt(buf), _ll(rows), L, ld, cols, dh, _p(table), int(inverse))
    return buf


def copy_rows(x, out, *, rows, cols, ldi=None, ldo=None, in_remap=(0, 0, 0), out_remap=(0, 0, 0)):
    _need_cuda(x, out)
    _call("tcavp_copy_rows", "copy_rows_kernel", _p(x), cols if ldi is None else ldi, dt(x), *in_remap, _p(out), cols if ldo is None else ldo,
          dt(out), *out_remap, _ll(rows), cols)
    return out


def masked_mean_bwd(dout, lens, dx, *, B, P, D):
    _need_cuda(dout, lens, dx)
    _call("tcavp_masked_mean_bwd", "masked_mean_bwd_kernel", _p(dout), dt(dout), _p(lens), _p(dx), dt(dx), B, P, D)
    return dx


def nlinear_bwd(g, *, B, C, T_in, T_out, x_in=None, w=None, din=None, dw=None):
    _need_cuda(g, x_in, w, din, dw)
    _call("tcavp_nlinear_bwd", "nlinear_bwd_kernel", _p(g), dt(g), _p(x_in), 0 if x_in is None else dt(x_in), _p(w), _p(din),
          0 if din is None else dt(din), _p(dw), B, C, T_in, T_out)


def head_assemble(o, x, decoded, *, B, T_in, T_out):
    _need_cuda(o, x, decoded)
    _call("tcavp_head_assemble", "head_assemble_kernel", _p(o), _p(x), _p(decoded), B, T_in, T_out)
    return decoded


def traj_loss_bwd(decoded, y, norm_stat, d_o, *, B, T_out, gscale=None):
    _need_cuda(decoded, y, norm_stat, d_o, gscale)
    _call("tcavp_traj_loss_bwd", "traj_loss_bwd_kernel", _p(decoded), _p(y), _p(norm_stat), _p(gscale), _p(d_o), B, T_out)
    return d_o


def skinny_dw(Y, Z, out, *, M, N, J, ldy=None, ldz=None, ldo=None, row_scale=None):
    """out[n][j] += sum_m row_scale[m] * Y[m][n] * Z[m][j]   (out fp32)."""
    _need_cuda(Y, Z, out, row_scale)
    tc = Y.dtype == torch.bfloat16 and Z.dtype == torch.bfloat16 and N % 8 == 0 and J % 8 == 0
    _call("tcavp_skinny_dw", "dw_tc_kernel[lora]" if tc else "skinny_dw_kernel", _p(Y), N if ldy is None else ldy, dt(Y), _p(Z), J if ldz is None else ldz, dt(Z),
          _p(row_scale), _p(out), J if ldo is None else ldo, _ll(M), N, J, flops=2.0 * M * N * J, nbytes=float(M * N * Y.element_size()))
    return out


def dw(dy, x, out, *, M, N, K, lddy=None, ldx=None, ldo=None):
    """out[n][k] += sum_m dy[m][n] * x[m][k]   (out fp32, zero-initialised by the caller; no transposes)."""
    _need_cuda(dy, x, out)
    if out.dtype != torch.float32:
        raise TypeError("dw: out must be fp32")
    tc = (dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and N % 8 == 0 and K % 8 == 0 and dy.data_ptr() % 16 == 0 and
          x.data_ptr() % 16 == 0 and (dy.stride(0) if lddy is None else lddy) % 8 == 0 and (x.stride(0) if ldx is None else ldx) % 8 == 0)
    _call("tcavp_dw", "dw_tc_kernel" if tc else "dw_simt_kernel", _p(dy), dy.stride(0) if lddy is None else lddy, dt(dy), _p(x), x.stride(0) if ldx is None else ldx, dt(x),
          _p(out), out.stride(0) if ldo is None else ldo, _ll(M), N, K, flops=2.0 * M * N * K,
          nbytes=float(M * (N * dy.element_size() + K * x.element_size())))
    return out


def attention_bwd(q, k, v, dout, dq, dk, dv, *, B, H, Hkv, Tq, Tk, dh, q_strides, k_strides, v_strides, do_strides, dq_strides,
                  dk_strides, dv_strides, scale, causal=False, key_mask=None, o=None, o_strides=None, drop=None):
    """dk / dv: fp32 accumulators (zeroed by the caller).  o = the forward output (enables the tensor-core kernel)."""
    _need_cuda(q, k, v, dout, dq, dk, dv, key_mask, o)
    if dk.dtype != torch.float32 or dv.dtype != torch.float32:
        raise TypeError("attention_bwd: dk / dv must be fp32")
    a = AttnArgs()
    a.B, a.H, a.Hkv, a.Tq, a.Tk, a.dh = B, H, Hkv, Tq, Tk, dh
    a.q, (a.q_sb, a.q_st) = q.data_ptr(), q_strides
    a.k, (a.k_sb, a.k_st) = k.data_ptr(), k_strides
    a.v, (a.v_sb, a.v_st) = v.data_ptr(), v_strides
    a.dtype, a.scale, a.causal = dt(q), scale, int(causal)
    if key_mask is not None:
        a.key_mask = key_mask.data_ptr()
    _set_drop(a, drop)
    tc = False
    if o is not None:
        a.out, (a.o_sb, a.o_st) = o.data_ptr(), o_strides
        tc = a.dtype == BF16 and H == Hkv and dh in (16, 32, 64, 96, 128) and max(Tq, Tk) <= 256
    fl = 10.0 * B * H * Tq * Tk * dh * (0.5 if causal else 1.0)
    with _Timed(f"attn_bwd_{'tc_' if tc else ''}kernel[dh{dh},q{Tq},k{Tk}]", fl, 0.0):
        _lib.check(_lib.load().tcavp_attention_bwd(byref(a), _p(dout), _ll(do_strides[0]), _ll(do_strides[1]), _p(dq), _ll(dq_strides[0]),
                                                   _ll(dq_strides[1]), _p(dk), _ll(dk_strides[0]), _ll(dk_strides[1]), _p(dv),
                                                   _ll(dv_strides[0]), _ll(dv_strides[1]), _stream()), "tcavp_attention_bwd")


def attention_bwd_owned_ok(q, *, H, Hkv, Tq, Tk, dh, o, causal=False):
    """True when tcavp_attention_bwd_owned (tensor-core kernel, dk / dv stored directly in the activation dtype) covers the shape."""
    if q.dtype != torch.bfloat16 or H != Hkv:
        return False
    if o is not None and dh in (16, 32, 64, 96, 128) and max(Tq, Tk) <= 256:
        return True
    return dh % 64 == 0 and Tq <= 64 and Tk <= 256 and not causal


def attention_bwd_owned(q, k, v, dout, dq, dk, dv, *, B, H, Tq, Tk, dh, q_strides, k_strides, v_strides, do_strides, dq_strides,
                        dk_strides, dv_strides, scale, causal=False, key_mask=None, o=None, o_strides=None, drop=None):
    """dk / dv are written (not accumulated) in their own dtype, e.g. straight into the packed d(qkv) buffer."""
    _need_cuda(q, k, v, dout, dq, dk, dv, key_mask, o)
    if dk.dtype != dv.dtype:
        raise TypeError("attention_bwd_owned: dk / dv dtypes differ")
    a = AttnArgs()
    a.B, a.H, a.Hkv, a.Tq, a.Tk, a.dh = B, H, H, Tq, Tk, dh
    a.q, (a.q_sb, a.q_st) = q.data_ptr(), q_strides
    a.k, (a.k_sb, a.k_st) = k.data_ptr(), k_strides
    a.v, (a.v_sb, a.v_st) = v.data_ptr(), v_strides
    if o is not None:
        a.out, (a.o_sb, a.o_st) = o.data_ptr(), o_strides
    a.dtype, a.scale, a.causal = dt(q), scale, int(causal)
    if key_mask is not None:
        a.key_mask = key_mask.data_ptr()
    _set_drop(a, drop)
    fl = 10.0 * B * H * Tq * Tk * dh * (0.5 if causal else 1.0)
    small = o is not None and dh in (16, 32, 64, 96, 128) and max(Tq, Tk) <= 256
    with _Timed(f"attn_{'bwd_tc' if small else 'x_bwd'}_kernel[dh{dh},q{Tq},k{Tk}]", fl, 0.0):
        _lib.check(_lib.load().tcavp_attention_bwd_owned(byref(a), _p(dout), _ll(do_strides[0]), _ll(do_strides[1]), _p(dq), _ll(dq_strides[0]),
                                                         _ll(dq_strides[1]), _p(dk), _ll(dk_strides[0]), _ll(dk_strides[1]), _p(dv),
                                                         _ll(dv_strides[0]), _ll(dv_strides[1]), dt(dk), _stream()), "tcavp_attention_bwd_owned")


def adamw_(param, grad, exp_avg, exp_avg_sq, *, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, step, grad_scale=1.0):
    _need_cuda(param, grad, exp_avg, exp_avg_sq)
    for t in (param, grad, exp_avg, exp_avg_sq):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError("adamw_: flat contiguous fp32 buffers required")
    _call("tcavp_adamw", "adamw_kernel", _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), _ll(param.numel()), c_float(lr), c_float(betas[0]),
          c_float(betas[1]), c_float(eps), c_float(weight_decay), int(step), c_float(grad_scale))
    return param


CLIP_WORKSPACE_BYTES = 9472       # include/tcavp.h: TCAVP_CLIP_WORKSPACE_BYTES


def _flat_f32(name, *ts):
    for t in ts:
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise TypeError(f"{name}: flat contiguous fp32 buffers required")


def clip_record(device):
    """A zeroed tcavp_clip_record on `device`: fp32 [total_norm, clip_coef, skip (int32 bits), reserved]."""
    return torch.zeros(4, dtype=torch.float32, device=device)


def clip_prologue(grad, record, workspace, *, grad_scale=1.0, max_norm=None, loss=None, skip_nonfinite=False):
    """record <- {total_norm = ||grad_scale * grad||_2, clip_coef (torch.nn.utils.clip_grad_norm_'s, 1 when max_norm is None),
    skip = skip_nonfinite and (total_norm or loss not finite)}.  workspace: >= CLIP_WORKSPACE_BYTES of device memory."""
    _need_cuda(grad, record, workspace, loss)
    _flat_f32("clip_prologue", grad, record, loss)
    if record.numel() != 4 or (loss is not None and loss.numel() != 1):
        raise ValueError("clip_prologue: record is fp32[4] (clip_record()), loss one fp32 value")
    _call("tcavp_clip_prologue", "clip_norm_kernel", _p(grad), _ll(grad.numel()), c_float(grad_scale), c_float(max_norm or 0.0), _p(loss),
          int(bool(skip_nonfinite)), _p(workspace), _ll(workspace.numel() * workspace.element_size()), _p(record), nbytes=_nb(grad))
    return record


def adamw_clipped_(param, grad, exp_avg, exp_avg_sq, *, record, step, skipped=None, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2,
                   grad_scale=1.0):
    """adamw_ with the clip coefficient and the skip decision of a clip_prologue record and the step number in the device int32
    counter `step` (incremented unless the step is skipped; `skipped` counts the skipped steps)."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, record, step, skipped)
    _flat_f32("adamw_clipped_", param, grad, exp_avg, exp_avg_sq, record)
    for t in (step, skipped):
        if t is not None and (t.dtype != torch.int32 or t.numel() != 1):
            raise TypeError("adamw_clipped_: step / skipped are one device int32 each")
    _call("tcavp_adamw_clipped", "adamw_clipped_kernel", _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), _ll(param.numel()), c_float(lr),
          c_float(betas[0]), c_float(betas[1]), c_float(eps), c_float(weight_decay), c_float(grad_scale), _p(record), _p(step), _p(skipped),
          nbytes=_nb(param, grad, exp_avg, exp_avg_sq) + _nb(param, exp_avg, exp_avg_sq))
    return param


def mark_nonfinite_(loss, dst):
    """dst[0] = NaN when the device scalar `loss` is not finite."""
    _need_cuda(loss, dst)
    _flat_f32("mark_nonfinite_", loss, dst)
    if loss.numel() != 1 or dst.numel() == 0:
        raise ValueError("mark_nonfinite_: loss is one value, dst not empty")
    _call("tcavp_mark_nonfinite", "mark_nonfinite_kernel", _p(loss), _p(dst))
    return dst
