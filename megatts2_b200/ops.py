"""Thin tensor-level wrappers over the C ABI (device pointers + strides in, nothing else).

PyTorch is used for device memory and streams only.  Every function raises if a
tensor is not a CUDA fp32 (or stated integer) tensor: there is no CPU path.
Activations are channels-last ``(B, T, C)`` here; the reference-facing modules
convert at their boundary.
"""
import ctypes as C
import math

import torch

from . import _lib as L

_F32 = torch.float32


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(t, dtype=_F32, name="tensor"):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise L.MttsError(f"{name}: expected a CUDA tensor (no CPU fallback in megatts2_b200)")
    if t.dtype != dtype:
        raise L.MttsError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _rows(t):
    """(B, T, C) view with unit channel stride -> (tensor, batch_stride, ld)."""
    if t.dim() == 2:
        t = t.unsqueeze(0)
    assert t.dim() == 3
    if t.stride(2) != 1 or (t.shape[1] > 1 and t.stride(1) < t.shape[2]):
        t = t.contiguous()
    return t, t.stride(0), t.stride(1) if t.shape[1] > 1 else max(t.stride(1), t.shape[2])


def empty(*shape, dtype=_F32, device=None):
    return torch.empty(*shape, dtype=dtype, device=device)


# ------------------------------------------------------------------------------ tap-GEMM
def conv1d(x, w_packed, bias=None, *, k, stride=1, dil=1, pad=0, pad_mode=L.PAD_ZERO, pre_act=L.ACT_NONE,
           pre_slope=0.0, post_act=L.ACT_NONE, post_slope=0.0, res=None, out=None, out_scale=1.0, accumulate=False,
           t_out=None, in_lens=None, w_tc=None):
    """x (B,T,Cin) channels-last, w_packed (k,Cin,Cout) -> (B,T_out,Cout).
    w_tc: optional operand planes, (3,k,Cout,Cin) bf16 [bf16x3] or (2,k,Cout,Cin) fp16 [f16x2] -> the tcgen05 engine
    is used when the shape is eligible."""
    x = _dev(x, name="x")
    x, x_sb, ldx = _rows(x)
    B, Tin, Cin = x.shape
    kk, Cin2, Cout = w_packed.shape
    assert kk == k and Cin2 == Cin, (w_packed.shape, k, Cin)
    if t_out is None:
        t_out = (Tin + 2 * pad - dil * (k - 1) - 1) // stride + 1
    if out is None:
        out = torch.empty(B, t_out, Cout, dtype=_F32, device=x.device)
    y, y_sb, ldy = _rows(_dev(out, name="out"))
    assert y.data_ptr() == out.data_ptr(), "out must have unit channel stride"
    p = L.ConvParams()
    p.x, p.x_batch_stride, p.ldx = x.data_ptr(), x_sb, ldx
    p.w = _dev(w_packed, name="w").data_ptr()
    p.bias = _dev(bias, name="bias").data_ptr() if bias is not None else None
    if res is not None:
        r, r_sb, ldr = _rows(_dev(res, name="res"))
        p.res, p.res_batch_stride, p.ldr = r.data_ptr(), r_sb, ldr
    p.y, p.y_batch_stride, p.ldy = y.data_ptr(), y_sb, ldy
    p.B, p.Tin, p.Tout, p.Cin, p.Cout = B, Tin, t_out, Cin, Cout
    p.k, p.stride, p.dil, p.pad, p.pad_mode = k, stride, dil, pad, pad_mode
    p.pre_act, p.pre_slope, p.post_act, p.post_slope = pre_act, pre_slope, post_act, post_slope
    p.out_scale, p.accumulate = out_scale, int(accumulate)
    p.in_lens = _dev(in_lens, torch.int32, "in_lens").data_ptr() if in_lens is not None else None
    if w_tc is not None:
        fmt = _plane_fmt(w_tc)
        assert w_tc.is_contiguous() and tuple(w_tc.shape) == (3 - fmt, k, Cout, Cin)
        nbytes = 6 * B * (t_out + dil * (k - 1)) * Cin + 4096
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        p.w_tc, p.tc_scratch, p.tc_scratch_bytes, p.tc_fmt = w_tc.data_ptr(), scratch.data_ptr(), nbytes, fmt
        tc_overflow_bind(x.device)
    L.check(L.lib().mtts_conv1d_f32(C.byref(p), _stream()))
    return out


def linear(x, w_packed, bias=None, **kw):
    """x (..., K) -> (..., N) with w_packed (1, K, N)."""
    shp = x.shape
    y = conv1d(x.reshape(1, -1, shp[-1]), w_packed, bias, k=1, **kw)
    return y.reshape(*shp[:-1], w_packed.shape[2])


def _plane_fmt(w_planes):
    if w_planes.dtype == torch.float16:
        return L.TC_F16X2
    if w_planes.dtype == torch.bfloat16:
        return L.TC_BF16X3
    raise L.MttsError(f"operand planes must be bf16 (bf16x3) or fp16 (f16x2), got {w_planes.dtype}")


def linear_tc(x, w_planes, bias=None, *, res=None, pre_act=L.ACT_NONE, pre_slope=0.0, post_act=L.ACT_NONE):
    """Tensor-core (tcgen05) dense layer: x (..., K) fp32, w_planes (3, N, K) bf16 [bf16x3] or (2, N, K) fp16 [f16x2]
    -> (..., N) fp32."""
    x = _dev(x, name="x")
    shp = x.shape
    x2 = x.reshape(-1, shp[-1])
    if x2.stride(1) != 1 or x2.stride(0) % 4 != 0 or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    M, K = x2.shape
    fmt = _plane_fmt(w_planes)
    npl, N, K2 = w_planes.shape
    assert K2 == K and npl == 3 - fmt and w_planes.is_contiguous()
    tc_overflow_bind(x.device)
    y = torch.empty(M, N, dtype=_F32, device=x.device)
    r2 = res.reshape(M, N) if res is not None else None
    lib = L.lib()
    nbytes = lib.mtts_linear_tc_scratch_bytes(M, K)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    L.check(lib.mtts_linear_tc_f32(_ptr(x2), x2.stride(0), M, K, _ptr(w_planes), N, _ptr(bias), _ptr(r2),
                                   r2.stride(0) if r2 is not None else 0, _ptr(y), N, pre_act, pre_slope, post_act,
                                   _ptr(scratch), nbytes, M, fmt, _stream()))
    return y.reshape(*shp[:-1], N)


def layernorm(x, gamma, beta, *, res=None, out=None, eps=1e-5, post_act=L.ACT_NONE, accumulate=False):
    x = _dev(x, name="x")
    Cc = x.shape[-1]
    x2 = x.reshape(-1, Cc)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    if out is None:
        out = torch.empty(x.shape, dtype=_F32, device=x.device)
    y2 = out.reshape(-1, Cc)
    r2 = res.reshape(-1, Cc) if res is not None else None
    L.check(L.lib().mtts_layernorm_f32(_ptr(x2), x2.stride(0), _ptr(_dev(gamma)), _ptr(_dev(beta)),
                                       _ptr(r2), r2.stride(0) if r2 is not None else 0, _ptr(y2), y2.stride(0),
                                       x2.shape[0], Cc, eps, post_act, int(accumulate), _stream()))
    return out


def attention(q, k, v, n_heads, mask=None):
    """q (B,Tq,D), k/v (B,Tk,D) (any row strides, unit channel stride) -> (B,Tq,D).
    mask: additive fp32 broadcastable to (B,H,Tq,Tk)."""
    q, k, v = _dev(q, name="q"), _dev(k, name="k"), _dev(v, name="v")
    B, Tq, D = q.shape
    Tk = k.shape[1]
    dh = D // n_heads
    for t in (q, k, v):
        assert t.stride(2) == 1
    o = torch.empty(B, Tq, D, dtype=_F32, device=q.device)
    p = L.AttnParams()
    p.q, p.q_sb, p.q_st = q.data_ptr(), q.stride(0), q.stride(1)
    p.k, p.k_sb, p.k_st = k.data_ptr(), k.stride(0), k.stride(1)
    p.v, p.v_sb, p.v_st = v.data_ptr(), v.stride(0), v.stride(1)
    p.o, p.o_sb, p.o_st = o.data_ptr(), o.stride(0), o.stride(1)
    if mask is not None:
        m = _dev(mask, name="mask")
        while m.dim() < 4:
            m = m.unsqueeze(0)
        m = m.expand(B, n_heads, Tq, Tk)
        if m.stride(3) != 1 and Tk > 1:
            m = m.contiguous()
        p.mask, p.mask_sb, p.mask_sh, p.mask_sq = m.data_ptr(), m.stride(0), m.stride(1), m.stride(2)
        keep = m
    p.B, p.H, p.Tq, p.Tk, p.dh = B, n_heads, Tq, Tk, dh
    p.scale = 1.0 / math.sqrt(dh)
    L.check(L.lib().mtts_attention_f32(C.byref(p), _stream()))
    return o


# ------------------------------------------------------------------------------ VQ
def vq_argmin(x, embed):
    """x (N, D) -> idx (N,) int64 (EuclideanCodebook.quantize)."""
    x = _dev(x, name="x")
    if x.stride(-1) != 1 or x.stride(0) % 4 != 0 or x.data_ptr() % 16 != 0:
        x = x.contiguous()
    embed = _dev(embed, name="embed").contiguous()
    idx = torch.empty(x.shape[0], dtype=torch.int64, device=x.device)
    L.check(L.lib().mtts_vq_argmin_f32(_ptr(x), x.stride(0), _ptr(embed), x.shape[0], x.shape[1], embed.shape[0],
                                       _ptr(idx), _stream()))
    return idx


def vq_gather(idx, embed, t_out=None, repeat=1, out=None):
    """idx (B, N) int64 -> (B, t_out, D) channels-last with each code repeated `repeat` times."""
    idx = _dev(idx, torch.int64, "idx").contiguous()
    embed = _dev(embed, name="embed").contiguous()
    B, N = idx.shape
    D = embed.shape[1]
    if t_out is None:
        t_out = N * repeat
    assert t_out <= N * repeat
    if out is None:
        out = torch.empty(B, t_out, D, dtype=_F32, device=idx.device)
    assert out.stride(2) == 1
    L.check(L.lib().mtts_vq_gather_f32(_ptr(idx), N, _ptr(embed), D, embed.shape[0], B, t_out, repeat,
                                       _ptr(out), out.stride(0), out.stride(1), _stream()))
    return out


# ------------------------------------------------------------------------------ misc
def maxpool_time(x, k):
    x, x_sb, ldx = _rows(_dev(x, name="x"))
    B, T, Cc = x.shape
    y = torch.empty(B, (T + k - 1) // k, Cc, dtype=_F32, device=x.device)
    L.check(L.lib().mtts_maxpool_time_f32(_ptr(x), x_sb, ldx, _ptr(y), y.stride(0), y.stride(1), B, T, Cc, k, _stream()))
    return y


def embed_pe(ids, table, pe=None, alpha=1.0, pe_offset=0):
    ids = _dev(ids, torch.int64, "ids").contiguous()
    table = _dev(table, name="table").contiguous()
    B, T = ids.shape
    D = table.shape[1]
    y = torch.empty(B, T, D, dtype=_F32, device=ids.device)
    if pe is not None:
        assert pe.shape[0] >= T + pe_offset and pe.shape[1] == D and pe.is_contiguous()
    L.check(L.lib().mtts_embed_pe_f32(_ptr(ids), T, _ptr(table), table.shape[0], D, _ptr(pe), float(alpha), pe_offset,
                                      B, T, _ptr(y), y.stride(0), y.stride(1), _stream()))
    return y


def add_pe(x, pe, alpha=1.0):
    x, x_sb, ldx = _rows(_dev(x, name="x"))
    B, T, D = x.shape
    assert pe.shape[0] >= T and pe.shape[1] == D and pe.is_contiguous()
    y = torch.empty(B, T, D, dtype=_F32, device=x.device)
    L.check(L.lib().mtts_add_pe_f32(_ptr(x), x_sb, ldx, _ptr(_dev(pe)), float(alpha), B, T, D, _ptr(y), y.stride(0),
                                    y.stride(1), _stream()))
    return y


def length_regulate(x, dur, l_out=None, return_host_totals=False):
    """x (B,Tp,D), dur (B,Tp) int32 -> (B, l_out, D), totals (B,) int32 (a host list with return_host_totals).
    l_out=None reads sum(dur) per utterance back to the host (one sync, like the reference's .numpy())."""
    x, x_sb, ldx = _rows(_dev(x, name="x"))
    dur = _dev(dur, torch.int32, "dur").contiguous()
    B, Tp, D = x.shape
    totals = torch.empty(B, dtype=torch.int32, device=x.device)
    if l_out is None:
        L.check(L.lib().mtts_length_regulate_f32(_ptr(x), x_sb, ldx, _ptr(dur), Tp, B, Tp, D, 0, None, 0, D,
                                                 _ptr(totals), _stream()))
        host_totals = totals.tolist()                 # B ints: the one host sync of the synthesis body
        l_out = max(host_totals) if host_totals else 0
    elif return_host_totals:
        host_totals = None
    y = torch.empty(B, l_out, D, dtype=_F32, device=x.device)
    L.check(L.lib().mtts_length_regulate_f32(_ptr(x), x_sb, ldx, _ptr(dur), Tp, B, Tp, D, l_out, _ptr(y),
                                             y.stride(0), y.stride(1) if l_out > 0 else D, _ptr(totals), _stream()))
    if return_host_totals:
        return y, (host_totals if host_totals is not None else totals.tolist())
    return y, totals


def mask_tail(x, keep):
    """x (B, ..., L) contiguous fp32, keep (B,) int32: zero x[b, ..., keep[b]:] in place (speechbrain mask_noise)."""
    x = _dev(x, name="x")
    assert x.is_contiguous()
    keep = _dev(keep, torch.int32, "keep").contiguous()
    B, Lx = x.shape[0], x.shape[-1]
    rows = x.numel() // max(B * Lx, 1)
    L.check(L.lib().mtts_mask_tail_f32(_ptr(x), B, rows, Lx, _ptr(keep), _stream()))
    return x


def to_channels_last(x_bct, pad_rep=0):
    """(B, C, T) any strides -> contiguous (B, T + 2*pad_rep, C)."""
    x = _dev(x_bct, name="x")
    B, Cc, T = x.shape
    y = torch.empty(B, T + 2 * pad_rep, Cc, dtype=_F32, device=x.device)
    L.check(L.lib().mtts_copy_strided_f32(_ptr(x), x.stride(0), x.stride(2), x.stride(1), _ptr(y), y.stride(0),
                                          y.stride(1), 1, B, T, Cc, pad_rep, _stream()))
    return y


def to_channels_first(x_btc):
    """(B, T, C) any strides -> contiguous (B, C, T)."""
    x = _dev(x_btc, name="x")
    B, T, Cc = x.shape
    y = torch.empty(B, Cc, T, dtype=_F32, device=x.device)
    L.check(L.lib().mtts_copy_strided_f32(_ptr(x), x.stride(0), x.stride(1), x.stride(2), _ptr(y), y.stride(0),
                                          1, y.stride(1), B, T, Cc, 0, _stream()))
    return y


def mel_spectrogram(wav, window, fb_w, fb_off, fb_start, n_mels=80, clamp=1e-5, frames_major=False, lens=None):
    """wav (B, L) -> (B, n_mels, F) or (B, F, n_mels) if frames_major; F = 1 + L // 256.
    ``lens`` (B,) int32 on the device: ragged batch, clip b is wav[b, :lens[b]]; frames past 1 + lens[b] // 256 are
    left at zero."""
    wav = _dev(wav, name="wav")
    if wav.stride(1) != 1:
        wav = wav.contiguous()
    B, Lw = wav.shape
    F = 1 + Lw // 256
    alloc = torch.zeros if lens is not None else torch.empty
    if frames_major:
        out = alloc(B, F, n_mels, dtype=_F32, device=wav.device)
        sb, sm, sf = out.stride(0), 1, out.stride(1)
    else:
        out = alloc(B, n_mels, F, dtype=_F32, device=wav.device)
        sb, sm, sf = out.stride(0), out.stride(1), 1
    tabs = (_ptr(_dev(window)), _ptr(_dev(fb_w)), _ptr(_dev(fb_off, torch.int32)), _ptr(_dev(fb_start, torch.int32)))
    if lens is None:
        L.check(L.lib().mtts_mel_spectrogram_f32(_ptr(wav), wav.stride(0), B, Lw, *tabs, n_mels, clamp, _ptr(out), sb, sm, sf,
                                                 _stream()))
    else:
        lens = _dev(lens, torch.int32, name="lens")
        assert lens.shape == (B,) and lens.is_contiguous()
        L.check(L.lib().mtts_mel_spectrogram_ragged_f32(_ptr(wav), wav.stride(0), B, Lw, _ptr(lens), *tabs, n_mels, clamp,
                                                        _ptr(out), sb, sm, sf, _stream()))
    return out


# ------------------------------------------------------------------------------ f16x2 range guard
_ovf_flags = {}


def _dev_index(device):
    return torch.cuda.current_device() if device.index is None else device.index


def tc_overflow_bind(device):
    """Registers (once per device) the int32 flag the f16x2 operand split raises when an activation leaves the
    fp16 range (|x| > 65504); returns the flag tensor."""
    idx = _dev_index(device)
    flag = _ovf_flags.get(idx)
    if flag is None:
        with torch.cuda.device(idx):
            flag = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", idx))
            L.check(L.lib().mtts_tc_overflow_bind(_ptr(flag)))
        _ovf_flags[idx] = flag
    return flag


def tc_overflow(device, reset=True):
    """True if any f16x2 split on `device` saw an out-of-range activation since the last reset (one host sync)."""
    flag = tc_overflow_bind(device)
    hit = bool(flag.item())
    if hit and reset:
        flag.zero_()
    return hit


# ------------------------------------------------------------------------------ workspace
_ws_cache = {}


def workspace(nbytes, device):
    """A scratch buffer per (device, stream) that only grows (torch caching allocator underneath); the base address
    is 256-byte aligned (the allocator's granularity is 512 bytes), which the C side's float4 / TMA carving relies on.
    Work on different streams never shares scratch."""
    tc_overflow_bind(device)
    key = (device.type, _dev_index(device), torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = None
        _ws_cache.pop(key, None)
        buf = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
        assert buf.data_ptr() % 256 == 0
        _ws_cache[key] = buf
    return buf


def _lib_launch_count():
    return int(L.lib().mtts_launch_count())


def launch_count():
    """Kernels launched by this process so far: the library's enqueue counter plus the kernel nodes executed by CUDA-graph
    replays (megatts2_b200/graphs.py).  A capture pass is counted by the library although it only records - once per graph,
    during warm-up."""
    from . import graphs
    return _lib_launch_count() + graphs.replayed_launches
