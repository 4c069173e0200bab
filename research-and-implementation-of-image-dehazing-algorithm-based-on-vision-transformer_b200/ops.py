"""PyTorch custom ops (autograd.Function) over the C ABI of include/lewin_b200.h.

PyTorch is plumbing here: it owns device memory, the current stream and autograd bookkeeping; every
FLOP of the LeWin block is executed by the sm_100a kernels behind the ABI.  No fallback path exists.

Ops
---
lewin_attn(x, ...)   attention half of LeWinTransformerBlock.forward (My_model_1.py:803-872) or, with
                     ``windowed=True``, WindowAttention.forward (My_model_1.py:400-415).
lewin_leff(y, ...)   LeFF half (My_model_1.py:873) or, with ``fused=False``, LeFF.forward (:496-534).
"""
from __future__ import annotations

import threading
import weakref
from collections import namedtuple

import torch

from . import _lib

_DT = {torch.float32: "f32", torch.bfloat16: "bf16"}


def _ptr(t):
    return None if t is None else t.data_ptr()


def _f32c(t):
    """Parameters cross the ABI as contiguous fp32 (the state_dict dtype)."""
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def ctypes_addr(arr):
    import ctypes
    return ctypes.cast(arr, ctypes.c_void_p).value


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dtype_tag(x):
    if not x.is_cuda:
        raise RuntimeError("lewin_b200 ops run on CUDA tensors only (sm_100a kernels, no CPU fallback)")
    try:
        return _DT[x.dtype]
    except KeyError:
        raise RuntimeError(f"lewin_b200: unsupported activation dtype {x.dtype} (float32 or bfloat16)") from None


def _deterministic():
    """The `deterministic` field of the backward calls: torch.use_deterministic_algorithms(True) (warn_only included, since
    the library has a deterministic implementation) asks for fixed-order parameter-gradient sums.  Read at backward time."""
    return int(torch.are_deterministic_algorithms_enabled())


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _zero_grads(like, device, separate=False):
    """fp32 zero gradient buffers for the given parameter tensors (None entries stay None): ONE flat allocation and one
    fill kernel, handed out as views (each backward call accumulates into them: with fp32 atomics, or with one add per element
    under torch.use_deterministic_algorithms).  separate=True gives every
    gradient its own storage (returns of a torch.library op may not alias each other)."""
    if separate:
        return [None if t is None else torch.zeros(t.shape, dtype=torch.float32, device=device) for t in like]
    sizes = [0 if t is None else t.numel() for t in like]
    flat = torch.zeros(sum((n + 3) // 4 * 4 for n in sizes), dtype=torch.float32, device=device)
    out, off = [], 0
    for t, n in zip(like, sizes):
        if t is None:
            out.append(None)
        else:
            out.append(flat[off:off + n].view(t.shape))
            off += (n + 3) // 4 * 4
    return out


def prepare_index_sample(index_sample, device):
    """int64 CPU tensor drawn as attn.py:91 -> int32 device tensor [64, 25]."""
    if index_sample.dtype != torch.int32 or index_sample.device != device:
        index_sample = index_sample.to(device=device, dtype=torch.int32, non_blocking=True)
    return index_sample.contiguous()


class KernelTimer:
    """Optional per-kernel CUDA-event timing through the ABI's `timing` field (used by bench.py).

    with KernelTimer() as kt: ...forward...;  torch.cuda.synchronize();  kt.summary() ->
    {(op, kernel): [ms, ...]} with the shape info of every launch in kt.launches."""

    active = None
    ATTN = ("ln_stats", "attn_fused", "gemm_qkv", "probsparse_core", "gemm_out")
    LEFF = ("ln_stats", "gemm_fc1_gelu", "dwconv_gelu", "gemm_fc2", "leff_tail")

    def __init__(self):
        self.launches = []     # (op, names, live_slots, info, events)

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def events_for(self, op, info, live_slots):
        import ctypes
        names = self.ATTN if op == "attn" else self.LEFF
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2 * len(names))]
        for e in evs:
            e.record()          # torch creates the cudaEvent lazily; force it so the handle is valid
        arr = (ctypes.c_void_p * len(evs))(*[e.cuda_event for e in evs])
        self.launches.append((op, names, tuple(live_slots), info, evs))
        return arr

    def summary(self):
        out = []
        for op, names, live, info, evs in self.launches:
            for k in live:
                out.append((op, names[k], info, evs[2 * k].elapsed_time(evs[2 * k + 1])))
        return out


class TopRecorder:
    """Collects the selected top-u query indices (M_top, attn.py:122) of every lewin_attn call made while active, in call
    order: ``with TopRecorder() as rec: model(x)`` -> ``rec.tops`` = [uint8 [B_, nH, 25], ...] (one per LeWin block).
    Test / diagnostic hook for the per-block, tie-aware selection check of a whole-model forward."""

    active = None

    def __init__(self):
        self.tops = []

    def __enter__(self):
        TopRecorder.active = self
        return self

    def __exit__(self, *exc):
        TopRecorder.active = None


class _WeightImages:
    """bf16 images of constant fp32 weights for the C >= 256 GEMMs (the ABI's optional w*_bf16 fields).

    One entry per live weight tensor (keyed by id, dropped by a weakref callback when the tensor dies), REPLACED when the
    tensor's version counter changes (optimizer step, load_state_dict) - stale versions never accumulate.  Guarded by a
    lock (nn.DataParallel replica threads).  A CUDA-graph capture must keep the images it baked into the graph alive:
    ``with images.pin() as held:`` collects every image handed out meanwhile (fullres.GraphedForward stores ``held``)."""

    def __init__(self):
        self._lock = threading.RLock()      # re-entrant: a weakref callback may fire while the owner thread holds it
        self._ent = {}            # id(w) -> (weakref, version, data_ptr, image)
        self._pins = []

    def get(self, w):
        key = id(w)
        with self._lock:
            ent = self._ent.get(key)
            if ent is not None and ent[0]() is w and ent[1] == w._version and ent[2] == w.data_ptr():
                img = ent[3]
            else:
                img = w.detach().to(torch.bfloat16).contiguous()
                ref = weakref.ref(w, lambda _r, k=key: self._drop(k))
                self._ent[key] = (ref, w._version, w.data_ptr(), img)
            for held in self._pins:
                held.append(img)
            return img

    def _drop(self, key):
        with self._lock:
            ent = self._ent.get(key)
            if ent is not None and ent[0]() is None:
                del self._ent[key]

    def __len__(self):
        return len(self._ent)

    class _Pin:
        def __init__(self, owner):
            self.owner, self.held = owner, []

        def __enter__(self):
            with self.owner._lock:
                self.owner._pins.append(self.held)
            return self.held

        def __exit__(self, *exc):
            with self.owner._lock:
                self.owner._pins.remove(self.held)

    def pin(self):
        return _WeightImages._Pin(self)


weight_images = _WeightImages()


def _bf16_image(w):
    return weight_images.get(w)


def _token_mask(token_mask, B, H, W, device):
    """The input mask per token as it crosses the ABI: contiguous fp32 [Bm, H, W] on the activations' device, Bm | B."""
    if token_mask is None:
        return None
    tm = token_mask.to(device=device, dtype=torch.float32).contiguous()
    if tm.dim() != 3 or tuple(tm.shape[1:]) != (H, W) or tm.shape[0] < 1 or B % tm.shape[0]:
        raise RuntimeError(f"lewin_b200.lewin_attn: token_mask must be [Bm, {H}, {W}] with Bm dividing B = {B}, "
                           f"got {tuple(token_mask.shape)}")
    return tm


# The tensors of an attention-half call as they cross the ABI, which its backward reads again: the fp32 parameters, the int32
# sample indices, q|k|v, ctx, the selection and the token mask.
AttnSaved = namedtuple("AttnSaved", "x ln_w ln_b w_qkv b_qkv w_out b_out rpb_table rpb_dense index_sample mask drop_scale qkv "
                                    "ctx top token_mask")


def _attn_args(geom, s, *, y, save):
    """LewinAttnFwdArgs of a forward (y given) or backward (y = None) call on the tensors ``s`` (an AttnSaved)."""
    B, H, W, nH, shift, windowed, use_rpb, analytic = geom[:8]
    return _lib.LewinAttnFwdArgs(
        B=B, H=H, W=W, C=s.x.shape[-1], nH=nH, shift=shift, windowed=int(windowed), use_rpb=int(use_rpb),
        analytic_shift_mask=int(analytic), nW_mask=0 if s.mask is None else s.mask.shape[0],
        save_for_backward=int(save), reserved=0,
        x=_ptr(s.x), y=_ptr(y), ln_w=_ptr(s.ln_w), ln_b=_ptr(s.ln_b), w_qkv=_ptr(s.w_qkv), b_qkv=_ptr(s.b_qkv),
        w_out=_ptr(s.w_out), b_out=_ptr(s.b_out), rpb_table=_ptr(s.rpb_table), rpb_dense=_ptr(s.rpb_dense),
        index_sample=_ptr(s.index_sample), mask=_ptr(s.mask), drop_scale=_ptr(s.drop_scale),
        qkv=_ptr(s.qkv), ctx=_ptr(s.ctx), top=_ptr(s.top), token_mask=_ptr(s.token_mask),
        Bm=0 if s.token_mask is None else s.token_mask.shape[0])


def _attn_forward(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask, drop_scale, geom,
                  token_mask=None):
    """One lewin_attn_fwd_* call.  Returns (y, top, saved): ``saved`` is the AttnSaved the backward call needs.  Shared by
    the autograd.Function below and the torch.library ops of compile_ops.py."""
    B, H, W, nH, shift, windowed, use_rpb, analytic, need_grad = geom[:9]
    band = geom[9] if len(geom) > 9 else None          # (y0, Hg): row band of a taller image (forward only)
    lib = _lib.load()
    dt = _dtype_tag(x)
    x = x.contiguous()
    C = x.shape[-1]
    tokens = B * H * W
    assert x.numel() == tokens * C, (x.shape, B, H, W, C)
    dev = x.device
    y = torch.empty_like(x)
    top = torch.empty((tokens // 64, nH, 25), dtype=torch.uint8, device=dev)
    ln_w_, ln_b_, w_qkv_, b_qkv_, w_out_, b_out_, tab_, dense_, mask_, ds_ = [
        _f32c(t) for t in (ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, mask, drop_scale)]
    s = AttnSaved(x, ln_w_, ln_b_, w_qkv_, b_qkv_, w_out_, b_out_, tab_, dense_, prepare_index_sample(index_sample, dev), mask_,
                  ds_, None, None, top, _token_mask(token_mask, B, H, W, dev))
    a = _attn_args(geom, s, y=y, save=need_grad)
    if band is not None:
        if need_grad:
            raise RuntimeError("lewin_b200.lewin_attn: row-band mode is forward only")
        a.band_mode, a.band_y0, a.band_Hg = 1, int(band[0]), int(band[1])
    kmask = lib.lewin_attn_fwd_kernel_mask(a, _lib.DTYPE_TAG[dt])
    if kmask == 2:          # LEWIN_ATTN_K_FUSED: q|k|v and ctx stay on chip, the ABI only wants valid placeholders
        qkv = cbuf = torch.empty((16,), dtype=x.dtype, device=dev)
    else:
        qkv = torch.empty((tokens, 3 * C), dtype=x.dtype, device=dev)
        cbuf = torch.empty((tokens, C), dtype=x.dtype, device=dev)
    a.qkv, a.ctx = _ptr(qkv), _ptr(cbuf)
    if dt == "bf16" and C >= 256 and not need_grad:      # constants of an inference call: convert once
        wq_b, wo_b = _bf16_image(w_qkv_), _bf16_image(w_out_)
        a.w_qkv_bf16, a.w_out_bf16 = _ptr(wq_b), _ptr(wo_b)
    if KernelTimer.active is not None:
        mask = kmask
        tim = KernelTimer.active.events_for("attn", dict(tokens=tokens, C=C, nH=nH, dtype=dt),
                                            tuple(k for k in range(5) if mask >> k & 1))
        a.timing = ctypes_addr(tim)
    ws = _workspace(lib.lewin_attn_fwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
    fn = getattr(lib, f"lewin_attn_fwd_{dt}")
    with torch.cuda.device(dev):
        _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_attn_fwd_{dt}")
    if TopRecorder.active is not None:
        TopRecorder.active.tops.append(top)
    return y, top, s._replace(qkv=qkv, ctx=cbuf)


def _attn_backward(saved, geom, dy, separate_grads=False):
    """One lewin_attn_bwd_* call on the AttnSaved of the forward -> (dx, d_ln_w, d_ln_b, d_w_qkv, d_b_qkv, d_w_out, d_b_out,
    d_rpb_table, d_rpb_dense); entries of absent parameters are None."""
    s = AttnSaved(*saved)
    lib = _lib.load()
    dt = _dtype_tag(s.x)
    dev = s.x.device
    dy = dy.contiguous()
    dx = torch.empty_like(s.x)
    d_ln_w, d_ln_b, d_w_qkv, d_b_qkv, d_w_out, d_b_out, d_tab, d_dense = _zero_grads(
        (s.ln_w, s.ln_b, s.w_qkv, s.b_qkv, s.w_out, s.b_out, s.rpb_table, s.rpb_dense if s.rpb_table is None else None), dev,
        separate_grads)
    a = _lib.LewinAttnBwdArgs(
        fwd=_attn_args(geom, s, y=None, save=True), dy=_ptr(dy), dx=_ptr(dx), d_ln_w=_ptr(d_ln_w), d_ln_b=_ptr(d_ln_b),
        d_w_qkv=_ptr(d_w_qkv), d_b_qkv=_ptr(d_b_qkv), d_w_out=_ptr(d_w_out), d_b_out=_ptr(d_b_out),
        d_rpb_table=_ptr(d_tab), d_rpb_dense=_ptr(d_dense), deterministic=_deterministic())
    ws = _workspace(lib.lewin_attn_bwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
    fn = getattr(lib, f"lewin_attn_bwd_{dt}")
    with torch.cuda.device(dev):
        _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_attn_bwd_{dt}")
    # table path: d(relative_position_bias_table); dense path (AttentionLayer.forward's gathered bias, attn.py:385):
    # d(relative_position_bias) [nH, 64, 64], which autograd scatters back into the caller's table through its own gather
    return (dx, d_ln_w, d_ln_b, d_w_qkv, d_b_qkv, d_w_out, d_b_out, d_tab, d_dense)


class _AttnFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask,
                drop_scale, geom, token_mask=None):
        y, top, saved = _attn_forward(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask,
                                      drop_scale, geom, token_mask)
        ctx.geom = geom
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(top)
        return y, top

    @staticmethod
    def backward(ctx, dy, _dtop):
        return _attn_backward(ctx.saved_tensors, ctx.geom, dy) + (None, None, None, None, None)


# The tensors of a LeFF-half call as they cross the ABI, which its backward reads again: the fp32 parameters, the hidden
# activations h1 / h2 and the pre-activations a1 / a2.
LeffSaved = namedtuple("LeffSaved", "y ln_w ln_b w1 b1 w_dw b_dw w2 b2 drop_scale h1 h2 a1 a2")


def _leff_args(geom, s, *, out, save):
    """LewinLeffFwdArgs of a forward (out given) or backward (out = None) call on the tensors ``s`` (a LeffSaved)."""
    B, H, W, fused = geom[:4]
    return _lib.LewinLeffFwdArgs(
        B=B, H=H, W=W, C=s.y.shape[-1], hidden=s.w1.shape[0], fused=int(fused), save_for_backward=int(save), ld_out=0,
        y=_ptr(s.y), out=_ptr(out), ln_w=_ptr(s.ln_w), ln_b=_ptr(s.ln_b), w1=_ptr(s.w1), b1=_ptr(s.b1),
        w_dw=_ptr(s.w_dw), b_dw=_ptr(s.b_dw), w2=_ptr(s.w2), b2=_ptr(s.b2), drop_scale=_ptr(s.drop_scale),
        h1=_ptr(s.h1), h2=_ptr(s.h2), a1=_ptr(s.a1), a2=_ptr(s.a2))


def _leff_forward(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, geom, out_view=None):
    """One lewin_leff_fwd_* call.  Returns (out, saved): ``saved`` (None for an inference call) is the LeffSaved the backward
    call needs.  Shared by the autograd.Function below and the torch.library ops of compile_ops.py."""
    B, H, W, fused, need_grad = geom
    lib = _lib.load()
    dt = _dtype_tag(y)
    y = y.contiguous()
    C = y.shape[-1]
    hidden = w1.shape[0]
    tokens = B * H * W
    assert y.numel() == tokens * C, (y.shape, B, H, W, C)
    dev = y.device
    out = torch.empty_like(y)
    h1 = torch.empty((tokens, hidden), dtype=y.dtype, device=dev)
    h2 = h1                       # placeholder until the library says whether h2 exists in global memory for this call
    a1 = torch.empty_like(h1) if need_grad else None
    a2 = torch.empty_like(h1) if need_grad else None
    s = LeffSaved(y, *[_f32c(t) for t in (ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale)], h1, h2, a1, a2)
    a = _leff_args(geom, s, out=out, save=need_grad)
    if dt == "bf16" and C >= 256 and not need_grad:
        w1_b, w2_b = _bf16_image(s.w1), _bf16_image(s.w2)
        a.w1_bf16, a.w2_bf16 = _ptr(w1_b), _ptr(w2_b)
    if out_view is not None and not need_grad and lib.lewin_leff_fwd_supports_ld_out(a, _lib.DTYPE_TAG[dt]):
        # the caller's column block of a wider buffer (the right half of the decoder's concat buffer): written in place
        out = out_view
        a.out, a.ld_out = _ptr(out), out.stride(-2)
    mask = lib.lewin_leff_fwd_kernel_mask(a, _lib.DTYPE_TAG[dt])
    if not (mask >> 4 & 1):       # LEWIN_LEFF_K_TAIL clear: the three-kernel pipeline writes h2 = GELU(dwconv(h1))
        h2 = torch.empty((tokens, hidden), dtype=y.dtype, device=dev)
        a.h2 = _ptr(h2)
    if KernelTimer.active is not None:
        tim = KernelTimer.active.events_for("leff", dict(tokens=tokens, C=C, hidden=hidden, dtype=dt),
                                            tuple(k for k in range(5) if mask >> k & 1))
        a.timing = ctypes_addr(tim)
    ws = _workspace(lib.lewin_leff_fwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
    fn = getattr(lib, f"lewin_leff_fwd_{dt}")
    with torch.cuda.device(dev):
        _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_leff_fwd_{dt}")
    return out, (s._replace(h2=h2) if need_grad else None)


def _leff_backward(saved, geom, dout, separate_grads=False):
    """One lewin_leff_bwd_* call on the LeffSaved of the forward -> (dy, d_ln_w, d_ln_b, d_w1, d_b1, d_w_dw, d_b_dw, d_w2,
    d_b2); entries of absent parameters are None."""
    s = LeffSaved(*saved)
    lib = _lib.load()
    dt = _dtype_tag(s.y)
    dev = s.y.device
    dout = dout.contiguous()
    dy = torch.empty_like(s.y)
    d_ln_w, d_ln_b, d_w1, d_b1, d_wdw, d_bdw, d_w2, d_b2 = _zero_grads(
        (s.ln_w, s.ln_b, s.w1, s.b1, s.w_dw, s.b_dw, s.w2, s.b2), dev, separate_grads)
    a = _lib.LewinLeffBwdArgs(
        fwd=_leff_args(geom, s, out=None, save=True), dout=_ptr(dout), dy=_ptr(dy), d_ln_w=_ptr(d_ln_w), d_ln_b=_ptr(d_ln_b),
        d_w1=_ptr(d_w1), d_b1=_ptr(d_b1), d_w_dw=_ptr(d_wdw), d_b_dw=_ptr(d_bdw), d_w2=_ptr(d_w2), d_b2=_ptr(d_b2),
        deterministic=_deterministic())
    ws = _workspace(lib.lewin_leff_bwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
    fn = getattr(lib, f"lewin_leff_bwd_{dt}")
    with torch.cuda.device(dev):
        _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_leff_bwd_{dt}")
    return (dy, d_ln_w, d_ln_b, d_w1, d_b1, d_wdw, d_bdw, d_w2, d_b2)


class _LeffFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, geom, out_view=None):
        out, saved = _leff_forward(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, geom, out_view)
        ctx.geom = geom
        if saved is not None:
            ctx.save_for_backward(*saved)
        return out

    @staticmethod
    def backward(ctx, dout):
        return _leff_backward(ctx.saved_tensors, ctx.geom, dout) + (None, None, None)


def lewin_attn(x, *, B, H, W, num_heads, shift, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out,
               rpb_table=None, rpb_dense=None, index_sample, mask=None, drop_scale=None,
               windowed=False, use_rpb=True, analytic_shift_mask=True, return_top=False, band=None, token_mask=None):
    """Attention half of a LeWin block.  Returns y (same shape as x) [and the selected top-u indices].
    token_mask: the input mask as one value per token, [Bm, H, W] with Bm | B (image b uses mask b mod Bm): the nearest-resized
    mask of My_model_1.py:791-798, evaluated inside the kernels in place of the dense [B*nW, 64, 64] mask the reference builds
    (fused block half only; combined with the analytic shift mask).
    band=(y0, Hg): x is a band of H rows, already in shifted-frame row order, of an image Hg rows tall whose shifted-frame
    row y0 is the band's first row (canvas-mode row sharding, fullres / canvas_bands; forward only)."""
    need = torch.is_grad_enabled() and any(
        isinstance(t, torch.Tensor) and t.requires_grad for t in (x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense))
    geom = (int(B), int(H), int(W), int(num_heads), int(shift), bool(windowed), bool(use_rpb), bool(analytic_shift_mask), need)
    if band is not None:
        geom = geom + ((int(band[0]), int(band[1])),)
    elif torch.compiler.is_compiling():        # traced by torch.compile / export: one opaque torch.library node (compile_ops.py)
        y, top = compile_ops.lewin_attn(x, B=B, H=H, W=W, num_heads=num_heads, shift=shift, ln_w=ln_w, ln_b=ln_b, w_qkv=w_qkv,
                                        b_qkv=b_qkv, w_out=w_out, b_out=b_out, rpb_table=rpb_table, rpb_dense=rpb_dense,
                                        index_sample=index_sample, mask=mask, drop_scale=drop_scale, windowed=windowed,
                                        use_rpb=use_rpb, analytic_shift_mask=analytic_shift_mask, need=need,
                                        token_mask=token_mask)
        return (y, top) if return_top else y
    y, top = _AttnFn.apply(x, ln_w, ln_b, w_qkv, b_qkv, w_out, b_out, rpb_table, rpb_dense, index_sample, mask,
                           drop_scale, geom, token_mask)
    return (y, top) if return_top else y


def lewin_leff(y, *, B, H, W, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale=None, fused=True, out=None):
    """LeFF half of a LeWin block (fused=True: out = y + s * LeFF(LN2(y)); fused=False: out = LeFF(y)).
    out: optional destination view shaped like y whose token stride may exceed C (a column block of a wider buffer);
    used - and returned - when the call is inference and the library can address it (otherwise a new tensor is returned)."""
    need = torch.is_grad_enabled() and any(
        isinstance(t, torch.Tensor) and t.requires_grad for t in (y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2))
    geom = (int(B), int(H), int(W), bool(fused), need)
    if torch.compiler.is_compiling():          # traced: one opaque torch.library node; the in-place `out` view is not offered there
        return compile_ops.lewin_leff(y, B=B, H=H, W=W, ln_w=ln_w, ln_b=ln_b, w1=w1, b1=b1, w_dw=w_dw, b_dw=b_dw, w2=w2, b2=b2,
                                      drop_scale=drop_scale, fused=fused, need=need)
    if out is not None:
        ok = (out.shape == y.shape and out.dtype == y.dtype and out.device == y.device and out.stride(-1) == 1 and
              out.stride(-2) % 8 == 0 and out.data_ptr() % 16 == 0 and
              (out.dim() < 3 or out.shape[0] == 1 or out.stride(0) == out.shape[1] * out.stride(1)))
        if not ok:
            out = None
    return _LeffFn.apply(y, ln_w, ln_b, w1, b1, w_dw, b_dw, w2, b2, drop_scale, geom, out)


def _core_args(geom, qkv, ctx, rpb_table, rpb_dense, index_sample, mask, top):
    """LewinCoreFwdArgs of a core-only forward or backward call (qkv [B_, 64, 3C], head_dim = C / nH)."""
    nH, use_rpb = geom
    return _lib.LewinCoreFwdArgs(B_=qkv.shape[0], nH=nH, use_rpb=int(use_rpb), nW_mask=0 if mask is None else mask.shape[0],
                                 head_dim=qkv.shape[-1] // 3 // nH, reserved=0,
                                 qkv=_ptr(qkv), ctx=_ptr(ctx), rpb_table=_ptr(rpb_table), rpb_dense=_ptr(rpb_dense),
                                 index_sample=_ptr(index_sample), mask=_ptr(mask), top=_ptr(top))


class _CoreFn(torch.autograd.Function):
    """ProbAttention.forward (attn.py:287-342) on projected q|k|v; backward = lewin_probsparse_core_bwd_* for the saved selection."""

    @staticmethod
    def forward(ctx, qkv, rpb_table, rpb_dense, mask, index_sample, geom):
        nH, use_rpb = geom
        lib = _lib.load()
        dt = _dtype_tag(qkv)
        qkv = qkv.contiguous()
        B_, L, C3 = qkv.shape
        C = C3 // 3
        if L != 64 or C % nH:
            raise RuntimeError(f"lewin_b200.probsparse_core: qkv must be [B_, 64, 3 * nH * head_dim], got {tuple(qkv.shape)} with nH={nH}")
        dev = qkv.device
        out = torch.empty((B_, L, C), dtype=qkv.dtype, device=dev)
        top = torch.empty((B_, nH, 25), dtype=torch.uint8, device=dev)
        tab_, dense_, mask_ = _f32c(rpb_table), _f32c(rpb_dense), _f32c(mask)
        idx = prepare_index_sample(index_sample, dev)          # alive until the call: the struct holds only its address
        a = _core_args(geom, qkv, out, tab_, dense_, idx, mask_, top)
        ws = _workspace(lib.lewin_probsparse_core_fwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
        fn = getattr(lib, f"lewin_probsparse_core_fwd_{dt}")
        with torch.cuda.device(dev):
            _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_probsparse_core_fwd_{dt}")
        ctx.geom, ctx.dt = geom, dt
        ctx.save_for_backward(qkv, tab_, dense_, mask_, top)
        ctx.mark_non_differentiable(top)
        return out, top

    @staticmethod
    def backward(ctx, dctx, _dtop):
        qkv, tab, dense, mask, top = ctx.saved_tensors
        lib = _lib.load()
        dt = ctx.dt
        dev = qkv.device
        dctx = dctx.contiguous()
        dqkv = torch.empty_like(qkv)
        d_tab, d_dense = _zero_grads((tab, dense if tab is None else None), dev)
        a = _lib.LewinCoreBwdArgs(fwd=_core_args(ctx.geom, qkv, dctx, tab, dense, None, mask, top), dctx=_ptr(dctx),
                                  dqkv=_ptr(dqkv), d_rpb_table=_ptr(d_tab), d_rpb_dense=_ptr(d_dense),
                                  deterministic=_deterministic())
        ws = _workspace(lib.lewin_probsparse_core_bwd_workspace_bytes(a, _lib.DTYPE_TAG[dt]), dev)
        fn = getattr(lib, f"lewin_probsparse_core_bwd_{dt}")
        with torch.cuda.device(dev):
            _lib.check(fn(a, ws.data_ptr(), ws.numel(), _stream()), f"lewin_probsparse_core_bwd_{dt}")
        return dqkv, d_tab, d_dense, None, None, None


def probsparse_core(qkv, *, num_heads, index_sample, rpb_table=None, rpb_dense=None, mask=None, use_rpb=True,
                    return_top=False):
    """ProbAttention.forward (attn.py:287-342) on projected q|k|v [B_, 64, 3C] -> context [B_, 64, C]; head_dim =
    C / num_heads in {32, 64, 128}.  Differentiable in qkv and the bias (table [225, nH] or gathered [nH, 64, 64])."""
    out, top = _CoreFn.apply(qkv, rpb_table, rpb_dense, mask, index_sample, (int(num_heads), bool(use_rpb)))
    return (out, top) if return_top else out


def upsample_supported(x, Cin, Cout, tokens):
    """The 2x2 / stride-2 transposed convolution runs as a token GEMM on the streamed-W tcgen05 kernel (bf16, no autograd)."""
    return x.is_cuda and x.dtype == torch.bfloat16 and Cin % 64 == 0 and Cout % 32 == 0 and tokens >= 1


def lewin_upsample(x, weight, bias, *, B, H, W, out=None):
    """Upsample.forward (My_model_1.py:633-648): x [B, H*W, Cin] bf16 -> [B, 4*H*W, Cout].  ``out`` may be a wider
    [B, 4*H*W, ld] buffer (ld >= Cout): columns [0, Cout) are written (the left half of torch.cat([up, skip], -1))."""
    lib = _lib.load()
    x = x.contiguous()
    Cin = x.shape[-1]
    Cout = weight.shape[1]
    dev = x.device
    if out is None:
        out = torch.empty((B, 4 * H * W, Cout), dtype=x.dtype, device=dev)
    assert out.is_contiguous() and out.shape[0] == B and out.shape[1] == 4 * H * W and out.shape[2] >= Cout
    w_, b_ = _f32c(weight), _f32c(bias)
    a = _lib.LewinUpsampleFwdArgs(B=B, H=H, W=W, Cin=Cin, Cout=Cout, ld_out=out.shape[2], reserved0=0, reserved1=0,
                                  x=_ptr(x), weight=_ptr(w_), bias=_ptr(b_), out=_ptr(out))
    ws = _workspace(lib.lewin_upsample_fwd_workspace_bytes(a, _lib.DTYPE_TAG["bf16"]), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lewin_upsample_fwd_bf16(a, ws.data_ptr(), ws.numel(), _stream()), "lewin_upsample_fwd_bf16")
    return out


def downsample_supported(x, Cin, W):
    """Downsample's 4x4 / stride-2 convolution runs as an implicit GEMM on tcgen05 (bf16, no autograd)."""
    return (x.is_cuda and x.dtype == torch.bfloat16 and (Cin == 32 or (Cin % 64 == 0 and Cin <= 512)) and
            W % 16 == 0)


def lewin_downsample(x, weight, bias, *, B, H, W, pad_h=True, out=None):
    """Downsample.forward (My_model_1.py:606-630): x [B, H*W, Cin] bf16 tokens (may be a column slice [..., :Cin] of a wider
    contiguous buffer) -> [B, Hout * W/2, 2*Cin] bf16, Hout = H/2 (pad_h) or H/2 - 1 (rows carry their own halo)."""
    lib = _lib.load()
    Cin = weight.shape[1]
    assert x.shape[-1] == Cin and x.stride(-1) == 1 and x.stride(-2) % 8 == 0
    ld_x = x.stride(-2)
    assert x.numel() == B * H * W * Cin and (x.dim() < 3 or x.shape[0] == 1 or x.stride(0) == H * W * ld_x)
    dev = x.device
    Hout = H // 2 if pad_h else H // 2 - 1
    if out is None:
        out = torch.empty((B, Hout * (W // 2), 2 * Cin), dtype=x.dtype, device=dev)
    w_, b_ = _f32c(weight), _f32c(bias)
    a = _lib.LewinDownsampleArgs(B=B, H=H, W=W, Cin=Cin, ld_x=ld_x, ld_out=out.stride(-2), pad_h=int(bool(pad_h)), reserved=0,
                                 x=_ptr(x), weight=_ptr(w_), bias=_ptr(b_), out=_ptr(out))
    ws = _workspace(lib.lewin_downsample_fwd_workspace_bytes(a, _lib.DTYPE_TAG["bf16"]), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lewin_downsample_fwd_bf16(a, ws.data_ptr(), ws.numel(), _stream()), "lewin_downsample_fwd_bf16")
    return out


def conv3x3_supported(x, Cin, Cout):
    """x: NCHW tensor in channels_last memory format, bf16, on the GPU; Cin, Cout multiples of 64 up to 512; W % 8 == 0."""
    return (x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and Cin % 64 == 0 and Cin <= 512 and
            Cout % 64 == 0 and Cout <= 512 and x.shape[3] % 8 == 0 and x.is_contiguous(memory_format=torch.channels_last))


def conv3x3_weight_images(weight):
    """bf16 operand images of a frozen Conv2d(Cin, Cout, 3, padding=1) weight [Cout, Cin, 3, 3]:
    forward [9, Cout, Cin] (tap = ky * 3 + kx) and data-gradient [9, Cin, Cout] (kernel flipped, channel axes swapped)."""
    w = weight.detach().float()
    Cout, Cin = w.shape[0], w.shape[1]
    fwd = w.permute(2, 3, 0, 1).reshape(9, Cout, Cin).to(torch.bfloat16).contiguous()
    bwd = w.flip(2, 3).permute(2, 3, 1, 0).reshape(9, Cin, Cout).to(torch.bfloat16).contiguous()
    return fwd, bwd


def lewin_conv3x3(x, w_img, bias, relu):
    """Conv2d(kernel 3, padding 1) + bias (+ ReLU) on a channels_last bf16 NCHW tensor through lewin_conv3x3_fwd_bf16 (implicit
    GEMM on tcgen05).  w_img: [9, Cout, Cin] bf16 (conv3x3_weight_images).  Returns a channels_last bf16 NCHW tensor."""
    lib = _lib.load()
    B, Cin, H, W = x.shape
    Cout = w_img.shape[1]
    assert w_img.shape == (9, Cout, Cin) and w_img.dtype == torch.bfloat16 and w_img.is_contiguous()
    assert x.dtype == torch.bfloat16 and x.is_contiguous(memory_format=torch.channels_last)
    out = torch.empty((B, Cout, H, W), dtype=torch.bfloat16, device=x.device, memory_format=torch.channels_last)
    b_ = _f32c(bias) if bias is not None else None
    a = _lib.LewinConv3x3Args(B=B, H=H, W=W, Cin=Cin, Cout=Cout, ld_x=Cin, ld_out=Cout, relu=int(bool(relu)),
                              x=_ptr(x), weight=None, w_bf16=_ptr(w_img), bias=_ptr(b_) if b_ is not None else None, out=_ptr(out))
    with torch.cuda.device(x.device):
        _lib.check(lib.lewin_conv3x3_fwd_bf16(a, None, 0, _stream()), "lewin_conv3x3_fwd_bf16")
    return out


class _ConvReluFn(torch.autograd.Function):
    """relu(conv3x3(x) + b) with frozen weights: forward and data gradient on the implicit-GEMM kernel (no weight gradient)."""

    @staticmethod
    def forward(ctx, x, w_fwd, w_bwd, bias):
        y = lewin_conv3x3(x, w_fwd, bias, True)
        if x.requires_grad:
            ctx.save_for_backward(y, w_bwd)
        return y

    @staticmethod
    def backward(ctx, dy):
        y, w_bwd = ctx.saved_tensors
        g = (dy.to(torch.bfloat16) * (y > 0)).contiguous(memory_format=torch.channels_last)
        return lewin_conv3x3(g, w_bwd, None, False), None, None, None


def conv3x3_relu(x, w_fwd, w_bwd, bias):
    return _ConvReluFn.apply(x, w_fwd, w_bwd, bias)


def output_proj_supported(x, Cin, Cout, W):
    return x.is_cuda and x.dtype == torch.bfloat16 and Cin % 64 == 0 and Cin <= 256 and 1 <= Cout <= 8


def lewin_output_proj(x, weight, bias, *, B, H, W, residual=None, pad_h=True):
    """OutputProj.forward (My_model_1.py:696-733): x [B, H*W, Cin] bf16 tokens -> fp32 image [B, Cout, Hout, W] (+ residual, the
    `x + y` of Uformer.forward), Hout = H (pad_h) or H - 2."""
    lib = _lib.load()
    Cout, Cin = weight.shape[0], weight.shape[1]
    x = x.contiguous()
    assert x.numel() == B * H * W * Cin
    dev = x.device
    Hout = H if pad_h else H - 2
    out = torch.empty((B, Cout, Hout, W), dtype=torch.float32, device=dev)
    if residual is not None:
        residual = residual.contiguous()
        assert residual.dtype == torch.float32 and tuple(residual.shape) == tuple(out.shape)
    w_, b_ = _f32c(weight), _f32c(bias)
    a = _lib.LewinOutputProjArgs(B=B, H=H, W=W, Cin=Cin, Cout=Cout, ld_x=Cin, pad_h=int(bool(pad_h)), reserved=0,
                                 x=_ptr(x), weight=_ptr(w_), bias=_ptr(b_), residual=_ptr(residual), out=_ptr(out))
    ws = _workspace(lib.lewin_output_proj_fwd_workspace_bytes(a, _lib.DTYPE_TAG["bf16"]), dev)
    with torch.cuda.device(dev):
        _lib.check(lib.lewin_output_proj_fwd_bf16(a, ws.data_ptr(), ws.numel(), _stream()), "lewin_output_proj_fwd_bf16")
    return out


def lewin_input_proj(x, weight, bias, negative_slope=0.01):
    """InputProj.forward (My_model_1.py:659-682) under bf16 autocast: x [B, Cin, H, W] fp32 CUDA -> tokens [B, H*W, Cout] bf16,
    convolution + bias + LeakyReLU in one kernel."""
    lib = _lib.load()
    if not (x.is_cuda and x.dtype == torch.float32):
        raise RuntimeError("lewin_input_proj takes an fp32 CUDA image")
    x = x.contiguous()
    B, Cin, H, W = x.shape
    Cout = weight.shape[0]
    out = torch.empty((B, H * W, Cout), dtype=torch.bfloat16, device=x.device)
    w_, b_ = _f32c(weight), _f32c(bias)
    a = _lib.LewinInputProjArgs(B=B, H=H, W=W, Cin=Cin, Cout=Cout, negative_slope=float(negative_slope), reserved0=0, reserved1=0,
                                x=_ptr(x), weight=_ptr(w_), bias=_ptr(b_), out=_ptr(out))
    with torch.cuda.device(x.device):
        _lib.check(lib.lewin_input_proj_fwd_bf16(a, _stream()), "lewin_input_proj_fwd_bf16")
    return out


from . import compile_ops  # noqa: E402  (registers torch.ops.lewin_b200.*; imports this module back, so it comes last)
