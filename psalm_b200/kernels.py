"""Torch-tensor wrappers over the C ABI (include/psalm_b200.h).  PyTorch is used only for device
memory, streams and library GEMMs; every function here launches hand-written sm_100a kernels and
raises (never falls back) when the library is missing or an argument is wrong."""
import torch

from . import _lib
from .msda import ms_deform_attn_forward, msda_encoder_fused  # noqa: F401  (re-exported)

_LAUNCHES = [0]  # kernels launched through this module (bench.py's gpu_launches counter)
PROFILE_EVENTS = None  # bench.py sets this to a dict: name -> [(start, end) CUDA events] around hot-kernel launches


def timed(name, fn, *args, **kw):
    """Run a hot-kernel launch; when bench.py profiles, bracket it with CUDA events on the current stream."""
    if PROFILE_EVENTS is None:
        return fn(*args, **kw)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn(*args, **kw)
    b.record()
    PROFILE_EVENTS.setdefault(name, []).append((a, b))
    return out


def timed_msda(fn, *args):
    return timed("msda", fn, *args)


def launches():
    return _LAUNCHES[0]


def _count(n=1):
    _LAUNCHES[0] += n


def _on_device(fn):
    """Launch on the device that owns the first tensor argument (the C ABI launches on the CURRENT device; a model
    on cuda:1 while cuda:0 is current would otherwise fail or, worse, launch with foreign pointers)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kw):
        t = next((a for a in args if isinstance(a, torch.Tensor)), None)
        if t is not None and t.is_cuda and t.device.index != torch.cuda.current_device():
            with torch.cuda.device(t.device):
                return fn(*args, **kw)
        return fn(*args, **kw)
    return wrapper


def _chk(t, name):
    if not t.is_cuda:
        raise _lib.PsalmKernelError("%s: expected a CUDA tensor, got %s (no CPU path)" % (name, t.device))
    if not t.is_contiguous():
        raise _lib.PsalmKernelError("%s: tensor must be contiguous" % name)


@_on_device
def window_attention(qkv, qkv_bias, rel_bias, B, H, W, C, nh, ws, shift):
    """qkv [B,H*W,3C] -> attention output [B,H*W,C] (before proj).  swin_trans.py:117-149,194-253."""
    for t, n in ((qkv, "qkv"), (qkv_bias, "qkv_bias"), (rel_bias, "rel_bias")):
        _chk(t, "window_attention." + n)
    if rel_bias.dtype != torch.float32 or tuple(rel_bias.shape) != (nh, (2 * ws - 1) ** 2):
        raise _lib.PsalmKernelError("window_attention: rel_bias must be the compact fp32 table [nh, (2*ws-1)^2]")
    if qkv_bias.dtype != qkv.dtype or tuple(qkv.shape) != (B, H * W, 3 * C):
        raise _lib.PsalmKernelError("window_attention: bad qkv / bias")
    out = torch.empty((B, H * W, C), dtype=qkv.dtype, device=qkv.device)
    rc = _lib.lib().psalm_window_attention(_lib.ptr(qkv), _lib.ptr(qkv_bias), _lib.ptr(rel_bias), _lib.ptr(out),
                                           B, H, W, C, nh, ws, shift, _lib.dtype_code(qkv.dtype),
                                           _lib.stream_ptr(qkv.device))
    _lib.check(rc, "psalm_window_attention")
    _count()
    return out


@_on_device
def rotary_inplace(qkv, cos, sin, B, T, nh, hd, rd):
    _chk(qkv, "rotary.qkv")
    _chk(cos, "rotary.cos")
    _chk(sin, "rotary.sin")
    rc = _lib.lib().psalm_rotary_inplace(_lib.ptr(qkv), _lib.ptr(cos), _lib.ptr(sin), B, T, nh, hd, rd,
                                         _lib.dtype_code(qkv.dtype), _lib.stream_ptr(qkv.device))
    _lib.check(rc, "psalm_rotary_inplace")
    _count()


@_on_device
def causal_attention(qkv, key_valid, B, T, nh, hd):
    """qkv [B,T,3,nh,hd] (rotary applied) -> [B,T,nh*hd]; key_valid uint8 [B,T] or None."""
    _chk(qkv, "causal_attention.qkv")
    if key_valid is not None:
        _chk(key_valid, "causal_attention.key_valid")
        if key_valid.dtype != torch.uint8:
            raise _lib.PsalmKernelError("causal_attention: key_valid must be uint8")
    out = torch.empty((B, T, nh * hd), dtype=qkv.dtype, device=qkv.device)
    rc = _lib.lib().psalm_causal_attention(_lib.ptr(qkv), _lib.ptr(key_valid) if key_valid is not None else None,
                                           _lib.ptr(out), B, T, nh, hd, _lib.dtype_code(qkv.dtype),
                                           _lib.stream_ptr(qkv.device))
    _lib.check(rc, "psalm_causal_attention")
    _count()
    return out


def pick_splits(B, nh, Lq, Lk):
    """Split-K factor so that a 100-query problem still fills ~2 waves of 148 SMs."""
    ctas = B * nh * ((Lq + 63) // 64)
    want = max(1, (2 * 148 + ctas - 1) // ctas)
    # every CTA walks at least 4 key tiles of 64 (two per key group) so that the partial-result traffic stays small
    # <= 16: the split-K partials are reduced inside one thread-block cluster (distributed shared memory)
    return int(max(1, min(want, (Lk + 255) // 256, 16)))


@_on_device
def cross_attention(q, k, v, mask_bits=None, row_open=None, nh=8, splits=None, workspace=None):
    """q [B,Lq,C], k/v [B,Lk,C] (already projected) -> [B,Lq,C]."""
    for t, n in ((q, "q"), (k, "k"), (v, "v")):
        _chk(t, "cross_attention." + n)
    B, Lq, C = q.shape
    Lk = k.shape[1]
    hd = C // nh
    if splits is None:
        splits = pick_splits(B, nh, Lq, Lk)
    if splits > 1:
        need = _lib.lib().psalm_cross_attention_workspace_bytes(B, nh, hd, Lq, splits)
        if workspace is None or workspace.numel() * workspace.element_size() < need:
            workspace = torch.empty(need // 4, dtype=torch.float32, device=q.device)
    out = torch.empty_like(q)
    rc = _lib.lib().psalm_cross_attention(
        _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(mask_bits) if mask_bits is not None else None,
        _lib.ptr(row_open) if row_open is not None else None, _lib.ptr(out),
        _lib.ptr(workspace) if splits > 1 else None, B, Lq, Lk, nh, hd, splits, _lib.dtype_code(q.dtype),
        _lib.stream_ptr(q.device))
    _lib.check(rc, "psalm_cross_attention")
    _count(2 if splits > 1 else 1)
    return out


@_on_device
def mask_logits(mask_embed, feats, out_dtype=None):
    """mask_embed [B,Q,C], feats [B,P,C] (token-major) -> [B,Q,P]."""
    _chk(mask_embed, "mask_logits.mask_embed")
    _chk(feats, "mask_logits.feats")
    B, Q, C = mask_embed.shape
    P = feats.shape[1]
    out_dtype = out_dtype or mask_embed.dtype
    out = torch.empty((B, Q, P), dtype=out_dtype, device=feats.device)
    rc = _lib.lib().psalm_mask_logits(_lib.ptr(mask_embed), _lib.ptr(feats), _lib.ptr(out), B, Q, P, C,
                                      _lib.dtype_code(feats.dtype), _lib.dtype_code(out_dtype),
                                      _lib.stream_ptr(feats.device))
    _lib.check(rc, "psalm_mask_logits")
    _count()
    return out


@_on_device
def bilinear_tokens(x, Hi, Wi, Ho, Wo, out=None, out_dtype=None, accumulate=False):
    """x [B,Hi*Wi,C] token-major -> [B,Ho*Wo,C]; F.interpolate(bilinear, align_corners=False) semantics."""
    _chk(x, "bilinear_tokens.x")
    B, _, C = x.shape
    out_dtype = out_dtype or x.dtype
    if out is None:
        if accumulate:
            raise _lib.PsalmKernelError("bilinear_tokens: accumulate needs an output tensor")
        out = torch.empty((B, Ho * Wo, C), dtype=out_dtype, device=x.device)
    _chk(out, "bilinear_tokens.out")
    rc = _lib.lib().psalm_bilinear_tokens(_lib.ptr(x), _lib.ptr(out), B, Hi, Wi, Ho, Wo, C, _lib.dtype_code(x.dtype),
                                          _lib.dtype_code(out.dtype), 1 if accumulate else 0,
                                          _lib.stream_ptr(x.device))
    _lib.check(rc, "psalm_bilinear_tokens")
    _count()
    return out


@_on_device
def attn_mask_bits(logits):
    """logits [B,Q,P] -> (bits uint32 [B,Q,ceil(P/32)] (as int32 tensor), row_open uint8 [B,Q])."""
    _chk(logits, "attn_mask_bits.logits")
    B, Q, P = logits.shape
    bits = torch.empty((B, Q, (P + 31) // 32), dtype=torch.int32, device=logits.device)
    row_open = torch.empty((B, Q), dtype=torch.uint8, device=logits.device)
    rc = _lib.lib().psalm_attn_mask_bits(_lib.ptr(logits), _lib.ptr(bits), _lib.ptr(row_open), B * Q, P,
                                         _lib.dtype_code(logits.dtype), _lib.stream_ptr(logits.device))
    _lib.check(rc, "psalm_attn_mask_bits")
    _count()
    return bits, row_open


_LN_WIDTHS = (128, 256, 512, 1024, 2048)


@_on_device
def add_layer_norm(x, weight, bias, eps=1e-5, r1=None, r2=None, return_sum=False):
    """y = LayerNorm(x + r1 + r2) (residuals optional); with return_sum also returns the summed stream."""
    C = x.shape[-1]
    if C not in _LN_WIDTHS:
        raise _lib.PsalmKernelError("add_layer_norm: width %d unsupported" % C)
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias")):
        _chk(t, "add_layer_norm." + n)
    for t in (r1, r2):
        if t is not None:
            _chk(t, "add_layer_norm.residual")
            if t.shape != x.shape or t.dtype != x.dtype:
                raise _lib.PsalmKernelError("add_layer_norm: residual shape / dtype mismatch")
    y = torch.empty_like(x)
    s = torch.empty_like(x) if return_sum else None
    rc = _lib.lib().psalm_add_layernorm(
        _lib.ptr(x), _lib.ptr(r1) if r1 is not None else None, _lib.ptr(r2) if r2 is not None else None,
        _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(s) if s is not None else None, _lib.ptr(y),
        x.numel() // C, C, float(eps), _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    _lib.check(rc, "psalm_add_layernorm")
    _count()
    return (s, y) if return_sum else y


@_on_device
def group_norm_tokens(x, weight, bias, groups=32, eps=1e-5, relu=False, pre_bias=None):
    """GroupNorm(groups) (+ReLU) of a token-major map [B,N,C]; `pre_bias` [C] = bias of the producing conv / Linear,
    added inside the kernel (GroupNorm(x + pre_bias))."""
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias")) + (((pre_bias, "pre_bias"),) if pre_bias is not None else ()):
        _chk(t, "group_norm_tokens." + n)
    B, N, C = x.shape
    stats = torch.empty(B * groups * (1 + (N + 255) // 256), dtype=torch.float64, device=x.device)
    y = torch.empty_like(x)
    rc = _lib.lib().psalm_groupnorm_tokens(_lib.ptr(x), _lib.ptr(pre_bias) if pre_bias is not None else None,
                                           _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(y), _lib.ptr(stats),
                                           B, N, C, groups, float(eps), 1 if relu else 0,
                                           _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    _lib.check(rc, "psalm_groupnorm_tokens")
    _count(3)
    return y


@_on_device
def postproc_crop_supported(Q, H4, W4, Hp, Wp, oh, ow, H, W, ncls):
    return bool(_lib.lib().psalm_postproc_crop_supported(Q, H4, W4, Hp, Wp, oh, ow, H, W, ncls))


def postproc_fused(logits, H, W, probsT=None, wq=None, negq=None, slot_query=None, ncls=0, crop=None):
    """logits [Q,H4,W4] -> dict(sem_seg, ids, in_mask, inst_masks, stats [Q,5]) at output size (H, W).
    stats columns: count(x>0), sum(sigmoid*[x>0]), count(x>=0), panoptic area, panoptic intersection.
    crop = (Hp, Wp, oh, ow): up-sample to the padded size (Hp, Wp), crop to (oh, ow), resize to (H, W) (the reference's
    sem_seg_postprocess flow) composed inside the kernel; None: (H, W) is the up-sampled size itself."""
    import ctypes
    _chk(logits, "postproc_fused.logits")
    Q, H4, W4 = logits.shape
    dev = logits.device
    K = 0 if slot_query is None else slot_query.shape[0]
    rows = ctypes.c_int()
    if crop is not None:
        _lib.check(_lib.lib().psalm_postproc_crop_partials(H, W, ctypes.byref(rows)), "psalm_postproc_crop_partials")
    else:
        _lib.check(_lib.lib().psalm_postproc_partials(Q, H4, W4, H, W, ncls, K, _lib.dtype_code(logits.dtype), ctypes.byref(rows)),
                   "psalm_postproc_partials")
    partials = torch.empty((rows.value, Q, 5), dtype=torch.float32, device=dev)
    out = {}
    sem = ids = inm = inst = None
    if probsT is not None:
        _chk(probsT, "postproc_fused.probsT")
        if probsT.dtype != torch.float16 or tuple(probsT.shape) != (144, 112):
            raise _lib.PsalmKernelError("postproc_fused: probsT must be fp16 [144,112]")
        sem = torch.empty((ncls, H, W), dtype=torch.float32, device=dev)
    if wq is not None:
        ids = torch.empty((H, W), dtype=torch.int32, device=dev)
        inm = torch.empty((H, W), dtype=torch.uint8, device=dev)
    K = 0
    if slot_query is not None:
        K = slot_query.shape[0]
        inst = torch.empty((K, H, W), dtype=torch.float32, device=dev)
    p = lambda t: _lib.ptr(t) if t is not None else None  # noqa: E731
    if crop is not None:
        Hp, Wp, oh, ow = crop
        rc = _lib.lib().psalm_postproc_fused_crop(p(logits), p(probsT), p(wq), p(negq), p(slot_query), p(sem), p(inst), p(ids),
                                                  p(inm), p(partials), Q, H4, W4, Hp, Wp, oh, ow, H, W, ncls, K,
                                                  _lib.dtype_code(logits.dtype), _lib.stream_ptr(dev))
    else:
        rc = _lib.lib().psalm_postproc_fused(p(logits), p(probsT), p(wq), p(negq), p(slot_query), p(sem), p(inst), p(ids),
                                             p(inm), p(partials), Q, H4, W4, H, W, ncls, K, _lib.dtype_code(logits.dtype),
                                             _lib.stream_ptr(dev))
    _lib.check(rc, "psalm_postproc_fused")
    _count()
    out.update(sem_seg=sem, ids=ids, in_mask=inm, inst_masks=inst, stats=partials.sum(0))
    return out


@_on_device
def mask_bits(mask_embed, feats):
    """Attention mask of the next decoder layer from (mask_embed [B,Q,C], pooled feats [B,P,C]):
    (bits int32 [B,Q,ceil(P/32)], row_open uint8 [B,Q]).  16-bit storage: one tensor-core kernel that never
    writes the logits; fp32 storage: exact fp32 projection + threshold kernel."""
    _chk(mask_embed, "mask_bits.mask_embed")
    _chk(feats, "mask_bits.feats")
    B, Q, C = mask_embed.shape
    P = feats.shape[1]
    if mask_embed.dtype == torch.float32 or C != 256 or Q > 112:
        return attn_mask_bits(mask_logits(mask_embed, feats, out_dtype=torch.float32))
    bits = torch.empty((B, Q, (P + 31) // 32), dtype=torch.int32, device=feats.device)
    row_open = torch.empty((B, Q), dtype=torch.uint8, device=feats.device)
    rc = _lib.lib().psalm_mask_bits_fused(_lib.ptr(mask_embed), _lib.ptr(feats), _lib.ptr(bits), _lib.ptr(row_open),
                                          B, Q, P, C, _lib.dtype_code(feats.dtype), _lib.stream_ptr(feats.device))
    _lib.check(rc, "psalm_mask_bits_fused")
    _count(2)
    return bits, row_open


def linear_act(x, weight, bias, act):
    """Linear + activation with the activation in the library GEMM's epilogue (cuBLASLt) for 16-bit CUDA
    tensors: act = "relu" or "gelu_tanh" (gelu_new).  Library plumbing, not a custom kernel."""
    import torch.nn.functional as F
    if x.is_cuda and x.dtype != torch.float32:
        shp = x.shape
        y = torch._addmm_activation(bias, x.reshape(-1, shp[-1]), weight.t(), use_gelu=(act == "gelu_tanh"))
        return y.view(*shp[:-1], weight.shape[0])
    y = F.linear(x, weight, bias)
    return F.relu(y) if act == "relu" else F.gelu(y, approximate="tanh")


@_on_device
def patch_merge_layer_norm(x, H, W, weight, bias, eps=1e-5):
    """Swin PatchMerging gather + LayerNorm (swin_trans.py:269-296): x [B, H*W, C] -> [B, ceil(H/2)*ceil(W/2), 4C]
    normalised over the concatenated 2x2 neighbourhood (zero padded to even H / W)."""
    for t, n in ((x, "x"), (weight, "weight"), (bias, "bias")):
        _chk(t, "patch_merge_layer_norm." + n)
    B, N, C = x.shape
    if N != H * W or weight.numel() != 4 * C:
        raise _lib.PsalmKernelError("patch_merge_layer_norm: x is [B, H*W, C], weight / bias have 4C entries")
    y = torch.empty((B, ((H + 1) // 2) * ((W + 1) // 2), 4 * C), dtype=x.dtype, device=x.device)
    rc = _lib.lib().psalm_patch_merge_layernorm(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(y), B, H, W, C,
                                                float(eps), _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    _lib.check(rc, "psalm_patch_merge_layernorm")
    _count()
    return y


@_on_device
def region_pool(tokens, points, region_image, h, w):
    """tokens [B, h*w, C]; points [R, P, 2] fp32 (y, x) in [0, 1]; region_image [R] int32 -> [R, C]: mean over the P
    points of grid_sample(align_corners=True) on the image's token map (context_cluster.py:333-400)."""
    for t, n in ((tokens, "tokens"), (points, "points"), (region_image, "region_image")):
        _chk(t, "region_pool." + n)
    B, N, C = tokens.shape
    R, P, two = points.shape
    if N != h * w or two != 2 or points.dtype != torch.float32 or region_image.dtype != torch.int32 or region_image.numel() != R:
        raise _lib.PsalmKernelError("region_pool: tokens [B,h*w,C], points [R,P,2] fp32, region_image [R] int32")
    out = torch.empty((R, C), dtype=tokens.dtype, device=tokens.device)
    rc = _lib.lib().psalm_region_pool(_lib.ptr(tokens), _lib.ptr(points), _lib.ptr(region_image), _lib.ptr(out), B, h, w, C, R, P,
                                      _lib.dtype_code(tokens.dtype), _lib.stream_ptr(tokens.device))
    _lib.check(rc, "psalm_region_pool")
    _count()
    return out


_RLE_DT = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16, torch.uint8: _lib.U8,
           torch.bool: _lib.U8}


@_on_device
def mask_rle(masks):
    """Binary masks [K,H,W] (K >= 1; fp32 / fp16 / bf16 / uint8 / bool, non-zero = foreground) -> the COCO RLE of every mask
    (pycocotools maskApi.c rleEncode + rleToString, csrc/rle.cu) on the current stream:
      counts      uint32 [sum of run counts] run lengths in column-major order, mask k's at run_offsets[k]:run_offsets[k+1]
      run_offsets int64 [K+1] on the device
      strings     uint8 [sum of string lengths] the compressed counts strings, on the device
      str_offsets int64 [K+1] on the host: mask k's string is strings[str_offsets[k]:str_offsets[k+1]].
    Two small host synchronisations (the total run count, then the string offsets) size the outputs exactly."""
    _chk(masks, "mask_rle.masks")
    if masks.dim() != 3 or masks.shape[0] == 0:
        raise _lib.PsalmKernelError("mask_rle: expected masks [K,H,W] with K >= 1, got %s" % (tuple(masks.shape),))
    if masks.dtype not in _RLE_DT:
        raise _lib.PsalmKernelError("mask_rle: unsupported dtype %s" % masks.dtype)
    K, H, W = masks.shape
    dev = masks.device
    L = _lib.lib()
    st = _lib.stream_ptr(dev)
    ws = torch.empty(L.psalm_mask_rle_workspace_bytes(K, H, W), dtype=torch.uint8, device=dev)
    run_offsets = torch.empty(K + 1, dtype=torch.int64, device=dev)
    rc = L.psalm_mask_rle_sizes(_lib.ptr(masks), _lib.ptr(ws), ws.numel(), _lib.ptr(run_offsets), K, H, W,
                                _RLE_DT[masks.dtype], st)
    _lib.check(rc, "psalm_mask_rle_sizes")
    _count(4)
    counts = torch.empty(int(run_offsets[K].item()), dtype=torch.int32, device=dev).view(torch.uint32)   # host sync 1
    str_offsets_dev = torch.empty(K + 1, dtype=torch.int64, device=dev)
    rc = L.psalm_mask_rle_runs(_lib.ptr(ws), ws.numel(), _lib.ptr(run_offsets), _lib.ptr(counts),
                               _lib.ptr(str_offsets_dev), K, H, W, st)
    _lib.check(rc, "psalm_mask_rle_runs")
    _count(3)
    str_offsets = str_offsets_dev.cpu()                                                                      # host sync 2
    strings = torch.empty(int(str_offsets[K]), dtype=torch.uint8, device=dev)
    rc = L.psalm_mask_rle_write(_lib.ptr(counts), _lib.ptr(run_offsets), _lib.ptr(str_offsets_dev),
                                _lib.ptr(strings), K, st)
    _lib.check(rc, "psalm_mask_rle_write")
    _count()
    return counts, run_offsets, strings, str_offsets


LINEAR_FUSED = True   # False: library GEMM + separate elementwise pass (A/B runs)
_EPILOGUES = {"bias": 0, "gelu_erf": 1, "head_major": 2}


def linear_fused_supported(x, weight, epilogue, rows_per_image=0):
    """True when `linear_fused` applies: 16-bit CUDA tensors, N % 256 == 0, K % 64 == 0."""
    if not (LINEAR_FUSED and x.is_cuda and x.dtype in (torch.bfloat16, torch.float16)):
        return False
    M = x.numel() // x.shape[-1]
    return bool(_lib.lib().psalm_linear_fused_supported(M, weight.shape[0], weight.shape[1], _EPILOGUES[epilogue],
                                                        rows_per_image, _lib.dtype_code(x.dtype)))


@_on_device
def linear_fused(x, weight, bias, epilogue, rows_per_image=0):
    """epilogue(x @ weight.T + bias) on the tcgen05 tensor cores (csrc/gemm_tc5.cu).  x [..., K] (rows contiguous),
    weight [N, K].  epilogue: "bias", "gelu_erf" (Swin Mlp.fc1 + nn.GELU, swin_trans.py:37-44) or "head_major"
    (MSDeformAttn value_proj stored [B, N/32, rows_per_image, 32], ms_deform_attn.py:95-99)."""
    _chk(weight, "linear_fused.weight")
    if not x.is_cuda:
        raise _lib.PsalmKernelError("linear_fused.x: expected a CUDA tensor, got %s (no CPU path)" % x.device)
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x if x.dim() == 2 else x.reshape(-1, K)     # a 2-D row-strided view is consumed in place (TMA row stride)
    if x2.stride(-1) != 1 or x2.stride(0) % 8 or x2.data_ptr() % 16:
        x2 = x2.contiguous()
    M = x2.shape[0]
    if epilogue == "head_major":
        out = torch.empty((M // rows_per_image, N // 32, rows_per_image, 32), dtype=x.dtype, device=x.device)
    else:
        out = torch.empty(tuple(x.shape[:-1]) + (N,), dtype=x.dtype, device=x.device)
    if bias is not None and (bias.dtype != x.dtype or not bias.is_contiguous()):
        raise _lib.PsalmKernelError("linear_fused: bias must be contiguous and of the storage dtype")
    rc = _lib.lib().psalm_linear_fused(_lib.ptr(x2), x2.stride(0), _lib.ptr(weight), _lib.ptr(bias) if bias is not None else None,
                                       _lib.ptr(out), M, N, K, _EPILOGUES[epilogue], rows_per_image,
                                       _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    _lib.check(rc, "psalm_linear_fused")
    _count()
    return out


@_on_device
def patchify(images, out_dtype, mean=None, std=None, patch=4):
    """images [B,Cin,H,W] (uint8 / float) -> patches [B, ceil(H/4)*ceil(W/4), Cin*16] in out_dtype, normalised with
    (x - mean) / std when given, zero padded to the patch grid.  coco_panoptic_mapper.py:161 + swin_trans.py:427-441."""
    _chk(images, "patchify.images")
    B, Cin, H, W = images.shape
    Wh, Ww = -(-H // patch), -(-W // patch)
    out = torch.empty((B, Wh * Ww, Cin * patch * patch), dtype=out_dtype, device=images.device)
    if (mean is None) != (std is None):
        raise _lib.PsalmKernelError("patchify: mean and std come together")
    for t in (mean, std):
        if t is not None and (t.dtype != torch.float32 or t.numel() != Cin or not t.is_cuda):
            raise _lib.PsalmKernelError("patchify: mean / std must be fp32 CUDA tensors of %d values" % Cin)
    rc = _lib.lib().psalm_patchify(_lib.ptr(images), _lib.ptr(out), _lib.ptr(mean) if mean is not None else None,
                                   _lib.ptr(std) if std is not None else None, B, Cin, H, W, patch,
                                   _lib.dtype_code(images.dtype), _lib.dtype_code(out_dtype), _lib.stream_ptr(images.device))
    _lib.check(rc, "psalm_patchify")
    _count()
    return out, (Wh, Ww)


@_on_device
def masked_cross_attention(q, k, v, mask_bits=None, row_open=None, nh=8, workspace=None):
    """q [B,Lq,256]; k, v [B,Lk,256] possibly ROW-STRIDED views (last dim contiguous, batch stride = Lk * row stride)
    -> [B,Lq,256].  TMA-fed kernel of csrc/xattn_tma.cu (16-bit storage, 8 heads x 32)."""
    _chk(q, "masked_cross_attention.q")
    B, Lq, C = q.shape
    Lk = k.shape[1]
    ld = k.stride(1)
    for t, n in ((k, "k"), (v, "v")):
        if not t.is_cuda or t.dtype != q.dtype or tuple(t.shape) != (B, Lk, C) or t.stride(2) != 1 or t.stride(1) != ld or \
                (B > 1 and t.stride(0) != Lk * ld):
            raise _lib.PsalmKernelError("masked_cross_attention.%s: expected a [B,Lk,%d] view with contiguous rows and a "
                                        "common row stride" % (n, C))
    L = _lib.lib()
    need = L.psalm_masked_cross_attention_workspace_bytes(B, Lq, Lk)
    if need and (workspace is None or workspace.numel() * workspace.element_size() < need):
        workspace = torch.empty(need // 4, dtype=torch.float32, device=q.device)
    out = torch.empty_like(q)
    rc = L.psalm_masked_cross_attention(
        _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), ld, _lib.ptr(mask_bits) if mask_bits is not None else None,
        _lib.ptr(row_open) if row_open is not None else None, _lib.ptr(out),
        _lib.ptr(workspace) if need else None, workspace.numel() * workspace.element_size() if need else 0,
        B, Lq, Lk, nh, C // nh, _lib.dtype_code(q.dtype), _lib.stream_ptr(q.device))
    _lib.check(rc, "psalm_masked_cross_attention")
    _count(2 if need else 1)
    return out


@_on_device
def kv_cache_write(qkv, kcache, vcache, block_table, start_pos):
    """qkv [B,T,3,nh,hd] (rotary applied): K / V rows of the T tokens -> cache pages [num_pages,nh,page,hd] at positions
    start_pos[b] + t through block_table [B,max_pages] (int32)."""
    _chk(qkv, "kv_cache_write.qkv")
    B, T, _, nh, hd = qkv.shape
    rc = _lib.lib().psalm_kv_cache_write(_lib.ptr(qkv), _lib.ptr(kcache), _lib.ptr(vcache), _lib.ptr(block_table),
                                         _lib.ptr(start_pos), B, T, nh, hd, kcache.shape[2], block_table.shape[1],
                                         _lib.dtype_code(qkv.dtype), _lib.stream_ptr(qkv.device))
    _lib.check(rc, "psalm_kv_cache_write")
    _count()


@_on_device
def paged_decode_attention(qkv, kcache, vcache, block_table, seq_lens):
    """qkv [B,1,3,nh,hd] of the new token (its K / V already written to the cache) -> [B,1,nh*hd]: attention of the new
    query over the first seq_lens[b] cached keys."""
    _chk(qkv, "paged_decode_attention.qkv")
    B, T, _, nh, hd = qkv.shape
    if T != 1:
        raise _lib.PsalmKernelError("paged_decode_attention: one query token per sequence")
    out = torch.empty((B, 1, nh * hd), dtype=qkv.dtype, device=qkv.device)
    rc = _lib.lib().psalm_paged_decode_attention(_lib.ptr(qkv), 3 * nh * hd, _lib.ptr(kcache), _lib.ptr(vcache),
                                                 _lib.ptr(block_table), _lib.ptr(seq_lens), _lib.ptr(out), B, nh, hd,
                                                 kcache.shape[2], block_table.shape[1], _lib.dtype_code(qkv.dtype),
                                                 _lib.stream_ptr(qkv.device))
    _lib.check(rc, "psalm_paged_decode_attention")
    _count()
    return out
