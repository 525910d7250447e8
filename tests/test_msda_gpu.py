"""Parity of the sm_100a MSDeformAttn kernels (through the C ABI) against the oracle and the
reference-generated golden vectors.  fp32: tight tolerance; 16-bit storage: output-rounding bound."""
import numpy as np
import pytest
import torch

from oracle import msda_oracle
from psalm_b200 import msda

pytestmark = pytest.mark.gpu

DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
# relative-to-max tolerance of a result rounded to the storage type (inputs are pre-rounded, math is fp32)
TOL = {"f32": 5e-6, "f16": 1.5e-3, "bf16": 1e-2}


def _starts(shapes):
    hw = [int(h) * int(w) for h, w in shapes]
    return [int(x) for x in np.concatenate([[0], np.cumsum(hw)[:-1]])]


def _run(value, shapes, loc, aw, dt, loc_dt=None, layout=0, device_shapes=False):
    dev = "cuda"
    v = torch.from_numpy(value).to(dev).to(DT[dt])
    if layout == 1:
        v = v.permute(0, 2, 1, 3).contiguous()
    ldt = DT[loc_dt or dt]
    l = torch.from_numpy(loc).to(dev).to(ldt)
    w = torch.from_numpy(aw).to(dev).to(ldt)
    sh = [(int(h), int(w_)) for h, w_ in shapes]
    st = _starts(sh)
    if device_shapes:
        sh_t = torch.tensor(sh, dtype=torch.long, device=dev)
        st_t = torch.tensor(st, dtype=torch.long, device=dev)
        out = msda.ms_deform_attn_forward(v, sh_t, st_t, l, w, 128, value_layout=layout)
    else:
        out = msda.ms_deform_attn_forward(v, sh, st, l, w, 128, value_layout=layout)
    torch.cuda.synchronize()
    # oracle on exactly the values the kernel saw (after rounding to the storage types)
    vq = torch.from_numpy(value).to(DT[dt]).double().numpy()
    lq = torch.from_numpy(loc).to(ldt).double().numpy()
    wq = torch.from_numpy(aw).to(ldt).double().numpy()
    ref = msda_oracle.msda_ref(vq, np.array(sh), lq, wq, np.float64)
    return out.double().cpu().numpy(), ref


def _check(out, ref, dt):
    scale = np.abs(ref).max() + 1e-30
    err = np.abs(out - ref).max() / scale
    assert err < TOL[dt], "max error / max|ref| = %.3e (tol %.1e)" % (err, TOL[dt])


@pytest.mark.parametrize("name", ["msda_ops_test.npz", "msda_m8d32.npz", "msda_ragged.npz"])
def test_fp32_matches_reference_golden(golden, name):
    """The reference's own check (ops/test.py:50-63, rtol 1e-2 / atol 1e-3) and a much tighter one."""
    g = golden(name)
    for device_shapes in (False, True):
        out, ref = _run(g["value"], g["shapes"], g["loc"], g["aw"], "f32", device_shapes=device_shapes)
        assert np.allclose(out, g["out_f32"], rtol=1e-2, atol=1e-3)
        assert np.allclose(out, g["out_f64"], rtol=1e-4, atol=1e-8)
        _check(out, ref, "f32")


@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("loc_f32", [True, False])
def test_dtypes_layouts(golden, dt, layout, loc_f32):
    g = golden("msda_m8d32.npz")
    out, ref = _run(g["value"], g["shapes"], g["loc"], g["aw"], dt, "f32" if loc_f32 else dt, layout)
    _check(out, ref, dt)


@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_encoder_geometry_patch_schedule(dt):
    """Lq == S (the pixel-decoder case): exercises the 2-D patch schedule, ragged tile edges,
    samples far outside the maps (zero padding) and batch > 1."""
    rng = np.random.default_rng(0)
    shapes = [(5, 7), (10, 13), (20, 27)]
    S = sum(h * w for h, w in shapes)
    B, M, D, L, P = 2, 8, 32, 3, 4
    value = rng.standard_normal((B, S, M, D)).astype(np.float32)
    loc = rng.uniform(-0.3, 1.3, (B, S, M, L, P, 2)).astype(np.float32)
    aw = rng.uniform(0, 1, (B, S, M, L, P)).astype(np.float32)
    aw /= aw.sum((-1, -2), keepdims=True)
    for layout in (0, 1):
        out, ref = _run(value, shapes, loc, aw, dt, "f32", layout)
        _check(out, ref, dt)


def _fused_inputs(shapes, B, M, D, L, P, seed):
    rng = np.random.default_rng(seed)
    S = sum(h * w for h, w in shapes)
    value = rng.standard_normal((B, S, M, D)).astype(np.float32)
    off = (rng.standard_normal((B, S, M, L, P, 2)) * 3).astype(np.float32)
    logit = rng.standard_normal((B, S, M, L * P)).astype(np.float32)
    return value, off, logit


@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("impl", [1, 2, 3], ids=["single-group", "paired-columns", "tma-tiles"])
@pytest.mark.parametrize("shapes", [[(6, 9), (12, 18), (24, 36)], [(5, 7), (11, 13), (21, 27)], [(16, 16), (32, 32), (64, 64)],
                                    [(42, 42), (84, 84), (167, 167)]], ids=["even", "odd", "pow2", "ade1333"])
def test_fused_encoder_kernel(dt, impl, shapes):
    """softmax + reference points + location arithmetic fused in-kernel equals the unfused module
    arithmetic (ops/modules/ms_deform_attn.py:103-110 + get_reference_points, msdeformattn.py:76-87);
    both lane mappings of the kernel, even and odd map widths (ragged tiles, unaligned column pairs)."""
    from oracle import psalm_oracle as O
    from psalm_b200 import _lib
    if impl == 3 and dt == "f32":
        pytest.skip("the TMA-tile kernel is the 16-bit storage path")
    B, M, D, L, P = 2, 8, 32, 3, 4
    value, off, logit = _fused_inputs(shapes, B, M, D, L, P, 1)    # offsets ~ N(0, 3^2): ~10 % of the samples leave a 5-pixel halo
    S = value.shape[1]
    tdt = DT[dt]
    vq = torch.from_numpy(value).to(tdt)
    offq = torch.from_numpy(off).to(tdt)
    lgq = torch.from_numpy(logit).to(tdt)
    ow = torch.cat([offq.reshape(B, S, -1), lgq.reshape(B, S, -1)], -1).contiguous().cuda()
    v_hm = vq.permute(0, 2, 1, 3).contiguous().cuda()
    try:
        _lib.check(_lib.lib().psalm_set_msda_impl(impl), "set_msda_impl")
        out = msda.msda_encoder_fused(v_hm, ow, shapes, _starts(shapes), P)
        torch.cuda.synchronize()
    finally:
        _lib.lib().psalm_set_msda_impl(0)
    ref_pts = O.encoder_reference_points(shapes, B).double()
    normalizer = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float64)
    loc = ref_pts[:, :, None, :, None, :] + offq.double() / normalizer[None, None, None, :, None, :]
    aw = torch.softmax(lgq.double(), -1).view(B, S, M, L, P)
    ref = msda_oracle.msda_ref(vq.double().numpy(), np.array(shapes), loc.numpy(), aw.numpy(), np.float64)
    if dt == "f32" and max(w for _, w in shapes) > 100:
        # fp32 sampling positions (ref * W + offset) carry an absolute error ~ ulp(W): 1.4e-5 of the output at W = 167
        scale = np.abs(ref).max()
        assert np.abs(out.double().cpu().numpy() - ref).max() / scale < 4e-5
    else:
        _check(out.double().cpu().numpy(), ref, dt)


def test_full_size_properties():
    """1024^2 geometry (S = Lq = 21504, M = 8, D = 32): size-independent properties instead of the
    (slow) oracle: (a) constant value maps + in-range samples -> output == sum of weights * const;
    (b) linearity in value; (c) the two value layouts agree bit-for-bit."""
    torch.manual_seed(0)
    shapes = [(32, 32), (64, 64), (128, 128)]
    st = _starts(shapes)
    S, B, M, D, L, P = 21504, 1, 8, 32, 3, 4
    dev = "cuda"
    loc = torch.rand(B, S, M, L, P, 2, device=dev) * 0.9 + 0.05   # at least 1.6 px inside every map
    aw = torch.rand(B, S, M, L, P, device=dev)
    aw = aw / aw.sum((-1, -2), keepdim=True)
    const = torch.arange(1, M + 1, device=dev, dtype=torch.float32).view(1, 1, M, 1).expand(B, S, M, D).contiguous()
    out = msda.ms_deform_attn_forward(const, shapes, st, loc, aw)
    assert torch.allclose(out.view(B, S, M, D), const, rtol=1e-5, atol=1e-5)
    v1 = torch.randn(B, S, M, D, device=dev)
    v2 = torch.randn(B, S, M, D, device=dev)
    o1 = msda.ms_deform_attn_forward(v1, shapes, st, loc, aw)
    o2 = msda.ms_deform_attn_forward(v2, shapes, st, loc, aw)
    o12 = msda.ms_deform_attn_forward((2 * v1 - 3 * v2).contiguous(), shapes, st, loc, aw)
    assert torch.allclose(o12, 2 * o1 - 3 * o2, rtol=1e-4, atol=1e-4)
    o1_hm = msda.ms_deform_attn_forward(v1.permute(0, 2, 1, 3).contiguous(), shapes, st, loc, aw, value_layout=1)
    assert torch.equal(o1_hm, o1)
    # device-side shapes (reference contract) give the same numbers as the host-shape patch schedule
    sh_t = torch.tensor(shapes, dtype=torch.long, device=dev)
    st_t = torch.tensor(st, dtype=torch.long, device=dev)
    assert torch.equal(msda.ms_deform_attn_forward(v1, sh_t, st_t, loc, aw), o1)


def test_errors_are_loud():
    dev = "cuda"
    v = torch.zeros(1, 4, 1, 4, device=dev)
    loc = torch.zeros(1, 2, 1, 1, 1, 2, device=dev)
    w = torch.zeros(1, 2, 1, 1, 1, device=dev)
    with pytest.raises(RuntimeError):  # sum(H*W) != S
        msda.ms_deform_attn_forward(v, [(3, 3)], [0], loc, w)
    with pytest.raises(RuntimeError, match="contiguous"):
        msda.ms_deform_attn_forward(v.expand(2, 4, 1, 4)[:, ::2], [(2, 1)], [0], loc, w)


@pytest.mark.parametrize("dt", ["f32", "f16"])
def test_against_the_reference_cuda_kernel(golden, dt):
    """Same operands into the reference's ms_deform_attn_forward (ms_deformable_im2col_gpu_kernel) and ours, at the
    1024^2 encoder geometry: the two kernels must agree to accumulation-order noise.  The reference's outputs come
    from tests/golden/msda_reference_cuda_op.npz (oracle/gen_golden_ref_op.py ran its op on a B200): every output
    row of 144 seeded queries, and the max |out| of the full tensor as the error scale."""
    from oracle import gen_golden_ref_op as R
    g = golden("msda_reference_cuda_op.npz")
    value, loc, aw = R.ref_op_inputs()
    rows = g["rows"]
    assert np.array_equal(loc[0, rows[0, :8]], g["loc_probe"]), "the seeded operands changed: regenerate the fixture"
    dev = "cuda"
    v, loc, aw = (torch.from_numpy(x).to(DT[dt]).to(dev) for x in (value, loc, aw))
    sh_t = torch.tensor(R.SHAPES, dtype=torch.long, device=dev)
    st_t = torch.tensor(R.starts(R.SHAPES), dtype=torch.long, device=dev)
    ours = msda.ms_deform_attn_forward(v, sh_t, st_t, loc, aw, 128)
    torch.cuda.synchronize()
    theirs = torch.from_numpy(g["out_" + dt])
    assert ours.shape == (R.B, v.shape[1], R.M * R.D) and ours.dtype == theirs.dtype
    ours = torch.stack([ours[b, torch.from_numpy(rows[b]).to(dev)] for b in range(R.B)]).cpu()
    err = (ours.double() - theirs.double()).abs().max() / float(g["maxabs_" + dt])
    # fp32: both accumulate in fp32 (different order); fp16: the reference accumulates in HALF, we in fp32
    assert err < (2e-6 if dt == "f32" else 5e-3), err


def test_compat_module_runs_the_reference_autograd_function():
    """`import MultiScaleDeformableAttention` (the pybind module name the reference imports,
    ops/functions/ms_deform_attn_func.py:21-29) resolves to psalm_b200/compat, and a restated
    MSDeformAttnFunction.forward (func.py:34-39) runs on it unmodified; backward raises (inference build)."""
    import importlib
    import os
    import sys
    compat = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "psalm_b200", "compat")
    sys.path.insert(0, compat)
    try:
        sys.modules.pop("MultiScaleDeformableAttention", None)
        MSDA = importlib.import_module("MultiScaleDeformableAttention")
    finally:
        sys.path.remove(compat)

    class MSDeformAttnFunction(torch.autograd.Function):   # restated from func.py:32-39
        @staticmethod
        def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights,
                    im2col_step):
            ctx.im2col_step = im2col_step
            output = MSDA.ms_deform_attn_forward(value, value_spatial_shapes, value_level_start_index,
                                                 sampling_locations, attention_weights, ctx.im2col_step)
            ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                                  attention_weights)
            return output

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "msda_m8d32.npz"))
    dev = "cuda"
    shapes = torch.from_numpy(g["shapes"]).long().to(dev)
    starts = torch.tensor(_starts(g["shapes"]), dtype=torch.long, device=dev)
    out = MSDeformAttnFunction.apply(torch.from_numpy(g["value"]).to(dev), shapes, starts,
                                     torch.from_numpy(g["loc"]).to(dev), torch.from_numpy(g["aw"]).to(dev), 128)
    torch.cuda.synchronize()
    assert np.allclose(out.cpu().numpy(), g["out_f32"], rtol=1e-2, atol=1e-3)     # the reference's own tolerance
    assert np.allclose(out.cpu().numpy(), g["out_f64"], rtol=1e-4, atol=1e-8)
    with pytest.raises(NotImplementedError):
        MSDA.ms_deform_attn_backward()


def test_output_is_fully_overwritten():
    """The reference zero-initialises its output (ms_deform_attn_cuda.cu:59); ours allocates with torch.empty, so
    every element must be written by the kernel: poison the allocator's next block first."""
    torch.manual_seed(3)
    shapes = [(5, 7), (3, 4)]
    S, M, D, L, P = 47, 2, 32, 2, 3
    v = torch.randn(1, S, M, D, device="cuda")
    loc = torch.rand(1, S, M, L, P, 2, device="cuda") * 3 - 1      # many samples fall outside (zero contribution)
    aw = torch.softmax(torch.randn(1, S, M, L * P, device="cuda"), -1).view(1, S, M, L, P)
    for _ in range(3):
        poison = torch.full((1, S, M * D), float("nan"), device="cuda")
        del poison                                                   # same size: the next empty() reuses this block
        out = msda.ms_deform_attn_forward(v, shapes, _starts(shapes), loc, aw, 128)
        assert torch.isfinite(out).all()
