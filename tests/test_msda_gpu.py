"""GPU parity of the sm_100a MSDeformAttn kernels (through the C ABI) against the C oracle, the
reference-generated golden vectors and, at full size, the reference's own CUDA kernels + properties.

Tolerances: fp64 1e-10 rel (reference check: torch.allclose default, ops/test.py:40);
fp32 1e-4 rel / 1e-5 abs-of-scale, far inside the north star's 1e-3 (ops/test.py:56 uses 1e-2/1e-3).
"""
import glob
import os
import zlib

import numpy as np
import pytest
import torch

from oracle import msda as oracle_msda

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(os.path.basename(p)[5:-4] for p in glob.glob(os.path.join(GOLDEN, "msda_*.npz")))
FULL_SHAPES = [(48, 160), (24, 80), (12, 40), (6, 20)]


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _tol(dtype):
    return (1e-10, 1e-12) if dtype in (np.float64, torch.float64) else (1e-4, 1e-5)


def _close(a, b, rtol, atol, name):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else b
    scale = max(1.0, float(np.abs(b).max())) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol * scale, err_msg=name)


def _run_cuda(value, shapes, lsi, loc, attn, grad_out):
    from monodetr_b200.msda import ms_deform_attn_backward, ms_deform_attn_forward
    out = ms_deform_attn_forward(value, shapes, lsi, loc, attn, 64)
    gv, gl, ga = ms_deform_attn_backward(value, shapes, lsi, loc, attn, grad_out, 64)
    torch.cuda.synchronize()
    return out, gv, gl, ga


def _make(seed, shapes, N, M, D, Lq, P, dtype, lo=-0.1, hi=1.1):
    g = torch.Generator().manual_seed(seed)
    shapes_t = torch.as_tensor(shapes, dtype=torch.long)
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    S = int(shapes_t.prod(1).sum())
    L = len(shapes)
    value = torch.randn(N, S, M, D, generator=g, dtype=dtype)
    loc = torch.rand(N, Lq, M, L, P, 2, generator=g, dtype=dtype) * (hi - lo) + lo
    attn = torch.softmax(torch.randn(N, Lq, M, L * P, generator=g, dtype=dtype), -1).view(N, Lq, M, L, P)
    grad_out = torch.randn(N, Lq, M * D, generator=g, dtype=dtype)
    return shapes_t, lsi, value, loc, attn, grad_out


@pytest.mark.parametrize("name", CASES)
def test_golden_vectors(name):
    g = np.load(os.path.join(GOLDEN, f"msda_{name}.npz"))
    rtol, atol = _tol(g["value"].dtype)
    out, gv, gl, ga = _run_cuda(*(_dev(g[k]) for k in ("value", "shapes", "lsi", "loc", "attn", "grad_out")))
    _close(out, g["out"], rtol, atol, "out")
    _close(gv, g["grad_value"], rtol, atol, "grad_value")
    _close(gl, g["grad_loc"], rtol, atol, "grad_loc")
    _close(ga, g["grad_attn"], rtol, atol, "grad_attn")


@pytest.mark.parametrize("cfg", [
    # (shapes, N, M, D, Lq, P, dtype)  -- fast path D in {16,32,64}, P=4; everything else generic
    ([(12, 40), (6, 20), (3, 10), (2, 5)], 2, 8, 32, 53, 4, torch.float32),
    ([(12, 40), (6, 20), (3, 10), (2, 5)], 1, 8, 32, 1, 4, torch.float32),      # single query, ragged warp tail
    ([(12, 40), (6, 20), (3, 10), (2, 5)], 3, 7, 32, 5, 4, torch.float32),      # M not a multiple of 4
    ([(9, 11), (4, 5), (2, 2), (1, 1)], 2, 4, 64, 9, 4, torch.float32),
    ([(9, 11), (4, 5), (2, 2), (1, 1)], 2, 6, 16, 10, 4, torch.float32),
    ([(9, 11), (4, 5)], 2, 4, 32, 9, 4, torch.float32),                          # L=2: fast fwd, generic bwd
    ([(6, 4), (3, 2)], 1, 2, 30, 2, 2, torch.float64),                           # reference gradcheck channel counts
    ([(6, 4), (3, 2)], 1, 2, 71, 2, 2, torch.float64),
    ([(6, 4), (3, 2)], 1, 2, 1025, 2, 2, torch.float64),
    ([(6, 4), (3, 2)], 1, 2, 8, 2, 3, torch.float32),
    ([(1, 1)], 1, 1, 32, 3, 4, torch.float32),                                   # 1x1 level: every corner clipped
])
def test_against_oracle(cfg):
    shapes, N, M, D, Lq, P, dtype = cfg
    shapes_t, lsi, value, loc, attn, grad_out = _make(zlib.crc32(repr(cfg).encode()) % 1000, shapes, N, M, D, Lq, P, dtype, -0.2, 1.2)
    rtol, atol = _tol(dtype)
    out, gv, gl, ga = _run_cuda(*(t.cuda() for t in (value, shapes_t, lsi, loc, attn, grad_out)))
    npv = [t.numpy() for t in (value, shapes_t, lsi, loc, attn)]
    _close(out, oracle_msda.msda_forward(*npv), rtol, atol, "out")
    ogv, ogl, oga = oracle_msda.msda_backward(*npv, grad_out.numpy())
    _close(gv, ogv, rtol, atol, "grad_value")
    _close(gl, ogl, rtol, atol, "grad_loc")
    _close(ga, oga, rtol, atol, "grad_attn")


def test_empty_inputs():
    from monodetr_b200.msda import ms_deform_attn_backward, ms_deform_attn_forward
    shapes_t, lsi, value, loc, attn, grad_out = _make(1, [(4, 4)], 2, 2, 32, 0, 4, torch.float32)
    out = ms_deform_attn_forward(value.cuda(), shapes_t.cuda(), lsi.cuda(), loc.cuda(), attn.cuda(), 64)
    assert out.shape == (2, 0, 64)
    gv, gl, ga = ms_deform_attn_backward(value.cuda(), shapes_t.cuda(), lsi.cuda(), loc.cuda(), attn.cuda(),
                                         grad_out.cuda(), 64)
    assert gv.shape == value.shape and not gv.any() and gl.numel() == 0 and ga.numel() == 0


def test_all_points_outside_give_exact_zero():
    shapes_t, lsi, value, loc, attn, grad_out = _make(2, FULL_SHAPES, 1, 8, 32, 64, 4, torch.float32)
    loc = loc * 0 + 5.0
    loc[..., 0, :, :] = -4.0
    out, gv, gl, ga = _run_cuda(*(t.cuda() for t in (value, shapes_t, lsi, loc, attn, grad_out)))
    for t in (out, gv, gl, ga):
        assert not t.any()


def test_autograd_function_matches_oracle_gradients():
    from monodetr_b200.msda import MSDeformAttnFunction
    shapes_t, lsi, value, loc, attn, grad_out = _make(5, [(6, 20), (3, 10), (2, 5), (1, 3)], 2, 8, 32, 17, 4, torch.float32)
    v, lo, a = (t.cuda().requires_grad_(True) for t in (value, loc, attn))
    out = MSDeformAttnFunction.apply(v, shapes_t.cuda(), lsi.cuda(), lo, a, 64)
    out.backward(grad_out.cuda())
    npv = [t.numpy() for t in (value, shapes_t, lsi, loc, attn)]
    ogv, ogl, oga = oracle_msda.msda_backward(*npv, grad_out.numpy())
    _close(v.grad, ogv, 1e-4, 1e-5, "grad_value")
    _close(lo.grad, ogl, 1e-4, 1e-5, "grad_loc")
    _close(a.grad, oga, 1e-4, 1e-5, "grad_attn")


def test_gradcheck_fp64_like_reference():
    """The reference's check_gradient_numerical (ops/test.py:63-78) on the generic fp64 kernels."""
    from torch.autograd import gradcheck
    from monodetr_b200.msda import MSDeformAttnFunction
    shapes_t, lsi, value, loc, attn, _ = _make(3, [(6, 4), (3, 2)], 1, 2, 30, 2, 2, torch.float64, 0.0, 1.0)
    value = value * 0.01
    args = (value.cuda().requires_grad_(True), shapes_t.cuda(), lsi.cuda(), loc.cuda().requires_grad_(True),
            attn.cuda().requires_grad_(True), 2)
    assert gradcheck(MSDeformAttnFunction.apply, args)


def full_size_case(Lq):
    """BASELINE config-2 shapes (4 levels of a 1280x384 image, 8 heads x 32, 4 points): value, shapes, lsi, loc, attn, grad_out."""
    N = 2 if Lq == 10200 else 8
    shapes_t, lsi, value, loc, attn, grad_out = _make(7 + Lq, FULL_SHAPES, N, 8, 32, Lq, 4, torch.float32, 0.0, 1.0)
    return value, shapes_t, lsi, loc, attn, grad_out


@pytest.mark.parametrize("Lq", [50, 550, 10200])
def test_full_size_against_oracle_and_reference_kernels(Lq):
    """Against the C oracle, and against the reference's own CUDA kernels on the same inputs: their results are stored
    as max|x| and a seeded sample in tests/golden/reference_msda_kernels.npz (tools/gen_golden_msda_ref_kernels.py)."""
    value, shapes_t, lsi, loc, attn, grad_out = full_size_case(Lq)
    dv = [t.cuda() for t in (value, shapes_t, lsi, loc, attn, grad_out)]
    out, gv, gl, ga = _run_cuda(*dv)
    npv = [t.numpy() for t in (value, shapes_t, lsi, loc, attn)]
    _close(out, oracle_msda.msda_forward(*npv), 1e-4, 1e-5, "out")
    ogv, ogl, oga = oracle_msda.msda_backward(*npv, grad_out.numpy())
    _close(gv, ogv, 2e-4, 2e-5, "grad_value")   # fp32 atomics: summation order differs run to run
    _close(gl, ogl, 1e-4, 1e-5, "grad_loc")
    _close(ga, oga, 1e-4, 1e-5, "grad_attn")
    g = np.load(os.path.join(GOLDEN, "reference_msda_kernels.npz"))
    for name, t, rtol, atol in (("out", out, 1e-4, 1e-5), ("grad_value", gv, 2e-4, 2e-5), ("grad_loc", gl, 1e-4, 1e-5),
                                ("grad_attn", ga, 1e-4, 1e-5)):
        key = f"Lq{Lq}.{name}"
        a = t.detach().cpu().numpy().reshape(-1)
        ref_max = float(g[key + ".absmax"])
        atol *= max(1.0, ref_max)
        np.testing.assert_allclose(a[g[key + ".idx"]], g[key + ".val"], rtol=rtol, atol=atol, err_msg=name + " vs reference CUDA kernel")
        np.testing.assert_allclose(np.abs(a).max(), ref_max, rtol=rtol, atol=atol, err_msg=name + " max vs reference CUDA kernel")


def test_full_size_properties():
    """Size-independent properties at B=8, Lq=10200: linearity in value, and sum(grad_attn*attn) == <out, grad_out>."""
    from monodetr_b200.msda import ms_deform_attn_backward, ms_deform_attn_forward
    shapes_t, lsi, value, loc, attn, grad_out = _make(99, FULL_SHAPES, 8, 8, 32, 10200, 4, torch.float32, 0.0, 1.0)
    v, sh, ls, lo, a, go = (t.cuda() for t in (value, shapes_t, lsi, loc, attn, grad_out))
    v2 = torch.randn_like(v)
    o1 = ms_deform_attn_forward(v, sh, ls, lo, a, 64)
    o2 = ms_deform_attn_forward(v2, sh, ls, lo, a, 64)
    o12 = ms_deform_attn_forward(v * 0.5 + v2 * 2.0, sh, ls, lo, a, 64)
    assert torch.allclose(o12, o1 * 0.5 + o2 * 2.0, rtol=1e-4, atol=1e-4)
    gv, gl, ga = ms_deform_attn_backward(v, sh, ls, lo, a, go, 64)
    # out is linear in attn and in value: <grad_attn, attn> == <grad_value, value> == <out, grad_out>
    ref = (o1.double() * go.double()).sum()
    assert abs((ga.double() * a.double()).sum() - ref) <= 1e-5 * abs(ref) + 1e-2
    assert abs((gv.double() * v.double()).sum() - ref) <= 1e-4 * abs(ref) + 1e-1


@pytest.mark.parametrize("Lq,rd,B", [(10200, 2, 2), (550, 6, 3), (53, 2, 1)])
def test_fused_preprocessing_matches_the_two_step_path(Lq, rd, B):
    """MSDeformAttn module path: softmax / sampling-location pre-processing INSIDE the sampling kernels
    (mdb_msda_fused_*) against the separate pre-processing kernel + the op (both pinned above / in test_elementwise_gpu.py),
    forward and the gradients wrt value, raw offsets and raw logits."""
    from monodetr_b200 import functional as Fn
    g = torch.Generator(device="cuda").manual_seed(Lq + rd)
    shapes_t = torch.as_tensor(FULL_SHAPES, dtype=torch.long, device="cuda")
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    S = int(shapes_t.prod(1).sum())
    value = torch.randn(B, S, 8, 32, device="cuda", generator=g)
    off = torch.randn(B, Lq, 8 * 4 * 4 * 2, device="cuda", generator=g) * 3
    logits = torch.randn(B, Lq, 8 * 16, device="cuda", generator=g) * 2
    ref = torch.rand(B, Lq, 4, rd, device="cuda", generator=g)
    if rd == 6:
        ref[..., 2:] *= 0.2
    dout = torch.randn(B, Lq, 256, device="cuda", generator=g)
    ins = [t.clone().requires_grad_() for t in (value, off, logits)]
    assert Fn.msda_fused_applicable(ins[0], ref, 4, 4)
    out = Fn.msda_fused(ins[0], shapes_t, lsi, ins[1], ins[2], ref)
    gv, go, gl = torch.autograd.grad(out, ins, dout)
    v2, o2, l2 = [t.clone().requires_grad_() for t in (value, off, logits)]
    loc, attn = Fn.msda_prep(o2, l2, ref, shapes_t, 8, 4, 4)
    ref_out = Fn.msda(v2, shapes_t, lsi, loc, attn)
    rv, ro, rl = torch.autograd.grad(ref_out, (v2, o2, l2), dout)
    _close(out, ref_out, 1e-5, 1e-6, "out")
    _close(gv, rv, 2e-4, 2e-5, "grad_value")
    _close(go, ro, 1e-4, 1e-5, "grad_offsets")
    _close(gl, rl, 1e-4, 1e-5, "grad_logits")
    assert not Fn.msda_fused_applicable(ins[0], ref.clone().requires_grad_(), 4, 4)      # boxes that need a gradient: two-step path


@pytest.fixture
def deterministic_mode():
    import monodetr_b200
    prev = monodetr_b200.set_deterministic(True)
    try:
        yield
    finally:
        monodetr_b200.set_deterministic(prev)


@pytest.mark.parametrize("cfg", [
    (FULL_SHAPES, 2, 8, 32, 1100, 4, torch.float32),                            # the model's configuration (fast-path shape)
    ([(9, 11), (4, 5), (2, 2), (1, 1)], 2, 6, 16, 40, 4, torch.float32),
    ([(6, 4), (3, 2)], 1, 2, 71, 6, 2, torch.float64),                          # generic shapes: ragged D, fp64
])
def test_deterministic_backward_is_bit_reproducible_and_matches_the_oracle(cfg, deterministic_mode):
    """mdb_set_deterministic(1): the value gradient is accumulated in a fixed order (the default path and the reference's
    kernel, ms_deform_im2col_cuda.cuh:125-152, scatter with atomics): two runs give the same bits, the values are the oracle's,
    and they agree with the default (atomic) path to rounding.  Points are concentrated so that rows really collide."""
    from monodetr_b200.msda import ms_deform_attn_backward
    import monodetr_b200
    shapes, N, M, D, Lq, P, dtype = cfg
    shapes_t, lsi, value, loc, attn, grad_out = _make(11 + Lq, shapes, N, M, D, Lq, P, dtype, 0.3, 0.7)
    dv = [t.cuda() for t in (value, shapes_t, lsi, loc, attn, grad_out)]
    runs = [ms_deform_attn_backward(*dv, 64) for _ in range(2)]
    torch.cuda.synchronize()
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    rtol, atol = _tol(dtype)
    npv = [t.numpy() for t in (value, shapes_t, lsi, loc, attn)]
    for got, want, name in zip(runs[0], oracle_msda.msda_backward(*npv, grad_out.numpy()), ("grad_value", "grad_loc", "grad_attn")):
        _close(got, want, 2 * rtol, 2 * atol, name)
    monodetr_b200.set_deterministic(False)
    try:
        default = ms_deform_attn_backward(*dv, 64)
    finally:
        monodetr_b200.set_deterministic(True)
    for got, want, name in zip(runs[0], default, ("grad_value", "grad_loc", "grad_attn")):
        _close(got, want, 2 * rtol, 2 * atol, name + " vs the atomic path")


def test_deterministic_module_path_takes_the_ordered_scatter(deterministic_mode):
    """In the reproducible mode the MSDeformAttn module leaves the fused kernels (whose backward scatters with vector
    reductions) for the two-step path, and a whole module forward + backward is bit-identical from run to run."""
    from monodetr_b200 import functional as Fn
    from monodetr_b200.ms_deform_attn import MSDeformAttn
    torch.manual_seed(3)
    mod = MSDeformAttn(256, 4, 8, 4).cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    shapes = [(12, 40), (6, 20), (3, 10), (2, 5)]
    shapes_t = torch.as_tensor(shapes, dtype=torch.long, device="cuda")
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    S = int(shapes_t.prod(1).sum())
    src = torch.randn(2, S, 256, device="cuda", generator=g)
    query = torch.randn(2, 300, 256, device="cuda", generator=g)
    ref = torch.rand(2, 300, 4, 2, device="cuda", generator=g) * 0.2 + 0.4
    dout = torch.randn(2, 300, 256, device="cuda", generator=g)
    assert not Fn.msda_fused_applicable(src.view(2, S, 8, 32), ref, 4, 4)
    grads = []
    for _ in range(2):
        s, q = src.clone().requires_grad_(), query.clone().requires_grad_()
        out = mod(q, ref, s, shapes_t, lsi)
        params = [mod.value_proj.weight, mod.sampling_offsets.weight, mod.attention_weights.weight, mod.output_proj.weight]
        grads.append((out.detach(),) + torch.autograd.grad(out, [s, q] + params, dout))
    for a, b in zip(*grads):
        assert torch.equal(a, b)
