"""TEST INFRASTRUCTURE: a stand-in for libmonodetr_b200.so at the C-ABI level, computing on HOST memory with torch.

`FakeLib` implements the entry points of include/monodetr_b200.h that the model path calls -- in the 'tf32x3' arithmetic
mode (fp32 packed weights) and in the default 'bf16x3' mode (weights pre-split into (hi, lo) bf16 pairs) --, each from the header's own statement of what the call computes (forward formulas restated with
torch ops, backward entry points through torch.autograd of those restatements).  Pointers are plain host addresses
(`tensor.data_ptr()` of CPU tensors); results are written into the caller's buffers, exactly like the device library does.

Installed by `install(monkeypatch)` together with the few shims that let the product's HOST code run on a machine without a
GPU (a dummy CUDA stream API, `Tensor.is_cuda` -> True, `record_stream` -> no-op), it lets the `-m "not gpu"` suite drive
the whole product model -- every Python wrapper, autograd function, pointer / size / stride argument, branch-stream
fork / join -- and compare it with the oracle.  Nothing under monodetr_b200/ imports this file; the product keeps its
"no CPU path" property (without these test-scoped patches a CPU tensor raises, tests/test_capi_symbols.py).
"""
import contextlib
import ctypes
import math

import torch
import torch.nn.functional as F

from oracle.msda_torch import msda_core_torch


def _buf(ptr, n, ctype, dtype):
    if not ptr or n <= 0:
        return None
    return torch.frombuffer((ctype * n).from_address(int(ptr)), dtype=dtype)


def f32(ptr, *shape):
    t = _buf(ptr, math.prod(shape), ctypes.c_float, torch.float32)
    return None if t is None else t.view(*shape)


def f64(ptr, *shape):
    t = _buf(ptr, math.prod(shape), ctypes.c_double, torch.float64)
    return None if t is None else t.view(*shape)


def i64(ptr, *shape):
    t = _buf(ptr, math.prod(shape), ctypes.c_int64, torch.int64)
    return None if t is None else t.view(*shape)


def bf16(ptr, *shape):
    t = _buf(ptr, math.prod(shape), ctypes.c_uint16, torch.bfloat16)
    return None if t is None else t.view(*shape)


def u8(ptr, *shape):
    t = _buf(ptr, math.prod(shape), ctypes.c_uint8, torch.uint8)
    return None if t is None else t.view(*shape)


def strided(ptr, B, L, H, ld):
    """(B, L, H, 32) view of a token-strided buffer: token stride ld floats, batch stride L * ld."""
    n = (B * L - 1) * ld + H * 32
    return _buf(ptr, n, ctypes.c_float, torch.float32).as_strided((B, L, H, 32), (L * ld, ld, 32, 1))


def _ptrs(arr, n):
    """A HOST array argument (ctypes array of pointers / ints) as a python list of ints (None -> 0)."""
    return [int(arr[i] or 0) for i in range(n)]


def _grad(outs, ins, gouts):
    outs = [o for o in outs]
    return torch.autograd.grad(outs, ins, gouts, allow_unused=True)


def _prep(off, logits, ref, shapes, M, L, P, rd):
    B, Lq = off.shape[:2]
    off = off.view(B, Lq, M, L, P, 2)
    attn = F.softmax(logits.view(B, Lq, M, L * P), -1).view(B, Lq, M, L, P)
    if rd == 2:
        norm = torch.stack([shapes[:, 1], shapes[:, 0]], -1).to(off.dtype)
        loc = ref[:, :, None, :, None, :] + off / norm[None, None, None, :, None, :]
    else:   # ops/modules/ms_deform_attn.py:154-155
        loc = ref[:, :, None, :, None, :2] + off / P * (ref[:, :, None, :, None, 2::2] + ref[:, :, None, :, None, 3::2]) * 0.5
    return loc, attn


def _inverse_sigmoid(x, eps=1e-5):      # utils/misc.py:473-477
    x = x.clamp(min=0, max=1)
    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))


class FakeLib:
    """Attribute access returns the python implementation of the C function of that name; an entry point the model path should
    not need in this mode raises AttributeError (like a missing symbol would)."""

    def __init__(self, precision=1):
        self.precision = precision  # 1 = 'tf32x3': fp32 packed weights, the *_f32 entry points; 2 = 'bf16x3': pre-split (hi, lo) bf16 weights
        self.deterministic = 0
        self.calls = {}

    def __getattribute__(self, name):
        v = object.__getattribute__(self, name)
        if name.startswith("mdb_") and callable(v):
            calls = object.__getattribute__(self, "calls")
            calls[name] = calls.get(name, 0) + 1
        return v

    # ---- library state --------------------------------------------------------------------------------------------
    def mdb_abi_version(self):
        return 2

    def mdb_error_string(self, code):
        return b"fake device library: error %d" % code

    def mdb_get_precision(self):
        return self.precision

    def mdb_set_precision(self, mode):
        self.precision = mode
        return 0

    def mdb_get_deterministic(self):
        return self.deterministic

    def mdb_set_deterministic(self, on):
        self.deterministic = 1 if on else 0
        return 0

    def mdb_set_workspace(self, buf, nbytes):
        return 0

    def mdb_conv2d_forward_workspace_bytes(self, *a):
        return 0

    # ---- convolution / linear family (fp32 packed weights [tap][Cout][Cin], NHWC activations) ------------------------
    @staticmethod
    def _w_oihw(w, Cout, Cin, kh, kw):
        return f32(w, kh, kw, Cout, Cin).permute(2, 3, 0, 1)

    def mdb_conv2d_forward_f32(self, x, w, bias, residual, y, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream):
        Ho, Wo = (H + 2 * pad - kh) // stride + 1, (W + 2 * pad - kw) // stride + 1
        out = F.conv2d(f32(x, B, H, W, Cin).permute(0, 3, 1, 2), self._w_oihw(w, Cout, Cin, kh, kw), f32(bias, Cout), stride=stride,
                       padding=pad).permute(0, 2, 3, 1)
        if residual:
            out = out + f32(residual, B, Ho, Wo, Cout)
        if flags & 1:
            out = torch.relu(out)
        f32(y, B, Ho, Wo, Cout).copy_(out)
        return 0

    def mdb_conv2d_dgrad_f32(self, dy, w, residual, relu_mask, dx, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream):
        Ho, Wo = (H + 2 * pad - kh) // stride + 1, (W + 2 * pad - kw) // stride + 1
        g = torch.nn.grad.conv2d_input((B, Cin, H, W), self._w_oihw(w, Cout, Cin, kh, kw).contiguous(),
                                       f32(dy, B, Ho, Wo, Cout).permute(0, 3, 1, 2), stride=stride, padding=pad).permute(0, 2, 3, 1)
        if residual:
            g = g + f32(residual, B, H, W, Cin)
        if relu_mask:
            g = g * (f32(relu_mask, B, H, W, Cin) > 0)
        f32(dx, B, H, W, Cin).copy_(g)
        return 0

    def mdb_conv2d_wgrad_bias_f32(self, dy, x, rowscale, dw, db, B, H, W, Cin, Cout, kh, kw, stride, pad, accumulate, stream):
        Ho, Wo = (H + 2 * pad - kh) // stride + 1, (W + 2 * pad - kw) // stride + 1
        dyt = f32(dy, B, Ho, Wo, Cout)
        g = torch.nn.grad.conv2d_weight(f32(x, B, H, W, Cin).permute(0, 3, 1, 2), (Cout, Cin, kh, kw), dyt.permute(0, 3, 1, 2),
                                        stride=stride, padding=pad)
        if rowscale:
            g = g * f32(rowscale, Cout).view(-1, 1, 1, 1)
        g = g.permute(2, 3, 0, 1).reshape(kh * kw, Cout, Cin)
        out = f32(dw, kh * kw, Cout, Cin)
        out.copy_(out + g if accumulate else g)
        if db:
            s = dyt.sum((0, 1, 2))
            o = f32(db, Cout)
            o.copy_(o + s if accumulate else s)
        return 0

    def mdb_conv2d_wgrad_f32(self, dy, x, rowscale, dw, B, H, W, Cin, Cout, kh, kw, stride, pad, accumulate, stream):
        return self.mdb_conv2d_wgrad_bias_f32(dy, x, rowscale, dw, 0, B, H, W, Cin, Cout, kh, kw, stride, pad, accumulate, stream)

    # ---- precision mode 2: weights as (hi, lo) bf16 pairs, wf[tap][Cout][ceil(Cin/32)][hi 32 | lo 32] for the forward and the
    # transposed wd[tap][Cin][ceil(Cout/32)][hi 32 | lo 32] for the data gradient (zero-padded k-blocks) ------------------------
    def mdb_pack_gemm_weights_bf16x3(self, n, w, scale, wf, wd, O, I, taps, src_packed, stream):
        ws, ss = _ptrs(w, n), (_ptrs(scale, n) if scale else [0] * n)
        fs, ds = _ptrs(wf, n), (_ptrs(wd, n) if wd else [0] * n)
        for j in range(n):
            o, i, t = int(O[j]), int(I[j]), int(taps[j])
            src = f32(ws[j], t, o, i) if src_packed else f32(ws[j], o, i, t).permute(2, 0, 1)       # -> [tap][O][I]
            if ss[j]:
                src = src * f32(ss[j], o).view(1, -1, 1)
            hi = src.to(torch.bfloat16)
            lo = (src - hi.float()).to(torch.bfloat16)
            for dst, a, b, rows, cols in ((fs[j], hi, lo, o, i), (ds[j], hi.transpose(1, 2), lo.transpose(1, 2), i, o)):
                if not dst:
                    continue
                kb = (cols + 31) // 32
                out = bf16(dst, t, rows, kb, 2, 32)
                out.zero_()
                pad = kb * 32 - cols
                out[:, :, :, 0].copy_(F.pad(a, (0, pad)).reshape(t, rows, kb, 32))
                out[:, :, :, 1].copy_(F.pad(b, (0, pad)).reshape(t, rows, kb, 32))
        return 0

    @staticmethod
    def _decode_split(ptr, taps, rows, cols):
        """[tap][rows][ceil(cols/32)][hi 32 | lo 32] -> fp32 [tap][rows][cols] = hi + lo"""
        kb = (cols + 31) // 32
        t = bf16(ptr, taps, rows, kb, 2, 32).float()
        return (t[:, :, :, 0] + t[:, :, :, 1]).reshape(taps, rows, kb * 32)[:, :, :cols]

    def mdb_conv2d_forward_bf16x3(self, x, w_split, bias, residual, y, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream):
        w = self._decode_split(w_split, kh * kw, Cout, Cin).contiguous()                       # [tap][Cout][Cin]
        return self.mdb_conv2d_forward_f32(x, w.data_ptr(), bias, residual, y, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream)

    def mdb_conv2d_dgrad_bf16x3(self, dy, w_split_t, residual, relu_mask, dx, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream):
        w = self._decode_split(w_split_t, kh * kw, Cin, Cout).transpose(1, 2).contiguous()      # [tap][Cin][Cout] -> [tap][Cout][Cin]
        return self.mdb_conv2d_dgrad_f32(dy, w.data_ptr(), residual, relu_mask, dx, B, H, W, Cin, Cout, kh, kw, stride, pad, flags, stream)

    def mdb_pack_conv_weight_f32(self, w, scale, out, O, I, taps, stream):
        src = f32(w, O, I, taps)
        if scale:
            src = src * f32(scale, O).view(-1, 1, 1)
        f32(out, taps, O, I).copy_(src.permute(2, 0, 1))
        return 0

    def mdb_unpack_conv_wgrad_f32(self, dw, out, O, I, taps, accumulate, stream):
        g = f32(dw, taps, O, I).permute(1, 2, 0)
        o = f32(out, O, I, taps)
        o.copy_(o + g if accumulate else g)
        return 0

    def mdb_pack_conv_weights_multi_f32(self, n, w, scale, out, O, I, taps, stream):
        ws, ss, os_ = _ptrs(w, n), (_ptrs(scale, n) if scale else [0] * n), _ptrs(out, n)
        for j in range(n):
            self.mdb_pack_conv_weight_f32(ws[j], ss[j], os_[j], int(O[j]), int(I[j]), int(taps[j]), stream)
        return 0

    def mdb_unpack_conv_wgrads_multi_f32(self, n, dw, out, O, I, taps, stream):
        ds, os_ = _ptrs(dw, n), _ptrs(out, n)
        for j in range(n):
            self.mdb_unpack_conv_wgrad_f32(ds[j], os_[j], int(O[j]), int(I[j]), int(taps[j]), 0, stream)
        return 0

    def mdb_colsum_f32(self, x, out, M, N, accumulate, stream):
        s = f32(x, M, N).sum(0)
        o = f32(out, N)
        o.copy_(o + s if accumulate else s)
        return 0

    def mdb_round_tf32_f32(self, x, out, n, stream):
        f32(out, n).copy_(f32(x, n))
        return 0

    # ---- frozen stem -----------------------------------------------------------------------------------------------------
    def mdb_stem_conv7x7_bn_relu_f32(self, x, w, scale, bias, y, B, H, W, stream):
        H1, W1 = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
        o = F.conv2d(f32(x, B, 3, H, W), f32(w, 64, 3, 7, 7), None, stride=2, padding=3)
        o = torch.relu(o * f32(scale, 64).view(1, -1, 1, 1) + f32(bias, 64).view(1, -1, 1, 1))
        f32(y, B, H1, W1, 64).copy_(o.permute(0, 2, 3, 1))
        return 0

    def mdb_maxpool3x3s2_nhwc_f32(self, x, y, B, H, W, C, stream):
        H2, W2 = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
        f32(y, B, H2, W2, C).copy_(F.max_pool2d(f32(x, B, H, W, C).permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1))
        return 0

    # ---- elementwise helpers ------------------------------------------------------------------------------------------
    def mdb_relu_backward_f32(self, dy, y, out, n, scale, stream):
        f32(out, n).copy_(f32(dy, n) * (f32(y, n) > 0) * scale)
        return 0

    def mdb_mean3_f32(self, a, b, c, out, n, stream):
        f32(out, n).copy_((f32(a, n) + f32(b, n) + f32(c, n)) / 3)
        return 0

    def mdb_scale_f32(self, a, out, n, s, stream):
        f32(out, n).copy_(f32(a, n) * s)
        return 0

    def mdb_sum_mean_squares_forward_f32(self, count, x, n, loss, stream):
        xs = _ptrs(x, count)
        f32(loss, 1).copy_(sum((f32(xs[k], int(n[k])) ** 2).mean() for k in range(count)).view(1))
        return 0

    def mdb_sum_mean_squares_backward_f32(self, count, x, g, n, dloss, stream):
        xs, gs = _ptrs(x, count), _ptrs(g, count)
        dl = f32(dloss, 1)[0]
        for k in range(count):
            nk = int(n[k])
            f32(gs[k], nk).copy_(f32(xs[k], nk) * (2.0 / nk) * dl)
        return 0

    # ---- normalisation ------------------------------------------------------------------------------------------------
    def mdb_add_layernorm_forward_f32(self, x, res, gamma, beta, y, mean, rstd, M, C, eps, drop_p, seed, site, stream):
        assert drop_p == 0.0, "the fake library has no dropout generator: run the model with dropout 0"
        z = f32(x, M, C) if not res else f32(x, M, C) + f32(res, M, C)
        mu = z.mean(-1)
        rs = (z.var(-1, unbiased=False) + eps).rsqrt()
        f32(y, M, C).copy_((z - mu[:, None]) * rs[:, None] * f32(gamma, C) + f32(beta, C))
        f32(mean, M).copy_(mu)
        f32(rstd, M).copy_(rs)
        return 0

    def mdb_add_layernorm_backward_f32(self, dy, x, res, gamma, mean, rstd, dx, dres, dgamma, dbeta, M, C, drop_p, seed, site,
                                       accumulate, stream):
        assert drop_p == 0.0
        with torch.enable_grad():
            z = (f32(x, M, C) if not res else f32(x, M, C) + f32(res, M, C)).clone().requires_grad_()
            g = f32(gamma, C).clone().requires_grad_()
            b = torch.zeros(C, requires_grad=True)
            mu, rs = f32(mean, M), f32(rstd, M)                         # the statistics the forward call saved
            var = z.var(-1, unbiased=False, keepdim=True)
            eps_row = (1.0 / rs[:, None] ** 2 - var).detach()           # rstd = 1 / sqrt(var + eps): the call is not given eps
            yv = (z - z.mean(-1, keepdim=True)) * (var + eps_row).rsqrt() * g + b
            dz, dg, db = _grad([yv], [z, g, b], [f32(dy, M, C)])
        assert torch.allclose(mu, z.detach().mean(-1), atol=1e-4)
        f32(dx, M, C).copy_(dz)
        if dres:
            f32(dres, M, C).copy_(dz)
        for ptr, val in ((dgamma, dg), (dbeta, db)):
            o = f32(ptr, C)
            o.copy_(o + val if accumulate else val)
        return 0

    def mdb_groupnorm_forward_f32(self, x, gamma, beta, y, mean, rstd, ws, B, HW, C, G, eps, relu, stream):
        xt = f32(x, B, HW, C)
        o = F.group_norm(xt.transpose(1, 2), G, f32(gamma, C), f32(beta, C), eps).transpose(1, 2)
        f32(y, B, HW, C).copy_(torch.relu(o) if relu else o)
        xg = xt.view(B, HW, G, C // G)
        mu = xg.mean((1, 3))
        f32(mean, B, G).copy_(mu)
        f32(rstd, B, G).copy_((xg.var((1, 3), unbiased=False) + eps).rsqrt())
        self._gn_eps = eps
        return 0

    def mdb_groupnorm_backward_f32(self, dy, x, y, gamma, mean, rstd, dx, dgamma, dbeta, ws, B, HW, C, G, relu, stream):
        with torch.enable_grad():
            xt = f32(x, B, HW, C).clone().requires_grad_()
            g = f32(gamma, C).clone().requires_grad_()
            b = torch.zeros(C, requires_grad=True)
            o = F.group_norm(xt.transpose(1, 2), G, g, b, self._gn_eps).transpose(1, 2)
            gy = f32(dy, B, HW, C)
            if relu:
                gy = gy * (f32(y, B, HW, C) > 0)
            dxv, dg, db = _grad([o], [xt, g, b], [gy])
        f32(dx, B, HW, C).copy_(dxv)
        f32(dgamma, C).copy_(dg)
        f32(dbeta, C).copy_(db)
        return 0

    # ---- attention core ---------------------------------------------------------------------------------------------------
    @staticmethod
    def _attn(q, k, v, kpm):
        s = torch.einsum("bihd,bjhd->bhij", q, k) / math.sqrt(q.shape[-1])
        if kpm is not None:
            s = s.masked_fill(kpm[:, None, None, :] != 0, float("-inf"))
        return torch.einsum("bhij,bjhd->bihd", s.softmax(-1), v), torch.logsumexp(s, -1)

    def mdb_attention_forward_f32(self, q, k, v, kpm, out, lse, B, H, Lq, Lk, hd, ldq, ldk, ldv, ldo, drop_p, seed, site, stream):
        assert drop_p == 0.0 and hd == 32
        o, l = self._attn(strided(q, B, Lq, H, ldq), strided(k, B, Lk, H, ldk), strided(v, B, Lk, H, ldv), u8(kpm, B, Lk))
        strided(out, B, Lq, H, ldo).copy_(o)
        f32(lse, B, H, Lq).copy_(l)
        return 0

    def mdb_attention_backward_f32(self, q, k, v, kpm, out, lse, dout, ws, dq, dk, dv, B, H, Lq, Lk, hd, ldq, ldk, ldv, ldo, lddq,
                                   lddk, lddv, drop_p, seed, site, stream):
        assert drop_p == 0.0
        with torch.enable_grad():
            ins = [strided(p, B, L_, H, ld).clone().requires_grad_() for p, L_, ld in ((q, Lq, ldq), (k, Lk, ldk), (v, Lk, ldv))]
            o, _ = self._attn(*ins, u8(kpm, B, Lk))
            gq, gk, gv = _grad([o], ins, [strided(dout, B, Lq, H, ldo)])
        strided(dq, B, Lq, H, lddq).copy_(gq)
        strided(dk, B, Lk, H, lddk).copy_(gk)
        strided(dv, B, Lk, H, lddv).copy_(gv)
        return 0

    # ---- multi-scale deformable attention ----------------------------------------------------------------------------------
    def _msda_fwd(self, T, value, shapes, lsi, loc, attn, B, S, M, D, L, Lq, P, out):
        o = msda_core_torch(T(value, B, S, M, D), i64(shapes, L, 2), T(loc, B, Lq, M, L, P, 2), T(attn, B, Lq, M, L, P))
        T(out, B, Lq, M * D).copy_(o)
        return 0

    def _msda_bwd(self, T, value, shapes, lsi, loc, attn, gout, B, S, M, D, L, Lq, P, gv, gl, ga):
        with torch.enable_grad():
            ins = [T(value, B, S, M, D).clone().requires_grad_(), T(loc, B, Lq, M, L, P, 2).clone().requires_grad_(),
                   T(attn, B, Lq, M, L, P).clone().requires_grad_()]
            o = msda_core_torch(ins[0], i64(shapes, L, 2), ins[1], ins[2])
            a, b, c = _grad([o], ins, [T(gout, B, Lq, M * D)])
        T(gv, B, S, M, D).copy_(a)
        T(gl, B, Lq, M, L, P, 2).copy_(b)
        T(ga, B, Lq, M, L, P).copy_(c)
        return 0

    def mdb_msda_forward_f32(self, *a):
        return self._msda_fwd(f32, *a[:-1])

    def mdb_msda_forward_f64(self, *a):
        return self._msda_fwd(f64, *a[:-1])

    def mdb_msda_backward_f32(self, *a):
        return self._msda_bwd(f32, *a[:-1])

    def mdb_msda_backward_f64(self, *a):
        return self._msda_bwd(f64, *a[:-1])

    def mdb_msda_prep_forward_f32(self, off, logits, ref, shapes, B, Lq, M, L, P, rd, loc, attn, stream):
        lo, at = _prep(f32(off, B, Lq, M * L * P * 2), f32(logits, B, Lq, M * L * P), f32(ref, B, Lq, L, rd), i64(shapes, L, 2), M, L, P, rd)
        f32(loc, B, Lq, M, L, P, 2).copy_(lo)
        f32(attn, B, Lq, M, L, P).copy_(at)
        return 0

    def mdb_msda_prep_backward_f32(self, dloc, dattn, attn, ref, shapes, B, Lq, M, L, P, rd, doff, dlogits, stream):
        a = f32(attn, B, Lq, M, L * P)
        g = f32(dattn, B, Lq, M, L * P)
        f32(dlogits, B, Lq, M, L * P).copy_(a * (g - (a * g).sum(-1, keepdim=True)))
        sh, r = i64(shapes, L, 2), f32(ref, B, Lq, L, rd)
        if rd == 2:
            sc = (1.0 / torch.stack([sh[:, 1], sh[:, 0]], -1).float())[None, None, None, :, None, :]
        else:
            sc = ((r[..., 2::2] + r[..., 3::2]) * 0.5 / P)[:, :, None, :, None, :]
        f32(doff, B, Lq, M, L, P, 2).copy_(f32(dloc, B, Lq, M, L, P, 2) * sc)
        return 0

    def mdb_msda_fused_forward_f32(self, value, shapes, lsi, off, logits, ref, B, S, M, D, L, Lq, P, rd, out, stream):
        sh = i64(shapes, L, 2)
        lo, at = _prep(f32(off, B, Lq, M * L * P * 2), f32(logits, B, Lq, M * L * P), f32(ref, B, Lq, L, rd), sh, M, L, P, rd)
        f32(out, B, Lq, M * D).copy_(msda_core_torch(f32(value, B, S, M, D), sh, lo, at))
        return 0

    def mdb_msda_fused_backward_f32(self, value, shapes, lsi, off, logits, ref, gout, B, S, M, D, L, Lq, P, rd, gv, goff, glog, stream):
        sh = i64(shapes, L, 2)
        with torch.enable_grad():
            ins = [f32(value, B, S, M, D).clone().requires_grad_(), f32(off, B, Lq, M * L * P * 2).clone().requires_grad_(),
                   f32(logits, B, Lq, M * L * P).clone().requires_grad_()]
            lo, at = _prep(ins[1], ins[2], f32(ref, B, Lq, L, rd), sh, M, L, P, rd)
            a, b, c = _grad([msda_core_torch(ins[0], sh, lo, at)], ins, [f32(gout, B, Lq, M * D)])
        f32(gv, B, S, M, D).copy_(a)
        f32(goff, B, Lq, M * L * P * 2).copy_(b)
        f32(glog, B, Lq, M * L * P).copy_(c)
        return 0

    # ---- heads / depth predictor tail -------------------------------------------------------------------------------------
    @staticmethod
    def _box_refine(tmp, ref, rd):
        head = (tmp[:, :rd] + _inverse_sigmoid(ref)).sigmoid()
        return head if rd == 6 else torch.cat((head, tmp[:, rd:].sigmoid()), 1)

    def mdb_box_refine_forward_f32(self, tmp, ref, y, n, rd, stream):
        f32(y, n, 6).copy_(self._box_refine(f32(tmp, n, 6), f32(ref, n, rd), rd))
        return 0

    def mdb_box_refine_backward_f32(self, dy, y, ref, dtmp, dref, n, rd, stream):
        # (the kernel re-derives everything from y and ref; so does this: tmp = logit(y) - inverse_sigmoid(ref) on the first rd)
        with torch.enable_grad():
            yv, r = f32(y, n, 6), f32(ref, n, rd).clone().requires_grad_()
            t = torch.log(yv / (1 - yv))
            t = torch.cat((t[:, :rd] - _inverse_sigmoid(r.detach()), t[:, rd:]), 1).clone().requires_grad_()
            gt, gr = _grad([self._box_refine(t, r, rd)], [t, r], [f32(dy, n, 6)])
        f32(dtmp, n, 6).copy_(gt)
        if dref:
            f32(dref, n, rd).copy_(gr)
        return 0

    @staticmethod
    def _head_depth(coord, size3d, reg, wdepth, calibs, img_sizes):
        """monodetr.py:230-262"""
        h_norm = coord[:, :, 4] + coord[:, :, 5]
        box_h = torch.clamp(h_norm * img_sizes[:, 1:2], min=1.0)
        geo = size3d[:, :, 0] / box_h * calibs[:, 0, 0].unsqueeze(1)
        centre = ((coord[..., :2] - 0.5) * 2).unsqueeze(2).detach()
        dmap = F.grid_sample(wdepth.unsqueeze(1), centre, mode="bilinear", align_corners=True).squeeze(1)
        return torch.cat([((1.0 / (reg[:, :, 0:1].sigmoid() + 1e-6) - 1.0) + geo.unsqueeze(-1) + dmap) / 3, reg[:, :, 1:2]], -1)

    def mdb_head_depth_forward_f32(self, coord, size3d, reg, wdepth, calibs, img_sizes, out, B, N, H, W, stream):
        f32(out, B, N, 2).copy_(self._head_depth(f32(coord, B, N, 6), f32(size3d, B, N, 3), f32(reg, B, N, 2), f32(wdepth, B, H, W),
                                                 f32(calibs, B, 3, 4), f32(img_sizes, B, 2)))
        return 0

    def mdb_head_depth_backward_f32(self, dout, coord, size3d, reg, calibs, img_sizes, dcoord, dsize, dreg, dwd, B, N, H, W, stream):
        with torch.enable_grad():
            ins = [f32(coord, B, N, 6).clone().requires_grad_(), f32(size3d, B, N, 3).clone().requires_grad_(),
                   f32(reg, B, N, 2).clone().requires_grad_(), torch.zeros(B, H, W, requires_grad=True)]
            o = self._head_depth(*ins, f32(calibs, B, 3, 4), f32(img_sizes, B, 2))      # linear in the map: its gradient does not depend on it
            gs = _grad([o], ins, [f32(dout, B, N, 2)])
        for ptr, g, shp in ((dcoord, gs[0], (B, N, 6)), (dsize, gs[1], (B, N, 3)), (dreg, gs[2], (B, N, 2)), (dwd, gs[3], (B, H, W))):
            f32(ptr, *shp).copy_(g if g is not None else torch.zeros(shp))
        return 0

    @staticmethod
    def _depth_tail(logits, bins, emb, dmax):
        """depth_predictor.py:74-77, 93-104"""
        wd = (F.softmax(logits, -1) * bins).sum(-1)
        coord = wd.clamp(min=0, max=dmax)
        fl = coord.floor()
        delta = (coord - fl).unsqueeze(-1)
        i0 = fl.long()
        i1 = (i0 + 1).clamp(max=emb.shape[0] - 1)
        return wd, emb[i0] * (1 - delta) + emb[i1] * delta

    def mdb_depth_tail_forward_f32(self, logits, bins, emb, wdepth, ip, npix, nb, E, C, dmax, stream):
        wd, v = self._depth_tail(f32(logits, npix, nb), f32(bins, nb), f32(emb, E, C), dmax)
        f32(wdepth, npix).copy_(wd)
        f32(ip, npix, C).copy_(v)
        return 0

    def mdb_depth_tail_backward_f32(self, logits, bins, emb, d_ip, d_wd_ext, dlogits, demb, npix, nb, E, C, dmax, stream):
        with torch.enable_grad():
            lg, em = f32(logits, npix, nb).clone().requires_grad_(), f32(emb, E, C).clone().requires_grad_()
            wd, v = self._depth_tail(lg, f32(bins, nb), em, dmax)
            gwd = f32(d_wd_ext, npix) if d_wd_ext else torch.zeros(npix)
            gl, ge = _grad([wd, v], [lg, em], [gwd, f32(d_ip, npix, C)])
        f32(dlogits, npix, nb).copy_(gl)
        f32(demb, E, C).copy_(ge)
        return 0

    def mdb_depth_sample_forward_f32(self, depth, xy, out, B, H, W, N, stream):
        f32(out, B, N).copy_(F.grid_sample(f32(depth, B, H, W).unsqueeze(1), f32(xy, B, N, 2).unsqueeze(2), mode="bilinear",
                                           align_corners=True).view(B, N))
        return 0

    def mdb_depth_sample_backward_f32(self, dout, xy, ddepth, B, H, W, N, stream):
        with torch.enable_grad():
            d = torch.zeros(B, H, W, requires_grad=True)
            o = F.grid_sample(d.unsqueeze(1), f32(xy, B, N, 2).unsqueeze(2), mode="bilinear", align_corners=True).view(B, N)
            (g,) = _grad([o], [d], [f32(dout, B, N)])
        f32(ddepth, B, H, W).copy_(g)
        return 0


    # ---- the steps either side of the path (SURVEY.md 8f) -----------------------------------------------------------------------
    def mdb_adamw_step_f32(self, p, g, m, v, n, n_decay, beta1, omb1, beta2, omb2, eps, wd, step_size, step_size_dev, stream):
        """lib/helpers/optimizer_helper.py:104-127 per element; weight decay on the first n_decay elements of the flat layout."""
        P, G, M, V = f32(p, n), f32(g, n), f32(m, n), f32(v, n)
        step = float(f32(step_size_dev, 1)[0]) if step_size_dev else step_size
        M.mul_(beta1).add_(G, alpha=omb1)
        V.mul_(beta2).addcmul_(G, G, value=omb2)
        decay = torch.zeros(n)
        decay[:n_decay] = wd
        P.add_((P * decay).addcdiv_(M, V.sqrt().add_(eps), value=1), alpha=-step)
        return 0

    def mdb_extract_dets_f32(self, logits, boxes, dim3, depth, angle, B, Q, C, topk, dets, stream):
        from oracle import decode as od
        f32(dets, B, topk, 37).copy_(torch.from_numpy(od.extract_dets(
            f32(logits, B, Q, C).numpy(), f32(boxes, B, Q, 6).numpy(), f32(dim3, B, Q, 3).numpy(), f32(depth, B, Q, 2).numpy(),
            f32(angle, B, Q, 24).numpy(), topk)))
        return 0

    def mdb_decode_dets_f32(self, dets, img_size, P2, mean, B, topk, C, threshold, out, count, stream):
        from oracle import decode as od
        d = f32(dets, B, topk, 37)
        rows = od.decode_dets(d.numpy(), f32(img_size, B, 2).numpy(), f32(P2, B, 3, 4).numpy(), f32(mean, C, 3).numpy(), threshold)
        o = f32(out, B, topk, 14)
        o.zero_()
        cnt = _buf(count, B, ctypes.c_int32, torch.int32)
        for b in range(B):
            # (the kernel keeps the PREFIX of the score-sorted rows that reach the threshold; with sorted scores that is every such row)
            cnt[b] = len(rows[b])
            if rows[b]:
                o[b, :len(rows[b])] = torch.tensor(rows[b], dtype=torch.float64).float()
        return 0


class _Stream:
    cuda_stream = 0

    def __init__(self, *a, **k):
        pass

    def wait_stream(self, other):
        pass

    def wait_event(self, ev):
        pass

    def synchronize(self):
        pass


def install(monkeypatch, precision=1):
    """Route the product's host code to the fake library and give it a dummy CUDA stream API (test-scoped)."""
    from monodetr_b200 import _lib, functional, tc
    fake = FakeLib(precision)
    monkeypatch.setattr(_lib, "_lib", fake)
    # per-process caches that GPU tests run earlier in the same session fill with real CUDA streams / device buffers
    monkeypatch.setattr(functional, "_SIDE_STREAMS", {})
    monkeypatch.setattr(functional, "_BRANCH_STREAMS", {})
    monkeypatch.setattr(tc, "_WORKSPACE", {})
    stream = _Stream()
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: stream)
    monkeypatch.setattr(torch.cuda, "Stream", _Stream)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.Tensor, "record_stream", lambda self, s: None)
    return fake
