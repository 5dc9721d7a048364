"""Host-side logic of the production ResnetBlock unit (ops.ResnetBlockFn: fp16 shadows of act(GroupNorm(x)) and of the
gradients, statistics hand-over from the convolution epilogues, scale bookkeeping through dx_bound / amax scalars, cached
weight images) checked WITHOUT a GPU: ops.L.call is replaced by an emulation of the C-ABI entries' documented semantics
(include/mas_b200.h) that reads and writes the CPU tensors' memory through the pointers / mas_tensor4 strides the unit passes,
with REAL fp16 rounding of every fp16 buffer.  The result is compared with the outputs and gradients of the real reference
(tests/golden/blocks_tc.pt).  The kernels themselves are tested on the GPU (tests/test_gpu_parity.py)."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN


def _addr(v):
    if v is None:
        return 0
    if isinstance(v, torch.Tensor):
        return v.data_ptr()
    if isinstance(v, ctypes.c_void_p):
        return v.value or 0
    raise TypeError(type(v))


def _f32(p, n):
    return np.ctypeslib.as_array((ctypes.c_float * int(n)).from_address(_addr(p)))


def _f16(p, n):
    return np.ctypeslib.as_array((ctypes.c_uint16 * int(n)).from_address(_addr(p))).view(np.float16)


def _view4(p, t4, half=False):
    """[n, h, w, c] numpy view of a strided tensor described by a mas_tensor4 (element strides)."""
    dims = (t4.n, t4.h, t4.w, t4.c)
    strides = (t4.sn, t4.sh, t4.sw, t4.sc)
    extent = 1 + sum((d - 1) * s for d, s in zip(dims, strides))
    flat = _f16(p, extent) if half else _f32(p, extent)
    item = 2 if half else 4
    return np.lib.stride_tricks.as_strided(flat, dims, tuple(item * s for s in strides))


def _scale(amax):
    """tc_ptx.cuh operand_scale: 2^(14 - floor(log2 amax)), 1 for NULL / zero / non-finite."""
    if amax is None:
        return 1.0
    a = float(_f32(amax, 1)[0])
    return 1.0 if not np.isfinite(a) or a <= 0 else 2.0 ** (14 - int(np.floor(np.log2(a))))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).double()


class VqEmu:
    def __init__(self):
        self.names = []
        self.packs = {}

    def __call__(self, name, *a):
        self.names.append(name)
        getattr(self, name)(*a)

    # ---- GroupNorm -------------------------------------------------------------------------------------------------
    @staticmethod
    def _xhat(x, mean, rstd, N, HW, C, G):
        X = _f32(x, N * HW * C).reshape(N, HW, G, C // G).astype(np.float64)
        m = _f32(mean, N * G).reshape(N, 1, G, 1).astype(np.float64)
        r = _f32(rstd, N * G).reshape(N, 1, G, 1).astype(np.float64)
        return ((X - m) * r).reshape(N, HW, C), r

    def mas_gn_stats(self, x, N, HW, C, G, eps, mean, rstd, ws, ws_bytes):
        X = _f32(x, N * HW * C).reshape(N, HW, G, C // G).astype(np.float64)
        m = X.mean(axis=(1, 3))
        v = X.var(axis=(1, 3))
        _f32(mean, N * G)[...] = m.reshape(-1)
        _f32(rstd, N * G)[...] = (1.0 / np.sqrt(v + eps)).reshape(-1)

    def mas_gn_apply(self, x, mean, rstd, gamma, beta, y, N, HW, C, G, silu, mode):
        xh, _ = self._xhat(x, mean, rstd, N, HW, C, G)
        u = xh * _f32(gamma, C).astype(np.float64) + _f32(beta, C).astype(np.float64)
        a = u / (1.0 + np.exp(-u)) if silu else u
        if mode == 2:
            _f16(y, N * HW * C)[...] = a.reshape(-1).astype(np.float16)
        else:
            _f32(y, N * HW * C)[...] = a.reshape(-1)

    def mas_gn_finalize_partials(self, part, tiles_per_image, N, C, G, hw, eps, mean, rstd):
        P = _f32(part, N * tiles_per_image * 4 * (C // 4) * 2).reshape(N, tiles_per_image * 4, C // 4, 2).astype(np.float64)
        tot = P.sum(1)                                                   # [N, C/4, 2]
        per_group = tot.reshape(N, G, (C // 4) // G if C // 4 >= G else 1, 2) if (C // 4) % G == 0 else None
        assert per_group is not None, "channel quads must not straddle GroupNorm groups"
        s = per_group.sum(2)
        cnt = float(hw) * (C // G)
        m = s[..., 0] / cnt
        v = s[..., 1] / cnt - m * m
        _f32(mean, N * G)[...] = m.reshape(-1)
        _f32(rstd, N * G)[...] = (1.0 / np.sqrt(v + eps)).reshape(-1)

    def mas_gn_backward(self, dy, x, mean, rstd, gamma, beta, dx_add, dx, dgamma, dbeta, act_out, act_f16, dx_amax, add_amax, dx_f16,
                        dx_bound, N, HW, C, G, silu, ws, ws_bytes):
        xh, r = self._xhat(x, mean, rstd, N, HW, C, G)
        gm, bt = _f32(gamma, C).astype(np.float64), _f32(beta, C).astype(np.float64)
        u = xh * gm + bt
        sg = 1.0 / (1.0 + np.exp(-u))
        act = u * sg if silu else u
        dact = sg * (1.0 + u * (1.0 - sg)) if silu else np.ones_like(u)
        D = _f32(dy, N * HW * C).reshape(N, HW, C).astype(np.float64) * dact
        _f32(dgamma, C)[...] = (D * xh).sum((0, 1))
        _f32(dbeta, C)[...] = D.sum((0, 1))
        g = (D * gm).reshape(N, HW, G, C // G)
        xg = xh.reshape(N, HW, G, C // G)
        A = (g * xg).mean(axis=(1, 3), keepdims=True)
        B = g.mean(axis=(1, 3), keepdims=True)
        d = (r * (g - B - xg * A)).reshape(N, HW, C)
        if dx_add is not None:
            d = d + _f32(dx_add, N * HW * C).reshape(N, HW, C)
        if dx is not None:
            _f32(dx, N * HW * C)[...] = d.reshape(-1)
        if act_out is not None:
            (_f16 if act_f16 else _f32)(act_out, N * HW * C)[...] = act.reshape(-1).astype(np.float16 if act_f16 else np.float32)
        if dx_amax is not None:
            _f32(dx_amax, 1)[0] = np.abs(d).max()
        if dx_f16 is not None:
            assert dx_bound is not None and (dx_add is None or add_amax is not None)
            bound = 1.3 * float(np.abs(d).max()) + 1e-30          # any value >= max|dx| is a valid "rigorous bound"
            _f32(dx_bound, 1)[0] = bound
            _f16(dx_f16, N * HW * C)[...] = (d.reshape(-1) * _scale(dx_bound)).astype(np.float16)

    # ---- fp16 copies -------------------------------------------------------------------------------------------------
    def mas_amax(self, x, n, out):
        _f32(out, 1)[0] = np.abs(_f32(x, n)).max()

    def mas_to_half(self, x, y, n, amax):
        _f16(y, n)[...] = (_f32(x, n).astype(np.float64) * _scale(amax)).astype(np.float16)

    # ---- 3x3 convolution family ------------------------------------------------------------------------------------------
    def mas_pack_conv3x3_tc16(self, w, w_tc16, w_dgrad, Cout, Cin, transpose):
        W = _t(_f32(w, Cout * Cin * 9).reshape(Cout, Cin, 3, 3).astype(np.float16))        # operand rounding of the weights
        if w_dgrad is not None:
            self.packs[_addr(w_tc16)] = ("f", W)
            self.packs[_addr(w_dgrad)] = ("d", W)
        else:
            self.packs[_addr(w_tc16)] = ("d" if transpose else "f", W)

    def mas_conv3x3_fprop_tc16h(self, x16, xs, wpk, bias, residual, y, ys, stats_part, x_amax):
        kind, W = self.packs[_addr(wpk)]
        X = _t(_view4(x16, xs, half=True).astype(np.float64) / _scale(x_amax)).permute(0, 3, 1, 2)      # NCHW
        if kind == "f":
            O = F.conv2d(X, W, padding=1)
        else:                                                   # data gradient: flipped taps, channels swapped
            O = F.conv_transpose2d(X, W, padding=1)
        O = O.permute(0, 2, 3, 1).numpy()                       # NHWC
        cout = O.shape[-1]
        assert cout == ys.c and O.shape[:3] == (ys.n, ys.h, ys.w)
        if bias is not None:
            O = O + _f32(bias, cout).astype(np.float64)
        if residual is not None:
            O = O + _view4(residual, ys)
        _view4(y, ys)[...] = O
        if stats_part is not None:
            n, h, w = ys.n, ys.h, ys.w
            assert h % 16 == 0 and w % 8 == 0 and cout % 4 == 0
            T = O.reshape(n, h // 16, 4, 4, w // 8, 8, cout // 4, 4)          # [n, ty, group, 4 rows, tx, 8 cols, quad, 4 ch]
            s1 = T.sum(axis=(3, 5, 7)).transpose(0, 1, 3, 2, 4)              # [n, ty, tx, group, quad]
            s2 = (T * T).sum(axis=(3, 5, 7)).transpose(0, 1, 3, 2, 4)
            out = _f32(stats_part, n * (h // 16) * (w // 8) * 4 * (cout // 4) * 2).reshape(n, h // 16, w // 8, 4, cout // 4, 2)
            out[..., 0] = s1
            out[..., 1] = s2

    def mas_conv3x3_wgrad_tc16(self, x, flags, xs, dy, dys, dw, dbias, mode, gn_table, gn_silu, dy_amax, cout_rows, ws, ws_bytes):
        assert mode in (0, 2) and gn_table is None, "the emulation covers the stride-1 and the upsampling weight gradient"
        X = _view4(x, xs, half=bool(flags & 1)).astype(np.float64)
        if not flags & 1:
            X = X.astype(np.float16).astype(np.float64)          # fp32 activation converted unscaled by the kernel
        X = _t(X).permute(0, 3, 1, 2)
        if mode == 2:
            X = F.interpolate(X, scale_factor=2.0, mode="nearest")
        if flags & 2:
            D = _view4(dy, dys, half=True).astype(np.float64) / _scale(dy_amax)
        else:                                                    # fp32 dy, rounded to fp16 under the scale of *dy_amax by the kernel
            s = _scale(dy_amax)
            D = (_view4(dy, dys).astype(np.float64) * s).astype(np.float16).astype(np.float64) / s
        D = _t(D).permute(0, 3, 1, 2)
        cout, cin = dys.c, xs.c
        assert cout_rows == cout or (cout_rows % 128 == 0 and cout_rows > cout)     # padded rows come out zero
        # dw[co, ci, ty, tx] = sum_p dy[p, co] x[p + tap, ci]
        g = torch.nn.grad.conv2d_weight(X, (cout, cin, 3, 3), D, padding=1)
        out = np.zeros((cout_rows, cin * 9), dtype=np.float32)
        out[:cout] = g.numpy().reshape(cout, -1)
        _f32(dw, cout_rows * cin * 9)[...] = out.reshape(-1)
        if dbias is not None:
            ob = np.zeros(cout_rows, dtype=np.float32)
            ob[:cout] = D.sum((0, 2, 3)).numpy()
            _f32(dbias, cout_rows)[...] = ob

    def mas_conv3x3_fprop_tc16(self, x, xs, wpk, bias, residual, y, ys, mode, table, silu, stats_part, x_amax):
        """Register-staged form: fp32 (strided) input rounded to fp16 under the scale of *x_amax by the kernel; modes S1 (0),
        UP (2: nearest x2 upsample first), ZS (3: the data gradient of the stride-2 Downsample convolution)."""
        assert table is None and stats_part is None, "the emulation covers the plain launches of the Up/Downsample layers"
        kind, W = self.packs[_addr(wpk)]
        s = _scale(x_amax)
        X = _t((_view4(x, xs).astype(np.float64) * s).astype(np.float16).astype(np.float64) / s).permute(0, 3, 1, 2)
        if mode == 2:
            assert kind == "f"
            O = F.conv2d(F.interpolate(X, scale_factor=2.0, mode="nearest"), W, padding=1)           # modules.py:55-59
        elif mode == 3:
            assert kind == "d"                                  # pad(0,1,0,1) + stride 2 (modules.py:74-78), transposed
            O = F.conv_transpose2d(X, W, stride=2)[:, :, :2 * xs.h, :2 * xs.w]
        else:
            O = F.conv2d(X, W, padding=1) if kind == "f" else F.conv_transpose2d(X, W, padding=1)
        O = O.permute(0, 2, 3, 1).numpy()
        rows = O.shape[-1]                                       # weights / bias packed for round_up(Cout, 128) rows,
        assert O.shape[:3] == (ys.n, ys.h, ys.w) and rows >= ys.c and (rows == ys.c or rows % 128 == 0)   # only ys.c channels are stored
        if bias is not None:
            O = O + _f32(bias, rows).astype(np.float64)
        O = O[..., :ys.c]
        if residual is not None:
            O = O + _view4(residual, ys)
        _view4(y, ys)[...] = O

    def mas_sumpool2x2(self, x, y, N, H, W, C):
        X = _f32(x, N * 4 * H * W * C).reshape(N, H, 2, W, 2, C).astype(np.float64)
        _f32(y, N * H * W * C)[...] = X.sum(axis=(2, 4)).reshape(-1)

    def mas_space_to_depth(self, x, y, N, H, W, C):
        X = _f32(x, N * H * W * C).reshape(N, H // 2, 2, W // 2, 2, C)                      # [n, i, py, j, px, c]
        _f32(y, N * H * W * C)[...] = X.transpose(0, 1, 3, 2, 4, 5).reshape(-1)           # [n, i, j, (py, px, c)]

    def mas_s2d_pack_weights(self, w, w9, Cout, C):
        Wm = _f32(w, Cout * C * 9).reshape(Cout, C, 3, 3)
        out = np.zeros((Cout, 4, C, 3, 3), dtype=np.float32)
        for py in range(2):
            for px in range(2):
                for a in range(2):
                    for b in range(2):
                        ty, tx = 2 * a + py, 2 * b + px
                        if ty <= 2 and tx <= 2:
                            out[:, py * 2 + px, :, a + 1, b + 1] = Wm[:, :, ty, tx]
        _f32(w9, Cout * 4 * C * 9)[...] = out.reshape(-1)

    def mas_s2d_unpack_wgrad(self, dw9, dw, Cout, C):
        D9 = _f32(dw9, Cout * 4 * C * 9).reshape(Cout, 4, C, 3, 3)
        out = np.zeros((Cout, C, 3, 3), dtype=np.float32)
        for ty in range(3):
            for tx in range(3):
                out[:, :, ty, tx] = D9[:, (ty & 1) * 2 + (tx & 1), :, (ty >> 1) + 1, (tx >> 1) + 1]
        _f32(dw, Cout * C * 9)[...] = out.reshape(-1)

    # ---- 1x1 (shortcut) ----------------------------------------------------------------------------------------------------
    def mas_pack_gemm_tc(self, w, w_tc, N, K, transpose):
        W = _f32(w, N * K).reshape(N, K).astype(np.float64)
        self.packs[_addr(w_tc)] = ("g", W.T.copy() if transpose else W)

    def mas_gemm_rows_packed(self, A, lda, w_tc, C, ldc, M, N, K, alpha, bias, residual, stats_part):
        assert stats_part is None
        _, W = self.packs[_addr(w_tc)]
        assert W.shape == (N, K)
        Am = np.lib.stride_tricks.as_strided(_f32(A, (M - 1) * lda + K), (M, K), (4 * lda, 4)).astype(np.float64)
        o = alpha * (Am @ W.T)
        if bias is not None:
            o = o + _f32(bias, N)
        if residual is not None:
            o = o + np.lib.stride_tricks.as_strided(_f32(residual, (M - 1) * ldc + N), (M, N), (4 * ldc, 4))
        np.lib.stride_tricks.as_strided(_f32(C, (M - 1) * ldc + N), (M, N), (4 * ldc, 4))[...] = o

    def mas_conv1x1_wgrad(self, x, ldx, dy, ldy, M, cin, cout, dw, db, impl, ws, ws_bytes):
        X = np.lib.stride_tricks.as_strided(_f32(x, (M - 1) * ldx + cin), (M, cin), (4 * ldx, 4)).astype(np.float64)
        D = np.lib.stride_tricks.as_strided(_f32(dy, (M - 1) * ldy + cout), (M, cout), (4 * ldy, 4)).astype(np.float64)
        _f32(dw, cout * cin).reshape(cout, cin)[...] = D.T @ X
        if db is not None:
            _f32(db, cout)[...] = D.sum(0)

    # ---- AttnBlock as one call per direction (modules.py:139-191) --------------------------------------------------------
    @staticmethod
    def _attn_math(X, mean, rstd, nw, nb, qw, qb, kw, kb, vw, vb, pw, pb, N, HW, C, G):
        """fp64 torch graph of the block on X [N,HW,C] with the statistics given; returns (hn, qkv, P, O, out)."""
        xh = ((X.view(N, HW, G, C // G) - mean.view(N, 1, G, 1)) * rstd.view(N, 1, G, 1)).view(N, HW, C)
        hn = xh * nw + nb
        q, k, v = hn @ qw.t() + qb, hn @ kw.t() + kb, hn @ vw.t() + vb
        P = torch.softmax((q @ k.transpose(1, 2)) * float(C) ** -0.5, dim=-1)          # softmax over keys, modules.py:180-181
        O = P @ v
        return hn, torch.cat([q, k, v], -1), P, O, O @ pw.t() + pb + X

    def mas_attnblock_forward(self, x, N, HW, C, G, mean, rstd, nw, nb, qw, qb, kw, kb, vw, vb, pw, pb, hn, qkv, P, O, out, stats_part, impl,
                              ws, ws_bytes):
        g = lambda p, n: _t(_f32(p, n))
        z = lambda p: g(p, C) if p is not None else torch.zeros(C, dtype=torch.float64)
        X = g(x, N * HW * C).view(N, HW, C)
        r = self._attn_math(X, g(mean, N * G), g(rstd, N * G), g(nw, C), g(nb, C), g(qw, C * C).view(C, C), z(qb), g(kw, C * C).view(C, C), z(kb),
                            g(vw, C * C).view(C, C), z(vb), g(pw, C * C).view(C, C), z(pb), N, HW, C, G)
        for dst, val, n in ((hn, r[0], N * HW * C), (qkv, r[1], N * HW * 3 * C), (P, r[2], N * HW * HW), (O, r[3], N * HW * C), (out, r[4], N * HW * C)):
            _f32(dst, n)[...] = val.reshape(-1).numpy()
        if stats_part is not None:                               # 128-row tiles of the [N*HW, C] output: [tile][4 x 32 rows][C/4][sum, sumsq]
            T = r[4].reshape(N * HW // 128, 4, 32, C // 4, 4).numpy()
            sp = _f32(stats_part, (N * HW // 128) * 4 * (C // 4) * 2).reshape(N * HW // 128, 4, C // 4, 2)
            sp[..., 0] = T.sum(axis=(2, 4))
            sp[..., 1] = (T * T).sum(axis=(2, 4))

    def mas_attnblock_backward(self, dout, x, N, HW, C, G, mean, rstd, nw, nb, qw, kw, vw, pw, hn, qkv, P, O, dx, dnw, dnb, dqkv_w, dqkv_b, dpw,
                               dpb, dx_amax, impl, ws, ws_bytes):
        """Like the kernels, from the SAVED forward tensors (hn, qkv, P, O): the backward entry is not given the biases."""
        g = lambda p, n: _t(_f32(p, n))
        D = g(dout, N * HW * C).view(N, HW, C)
        Wp, Wcat = g(pw, C * C).view(C, C), torch.cat([g(qw, C * C).view(C, C), g(kw, C * C).view(C, C), g(vw, C * C).view(C, C)], 0)
        QKV = g(qkv, N * HW * 3 * C).view(N, HW, 3 * C)
        with torch.enable_grad():                                         # (autograd is off inside a Function's backward)
            Q, K, V = [t.clone().requires_grad_(True) for t in QKV.split(C, dim=-1)]
            Pm = torch.softmax((Q @ K.transpose(1, 2)) * float(C) ** -0.5, dim=-1)
            Om = Pm @ V
        # the tensors the unit saved in the forward pass are the ones it hands back
        assert torch.allclose(Pm.detach().reshape(-1), g(P, N * HW * HW), atol=1e-5) and torch.allclose(Om.detach().reshape(-1), g(O, N * HW * C), atol=1e-4)
        dO = D @ Wp                                                        # out = O Wp^T + bp + x
        Om.backward(dO)
        _f32(dpw, C * C)[...] = (D.reshape(-1, C).t() @ Om.detach().reshape(-1, C)).reshape(-1).numpy()
        _f32(dpb, C)[...] = D.sum((0, 1)).numpy()
        dqkv = torch.cat([Q.grad, K.grad, V.grad], -1).reshape(-1, 3 * C)
        H = g(hn, N * HW * C).view(-1, C)
        _f32(dqkv_w, 3 * C * C)[...] = (dqkv.t() @ H).reshape(-1).numpy()
        _f32(dqkv_b, 3 * C)[...] = dqkv.sum(0).numpy()
        dhn = (dqkv @ Wcat).view(N, HW, C)
        # GroupNorm (no activation) backward + the residual branch
        X = g(x, N * HW * C).view(N, HW, G, C // G)
        m, r = g(mean, N * G).view(N, 1, G, 1), g(rstd, N * G).view(N, 1, G, 1)
        xh = ((X - m) * r)
        assert torch.allclose((xh.reshape(N, HW, C) * g(nw, C) + g(nb, C)).reshape(-1), H.reshape(-1), atol=1e-4)      # saved hn = GN(x)
        _f32(dnw, C)[...] = (dhn * xh.reshape(N, HW, C)).sum((0, 1)).numpy()
        _f32(dnb, C)[...] = dhn.sum((0, 1)).numpy()
        gg = (dhn * g(nw, C)).view(N, HW, G, C // G)
        A = (gg * xh).mean(dim=(1, 3), keepdim=True)
        Bm = gg.mean(dim=(1, 3), keepdim=True)
        d = (r * (gg - Bm - xh * A)).reshape(N, HW, C) + D
        _f32(dx, N * HW * C)[...] = d.reshape(-1).numpy()
        if dx_amax is not None:
            _f32(dx_amax, 1)[0] = float(d.abs().max())

    # ---- general-shape fp32 convolution family (the SIMT entries: exact fp32, explicit strides) --------------------------
    def mas_pack_conv3x3(self, w, wp, Cout, Cin, flip_transpose, rtf32):
        self.packs[_addr(wp)] = ("d" if flip_transpose else "f", _t(_f32(w, Cout * Cin * 9).reshape(Cout, Cin, 3, 3)))

    @staticmethod
    def _conv_mode(X, W, kind, mode, out_hw):
        if kind == "f":
            if mode == 0:
                return F.conv2d(X, W, padding=1)
            if mode == 1:                                     # Downsample: pad (0,1,0,1), stride 2, no padding (modules.py:74-78)
                return F.conv2d(F.pad(X, (0, 1, 0, 1)), W, stride=2)
            if mode == 2:                                     # Upsample: nearest x2 first (modules.py:55-59)
                return F.conv2d(F.interpolate(X, scale_factor=2.0, mode="nearest"), W, padding=1)
        else:
            if mode == 0:
                return F.conv_transpose2d(X, W, padding=1)
            if mode == 3:                                     # data gradient of the stride-2 convolution
                return F.conv_transpose2d(X, W, stride=2)[:, :, :out_hw[0], :out_hw[1]]
        raise AssertionError(("conv mode", kind, mode))

    def mas_conv3x3_fprop(self, x, xs, wp, bias, residual, y, ys, mode, impl):
        kind, W = self.packs[_addr(wp)]
        O = self._conv_mode(_t(_view4(x, xs)).permute(0, 3, 1, 2), W, kind, mode, (ys.h, ys.w)).permute(0, 2, 3, 1).numpy()
        assert O.shape == (ys.n, ys.h, ys.w, ys.c), (O.shape, (ys.n, ys.h, ys.w, ys.c))
        if bias is not None:
            O = O + _f32(bias, ys.c).astype(np.float64)
        if residual is not None:
            O = O + _view4(residual, ys)
        _view4(y, ys)[...] = O

    def mas_conv3x3_wgrad(self, x, xs, dy, dys, dw, dbias, mode, impl, gn_table, gn_silu, ws, ws_bytes):
        assert gn_table is None
        X = _t(_view4(x, xs)).permute(0, 3, 1, 2)
        D = _t(_view4(dy, dys)).permute(0, 3, 1, 2)
        cout, cin = dys.c, xs.c
        if mode == 1:
            g = torch.nn.grad.conv2d_weight(F.pad(X, (0, 1, 0, 1)), (cout, cin, 3, 3), D, stride=2)
        elif mode == 2:
            g = torch.nn.grad.conv2d_weight(F.interpolate(X, scale_factor=2.0, mode="nearest"), (cout, cin, 3, 3), D, padding=1)
        else:
            assert mode == 0
            g = torch.nn.grad.conv2d_weight(X, (cout, cin, 3, 3), D, padding=1)
        _f32(dw, cout * cin * 9)[...] = g.numpy().reshape(-1)
        if dbias is not None:
            _f32(dbias, cout)[...] = D.sum((0, 2, 3)).numpy()

    # ---- 3-channel edge layers (conv_in / conv_out, modules.py:219,364) ------------------------------------------------------
    def mas_edge_small_cin_fprop(self, x, xt, w, bias, y, yt, flip_transpose):
        X = _t(_view4(x, xt)).permute(0, 3, 1, 2)
        if flip_transpose:                                    # conv_out's data gradient: w is its [3, C, 3, 3] weight
            O = F.conv_transpose2d(X, _t(_f32(w, 3 * yt.c * 9).reshape(3, yt.c, 3, 3)), padding=1)
        else:
            O = F.conv2d(X, _t(_f32(w, yt.c * 3 * 9).reshape(yt.c, 3, 3, 3)), padding=1)
        O = O.permute(0, 2, 3, 1).numpy()
        if bias is not None:
            O = O + _f32(bias, yt.c).astype(np.float64)
        _view4(y, yt)[...] = O

    def mas_edge_small_cout_fprop(self, x, xt, w, bias, y, yt):
        O = F.conv2d(_t(_view4(x, xt)).permute(0, 3, 1, 2), _t(_f32(w, 3 * xt.c * 9).reshape(3, xt.c, 3, 3)), padding=1).permute(0, 2, 3, 1).numpy()
        if bias is not None:
            O = O + _f32(bias, 3).astype(np.float64)
        _view4(y, yt)[...] = O

    def _edge_wgrad(self, x, xt, dy, dyt, dw, db):
        X = _t(_view4(x, xt)).permute(0, 3, 1, 2)
        D = _t(_view4(dy, dyt)).permute(0, 3, 1, 2)
        g = torch.nn.grad.conv2d_weight(X, (dyt.c, xt.c, 3, 3), D, padding=1)
        _f32(dw, dyt.c * xt.c * 9)[...] = g.numpy().reshape(-1)
        if db is not None:
            _f32(db, dyt.c)[...] = D.sum((0, 2, 3)).numpy()

    def mas_edge_small_cin_wgrad(self, x, xt, dy, dyt, dw, db, ws, ws_bytes):
        self._edge_wgrad(x, xt, dy, dyt, dw, db)

    def mas_edge_small_cout_wgrad(self, a, at, dy, dyt, dw, db, ws, ws_bytes):
        self._edge_wgrad(a, at, dy, dyt, dw, db)

    # ---- fp32 GEMM (1x1 convolutions off the tensor tiles) ------------------------------------------------------------------------
    def mas_gemm(self, A, B, C, M, N, K, batch, lda, ldb, ldc, sa, sb, sc, ta, tb, alpha, bias, residual, impl):
        def mat(p, rows, cols, ld, trans):
            if not trans:
                return np.lib.stride_tricks.as_strided(_f32(p, (rows - 1) * ld + cols), (rows, cols), (4 * ld, 4))
            return np.lib.stride_tricks.as_strided(_f32(p, (cols - 1) * ld + rows), (rows, cols), (4, 4 * ld))
        for i in range(batch):
            Am = mat(ctypes.c_void_p(_addr(A) + 4 * i * sa), M, K, lda, bool(ta)).astype(np.float64)
            Bm = mat(ctypes.c_void_p(_addr(B) + 4 * i * sb), N, K, ldb, not bool(tb)).astype(np.float64)
            o = alpha * (Am @ Bm.T)
            if bias is not None:
                o = o + _f32(bias, N)[None, :]
            if residual is not None:
                o = o + mat(ctypes.c_void_p(_addr(residual) + 4 * i * sc), M, N, ldc, False)
            mat(ctypes.c_void_p(_addr(C) + 4 * i * sc), M, N, ldc, False)[...] = o

    # ---- (Sync)BatchNorm of quant_conv, vqvae.py:16 ------------------------------------------------------------------------------
    @staticmethod
    def _f64(p, n):
        return np.ctypeslib.as_array((ctypes.c_double * int(n)).from_address(_addr(p)))

    def mas_bn_stats(self, x, R, C, out):
        X = _f32(x, R * C).reshape(R, C).astype(np.float64)
        o = self._f64(out, 2 * C + 1)
        o[:C], o[C:2 * C], o[2 * C] = X.sum(0), (X * X).sum(0), R

    def mas_bn_finalize(self, stats, count, C, eps, momentum, mean, invstd, running_mean, running_var):
        st = self._f64(stats, 2 * C + 1)
        cnt = count if count > 0 else st[2 * C]
        m = st[:C] / cnt
        v = st[C:2 * C] / cnt - m * m                                   # biased, what the normalisation uses
        _f32(mean, C)[...] = m
        _f32(invstd, C)[...] = 1.0 / np.sqrt(v + eps)
        if running_mean is not None:
            rm = _f32(running_mean, C)
            rm[...] = (1 - momentum) * rm + momentum * m
        if running_var is not None:
            rv = _f32(running_var, C)
            rv[...] = (1 - momentum) * rv + momentum * v * cnt / (cnt - 1)      # unbiased, like nn.(Sync)BatchNorm

    def mas_bn_invstd(self, running_var, eps, invstd, C):
        _f32(invstd, C)[...] = 1.0 / np.sqrt(_f32(running_var, C).astype(np.float64) + eps)

    def mas_bn_apply(self, x, mean, invstd, gamma, beta, y, R, C):
        X = _f32(x, R * C).reshape(R, C).astype(np.float64)
        _f32(y, R * C)[...] = ((X - _f32(mean, C)) * _f32(invstd, C) * _f32(gamma, C) + _f32(beta, C)).reshape(-1)

    def mas_bn_backward_reduce(self, dy, x, mean, invstd, R, C, out):
        D = _f32(dy, R * C).reshape(R, C).astype(np.float64)
        xh = (_f32(x, R * C).reshape(R, C).astype(np.float64) - _f32(mean, C)) * _f32(invstd, C)
        o = self._f64(out, 2 * C + 1)
        o[:C], o[C:2 * C], o[2 * C] = D.sum(0), (D * xh).sum(0), R

    def mas_bn_backward_apply(self, dy, x, mean, invstd, gamma, sums_global, sums_local, inv_count, dx, dgamma, dbeta, R, C):
        D = _f32(dy, R * C).reshape(R, C).astype(np.float64)
        xh = (_f32(x, R * C).reshape(R, C).astype(np.float64) - _f32(mean, C)) * _f32(invstd, C)
        sg, sl = self._f64(sums_global, 2 * C + 1), self._f64(sums_local, 2 * C + 1)
        ic = inv_count if inv_count > 0 else 1.0 / sg[2 * C]
        _f32(dx, R * C)[...] = (_f32(gamma, C) * _f32(invstd, C) * (D - sg[:C] * ic - xh * sg[C:2 * C] * ic)).reshape(-1)
        _f32(dgamma, C)[...] = sl[C:2 * C]
        _f32(dbeta, C)[...] = sl[:C]

    # ---- Codebook, modules.py:501-517 ------------------------------------------------------------------------------------------
    def mas_vq_forward(self, z, E, R, K, D, beta, idx_out, zq_out, loss_out, ws, ws_bytes):
        Z = torch.from_numpy(_f32(z, R * D).reshape(R, D).copy())
        Em = torch.from_numpy(_f32(E, K * D).reshape(K, D).copy())
        # the reference's fp32 association and first-index tie-break (modules.py:501-505)
        d = torch.sum(Z ** 2, dim=1, keepdim=True) + torch.sum(Em ** 2, dim=1) - 2 * torch.matmul(Z, Em.t())
        idx = torch.argmin(d, dim=1)
        np.ctypeslib.as_array((ctypes.c_int64 * R).from_address(_addr(idx_out)))[...] = idx.numpy()
        zq = Em[idx].double()
        _f32(zq_out, R * D)[...] = zq.reshape(-1).numpy()
        _f32(loss_out, 1)[0] = float((1 + beta) * ((zq - Z.double()) ** 2).mean())

    def mas_vq_forward_given(self, z, E, idx_in, R, K, D, beta, zq_out, loss_out, ws, ws_bytes):
        Z = _f32(z, R * D).reshape(R, D).astype(np.float64)
        Em = _f32(E, K * D).reshape(K, D).astype(np.float64)
        ix = np.ctypeslib.as_array((ctypes.c_int64 * R).from_address(_addr(idx_in)))
        _f32(zq_out, R * D)[...] = Em[ix].reshape(-1)
        _f32(loss_out, 1)[0] = (1 + beta) * ((Em[ix] - Z) ** 2).mean()

    def mas_vq_gather(self, E, idx, R, K, D, out):
        ix = np.ctypeslib.as_array((ctypes.c_int64 * R).from_address(_addr(idx)))
        _f32(out, R * D)[...] = _f32(E, K * D).reshape(K, D)[ix].reshape(-1)

    def mas_kmeans_update(self, x, idx, n, K, D, centres_old, centres_new, shift_out, ws, ws_bytes):
        X = _f32(x, n * D).reshape(n, D).astype(np.float64)
        ix = np.ctypeslib.as_array((ctypes.c_int64 * n).from_address(_addr(idx)))
        old = _f32(centres_old, K * D).reshape(K, D).astype(np.float64)
        new = old.copy()                                          # an empty cluster keeps its centre
        cnt = np.bincount(ix, minlength=K)
        sums = np.zeros((K, D))
        np.add.at(sums, ix, X)
        new[cnt > 0] = sums[cnt > 0] / cnt[cnt > 0, None]
        _f32(centres_new, K * D)[...] = new.reshape(-1)
        if shift_out is not None:
            _f32(shift_out, 1)[0] = np.sqrt(((new - old) ** 2).sum())

    def mas_vq_backward(self, g_zq, g_loss, z, E, idx, R, K, D, beta, grad_z, grad_E):
        Z = _f32(z, R * D).reshape(R, D).astype(np.float64)
        Em = _f32(E, K * D).reshape(K, D).astype(np.float64)
        ix = np.ctypeslib.as_array((ctypes.c_int64 * R).from_address(_addr(idx)))
        gl = float(_f32(g_loss, 1)[0]) if g_loss is not None else 0.0
        if grad_z is not None:
            gz = gl * (2.0 / (R * D)) * (Z - Em[ix])
            if g_zq is not None:
                gz = gz + _f32(g_zq, R * D).reshape(R, D)
            _f32(grad_z, R * D)[...] = gz.reshape(-1)
        if grad_E is not None:                                   # zeroed by the caller, accumulated here
            ge = _f32(grad_E, K * D).reshape(K, D)
            np.add.at(ge, ix, (gl * (2.0 * beta / (R * D)) * (Em[ix] - Z)).astype(np.float32))

    def mas_nchw_to_nhwc_pad(self, x, y, N, C, CP, H, W):
        out = np.zeros((N, H, W, CP), dtype=np.float32)
        out[..., :C] = _f32(x, N * C * H * W).reshape(N, C, H, W).transpose(0, 2, 3, 1)
        _f32(y, N * H * W * CP)[...] = out.reshape(-1)

    # ---- weighted BCE-with-logits of the VQ-SEG step, losses/loss_seg.py:15-22 ---------------------------------------------
    @staticmethod
    def _bce_views(logits, target, N, C, CP, H, W):
        X = _f32(logits, N * H * W * CP).reshape(N, H, W, CP)[..., :C].astype(np.float64)            # channels-last, pitch CP
        T = _f32(target, N * C * H * W).reshape(N, C, H, W).transpose(0, 2, 3, 1).astype(np.float64)    # NCHW target
        return X, T

    def mas_bce_cl_forward(self, logits, target, pos_weight, N, C, CP, H, W, loss_out, ws, ws_bytes):
        X, T = self._bce_views(logits, target, N, C, CP, H, W)
        pw = _f32(pos_weight, C).astype(np.float64)
        ls = -np.logaddexp(0.0, -X)                               # log sigmoid(x)
        l1 = -np.logaddexp(0.0, X)                                # log (1 - sigmoid(x))
        _f32(loss_out, 1)[0] = (-(pw * T * ls + (1 - T) * l1)).mean()

    def mas_bce_cl_backward(self, logits, target, pos_weight, g, N, C, CP, H, W, grad):
        X, T = self._bce_views(logits, target, N, C, CP, H, W)
        pw = _f32(pos_weight, C).astype(np.float64)
        sg = 1.0 / (1.0 + np.exp(-X))
        gg = float(_f32(g, 1)[0]) if g is not None else 1.0
        out = np.zeros((N, H, W, CP), dtype=np.float32)           # pad channels written as zeros
        out[..., :C] = gg * (-(pw * T * (1 - sg)) + (1 - T) * sg) / (N * C * H * W)
        _f32(grad, N * H * W * CP)[...] = out.reshape(-1)

    def mas_copy_strided(self, x, xs, y, ys):
        _view4(y, ys)[...] = _view4(x, xs)


@pytest.fixture
def vq_emu(monkeypatch):
    from mas_b200 import ops
    e = VqEmu()
    monkeypatch.setattr(ops.L, "call", e)
    def dense(t):
        return t.sc == 1 and t.sw == t.c and t.sh == t.w * t.c and t.sn == t.h * t.w * t.c

    def query(name, *a):
        if name == "mas_conv3x3_tc_eligible":        # include/mas_b200.h: dense NHWC, Cin % 8, Cout % 128, Hout % 16, Wout % 8, S1 / UP / ZS
            xs, ys, mode = a
            return int(dense(xs) and dense(ys) and xs.c % 8 == 0 and ys.c % 128 == 0 and ys.h % 16 == 0 and ys.w % 8 == 0 and mode in (0, 2, 3))
        if name == "mas_conv3x3_wgrad_tc_eligible":  # dense NHWC, Cin % 32, Cout % 128, H, W % 8, S1 / UP
            xs, dys, mode = a
            return int(dense(xs) and dense(dys) and xs.c % 32 == 0 and dys.c % 128 == 0 and dys.h % 8 == 0 and dys.w % 8 == 0 and mode in (0, 2))
        return 1 << 20                                # workspace sizes
    monkeypatch.setattr(ops.L, "query", query)
    monkeypatch.setattr(ops, "_need_cuda", lambda x: None)
    monkeypatch.setattr(ops, "_tc_on", lambda: True)
    ops._packs.clear()
    return e


def _sampled_err(t, fx, norm):
    smp, stride = fx
    got = t.detach().reshape(-1)[::stride].double()
    scale = norm * (smp.numel() / t.numel()) ** 0.5
    return float((got - smp.double()).norm() / max(scale, 1e-30))


@pytest.mark.parametrize("name", ["res_128_128", "res_128_256", "res_512_512"])
def test_resnet_block_unit_host_logic_against_reference_fixture(vq_emu, name):
    """The production ResnetBlock unit (shadow mode) above the emulated C-ABI reproduces the REAL reference's output, input
    gradient and every parameter gradient within the GPU test's tolerances - and takes the route it is meant to take."""
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from models import modules as M
    from oracle.seeded import assert_same_fill, fill_seeded, seeded_input
    from test_oracle import build_tc_block
    b = torch.load(os.path.join(GOLDEN, "blocks_tc.pt"), weights_only=False)[name]
    mod = build_tc_block(name, M)
    assert_same_fill(fill_seeded(mod, b["seed_w"]), b["param_checks"])
    x = seeded_input(b["shape"], b["seed_x"], 1.5, 0.3).requires_grad_(True)
    y = mod(x)
    assert _sampled_err(y, b["y"], b["y_norm"]) < 1e-3, name
    (y * torch.linspace(-1, 1, y.numel()).view(y.shape)).sum().backward()     # the weighting the fixture's gradients were taken with
    assert _sampled_err(x.grad, b["grad_x"], b["grad_x_norm"]) < 3e-3, name
    named = dict(mod.named_parameters())
    for k, gv in b["grads"].items():
        g = named[k].grad
        e = _sampled_err(g, gv, b["grad_norms"][k]) if isinstance(gv, tuple) else float((g.double() - gv.double()).norm() / gv.double().norm())
        assert e < 3e-3, (name, k, e)
    n = vq_emu.names
    # the route: both convolutions and both data gradients on the shadow-fed kernel, act(GN(x)) written once per norm as fp16,
    # statistics of the second norm from conv1's epilogue (one mas_gn_stats for the block input only), weights packed once
    assert n.count("mas_conv3x3_fprop_tc16h") == 4 and n.count("mas_conv3x3_wgrad_tc16") == 2
    assert n.count("mas_gn_apply") == 2 and n.count("mas_gn_stats") == 1 and n.count("mas_gn_finalize_partials") == 2
    assert n.count("mas_pack_conv3x3_tc16") == 2 and n.count("mas_gn_backward") == 2


@pytest.mark.parametrize("name", ["attn_512", "attn_res_512", "res_res_attn_512"])
def test_block_chains_host_logic_against_reference_fixture(vq_emu, name):
    """AttnBlock and the chains that hand GroupNorm statistics (take_stats) and gradient shadows from one unit to the next,
    above the emulated C-ABI, against the REAL reference (tests/golden/blocks_tc.pt)."""
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from models import modules as M
    from oracle.seeded import assert_same_fill, fill_seeded, seeded_input
    from test_oracle import build_tc_block
    b = torch.load(os.path.join(GOLDEN, "blocks_tc.pt"), weights_only=False)[name]
    mod = build_tc_block(name, M)
    assert_same_fill(fill_seeded(mod, b["seed_w"]), b["param_checks"])
    x = seeded_input(b["shape"], b["seed_x"], 1.5, 0.3).requires_grad_(True)
    y = mod(x)
    assert _sampled_err(y, b["y"], b["y_norm"]) < 1e-3, name
    (y * torch.linspace(-1, 1, y.numel()).view(y.shape)).sum().backward()
    assert _sampled_err(x.grad, b["grad_x"], b["grad_x_norm"]) < 3e-3, name
    named = dict(mod.named_parameters())
    for k, gv in b["grads"].items():
        if k.endswith("k.bias"):
            continue          # exactly zero in exact arithmetic (softmax over keys is invariant to a per-query constant)
        g = named[k].grad
        e = _sampled_err(g, gv, b["grad_norms"][k]) if isinstance(gv, tuple) else float((g.double() - gv.double()).norm() / gv.double().norm())
        assert e < 3e-3, (name, k, e)
    n = vq_emu.names
    # one statistics pass for the chain's input only: every later GroupNorm takes its statistics from a producer's epilogue
    assert n.count("mas_gn_stats") == 1, n.count("mas_gn_stats")
    assert n.count("mas_attnblock_forward") == 1 and n.count("mas_attnblock_backward") == 1


@pytest.mark.parametrize("name", ["up_128", "up_512", "down_128"])
def test_up_down_sample_host_logic_against_reference_fixture(vq_emu, name):
    """Upsample (nearest x2 folded into the convolution; data gradient = transposed convolution + 2x2 sum pool) and Downsample
    (stride 2 through space-to-depth; data gradient on the zero-stuffed map) above the emulated C-ABI, against the REAL reference."""
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from models import modules as M
    from oracle.seeded import assert_same_fill, fill_seeded, seeded_input
    from test_oracle import build_tc_block
    b = torch.load(os.path.join(GOLDEN, "blocks_tc.pt"), weights_only=False)[name]
    mod = build_tc_block(name, M)
    assert_same_fill(fill_seeded(mod, b["seed_w"]), b["param_checks"])
    # channels-last input, as inside the model (a caller's NCHW tensor would take the general-shape fp32 kernels instead)
    x = seeded_input(b["shape"], b["seed_x"], 1.5, 0.3).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = mod(x)
    assert _sampled_err(y.contiguous(), b["y"], b["y_norm"]) < 1e-3, name
    (y * torch.linspace(-1, 1, y.numel()).view(y.shape)).sum().backward()
    assert _sampled_err(x.grad.contiguous(), b["grad_x"], b["grad_x_norm"]) < 3e-3, name
    named = dict(mod.named_parameters())
    for k, gv in b["grads"].items():
        g = named[k].grad
        e = _sampled_err(g, gv, b["grad_norms"][k]) if isinstance(gv, tuple) else float((g.double() - gv.double()).norm() / gv.double().norm())
        assert e < 3e-3, (name, k, e)
    n = vq_emu.names
    assert "mas_conv3x3_fprop_tc16" in n and "mas_conv3x3_fprop" not in n          # the tensor-core route
    if name.startswith("down"):
        assert n.count("mas_space_to_depth") == 1 and n.count("mas_s2d_pack_weights") == 1 and n.count("mas_s2d_unpack_wgrad") == 1
    else:
        assert n.count("mas_sumpool2x2") == 1


def test_whole_model_host_logic_against_reference_fixture(vq_emu):
    """The whole drop-in VQBASE (Encoder -> quant_conv + BatchNorm -> Codebook -> post_quant_conv -> Decoder, proxy loss,
    backward) above the emulated C-ABI reproduces the REAL reference on tests/golden/vqbase_tiny.pt: reconstruction, codebook
    loss, code indices bit for bit, every parameter gradient, the BatchNorm running statistics."""
    from models import VQBASE
    g = torch.load(os.path.join(GOLDEN, "vqbase_tiny.pt"), weights_only=False)
    m = VQBASE(g["ddconfig"], g["n_embed"], g["embed_dim"], 10, 100)
    m.load_state_dict(g["state_dict"])
    m.quantize.q_counter = 10 ** 6
    m.train()
    x = g["x"]
    seen = {}
    hook = m.quantize.register_forward_hook(lambda _m, _i, o: seen.__setitem__("idx", o[2].detach().clone()))
    dec, diff = m(x)
    hook.remove()
    from conftest import rel_err as rel          # quantities that are zero in exact arithmetic (a conv bias in front of a one-channel-per-group GroupNorm) compare on an absolute scale
    assert dec.shape == g["dec"].shape and dec.is_contiguous() and diff.dim() == 0
    assert torch.equal(seen["idx"].view(-1), g["idx"].view(-1))
    assert rel(dec, g["dec"]) < 1e-5 and abs(float(diff.detach()) - float(g["diff"])) < 1e-5 * abs(float(g["diff"]))
    ((x - dec).abs().mean() + diff).backward()
    named = dict(m.named_parameters())
    for k, gv in g["grads"].items():
        assert named[k].grad is not None, k
        tol = 1e-4 if float(gv.double().norm()) > 1e-4 * gv.numel() ** 0.5 else 2e-3      # noise-level gradients: the GPU test's bound
        assert rel(named[k].grad, gv) < tol, (k, rel(named[k].grad, gv))
    assert rel(m.quant_conv[1].running_mean, g["running_mean"]) < 1e-5 and rel(m.quant_conv[1].running_var, g["running_var"]) < 1e-5
    assert int(m.quant_conv[1].num_batches_tracked) == 1
    n = vq_emu.names
    assert n.count("mas_vq_forward") == 1 and n.count("mas_vq_backward") == 1 and n.count("mas_bn_stats") == 1


def test_img_config_model_host_logic_against_reference_fixture(vq_emu):
    """The 95M-parameter img_config model (the benchmark's model) at 2 x 3 x 64 x 64 above the emulated C-ABI: every tensor-path
    ResnetBlock in shadow mode, AttnBlocks, Up / Downsample on the tensor route, the small-extent levels on the general-shape
    entries, BatchNorm, codebook - against the REAL reference (tests/golden/vqbase_img_64.pt), the way the GPU test checks it:
    pre-VQ activations, code indices (a mismatch must be a Voronoi-boundary crossing of OUR latent), then decoder output and
    every gradient with the quantiser pinned to the reference's codes."""
    from conftest import rel_err
    from mas_b200 import ops
    from models import VQBASE
    g = torch.load(os.path.join(GOLDEN, "vqbase_img_64.pt"), weights_only=False)
    torch.manual_seed(0)
    m = VQBASE(g["ddconfig"], 8192, 256, 3000, 12500)                       # seeded init == the reference's init (tests/test_abi.py)
    with torch.no_grad():
        m.quantize.embedding.weight.normal_()
    m.quantize.q_counter = 10 ** 6
    m.train()
    x = g["x"]
    h = {}
    hk = m.quant_conv.register_forward_hook(lambda _m, _i, o: h.__setitem__("q", o.detach()))
    hi = m.quantize.register_forward_hook(lambda _m, _i, o: h.__setitem__("idx", o[2].detach()))
    with torch.no_grad():
        m(x)
    hk.remove(); hi.remove()
    assert rel_err(h["q"], g["quant_in"]) < 3e-3                            # fp16 / TF32-sized operand rounding through 23 layers
    bad = torch.nonzero(h["idx"].view(-1) != g["idx"].view(-1)).flatten()
    assert bad.numel() <= 2
    if bad.numel():                                                         # ours must be the fp64 arg-min of OUR latent
        zf = h["q"].permute(0, 2, 3, 1).reshape(-1, 256)[bad].double()
        E = m.quantize.embedding.weight.detach().double()
        d = (zf * zf).sum(1, keepdim=True) + (E ** 2).sum(1)[None] - 2 * zf @ E.t()
        mine = d.gather(1, h["idx"].view(-1)[bad][:, None]).squeeze(1)
        assert bool((mine - d.min(1).values <= 4 * torch.finfo(torch.float32).eps * d.abs().max(1).values).all())
    # second pass with the decision pinned to the reference's codes: decoder output and every gradient
    m.quant_conv[1].reset_running_stats()
    cb = m.quantize
    idx_ref = g["idx"].view(-1)

    def fwd(z):
        zq, loss = ops.VQGivenFn.apply(z, cb.embedding.weight, cb.beta, idx_ref)
        return zq, loss, idx_ref
    cb.forward = fwd
    dec, diff = m(x)
    assert rel_err(dec, g["dec"]) < 5e-3
    assert abs(float(diff.detach()) - float(g["diff"])) < 5e-3 * abs(float(g["diff"]))
    ((x - dec).abs().mean() + diff).backward()
    named = dict(m.named_parameters())
    for k, gv in g["grads_small"].items():
        assert rel_err(named[k].grad, gv) < 2e-2, k
    worst = max(((abs(float(named[k].grad.double().norm()) - v) / max(v, 1e-4 * named[k].numel() ** 0.5)), k) for k, v in g["grad_norms"].items())
    assert worst[0] < 5e-2, worst
    n = vq_emu.names
    # 15 shadow-mode ResnetBlocks at >= 16 x 16: 2 convolutions in each forward pass, 2 more as data gradients in the backward
    assert n.count("mas_conv3x3_fprop_tc16h") == 90 and n.count("mas_attnblock_forward") == 14 and n.count("mas_vq_forward_given") == 1


def test_vqseg_step_host_logic_against_oracle(vq_emu):
    """The VQ-SEG step (159-channel maps: conv_in zero-padded to 160 input channels, conv_out run for 256 padded rows and returned
    as a channels-last view of a 160-channel buffer, weighted BCE forward / backward on that padded view, the gradient handed to
    the convolution's backward without a copy) above the emulated C-ABI against the CPU oracle (losses/loss_seg.py:6-22)."""
    from conftest import rel_err
    from mas_b200 import ops
    from models import VQBASE
    from oracle import vqgan_oracle as O
    dd = dict(z_channels=64, in_channels=159, out_channels=159, channels=[128, 128], num_res_blocks=1, resolution=64,
              attn_resolutions=[], dropout=0.0)
    torch.manual_seed(0)
    m = VQBASE(dd, 128, 64, 10, 100)
    with torch.no_grad():
        m.quantize.embedding.weight.normal_()
    m.quantize.q_counter = 10 ** 6
    m.train()
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    sd.update(params)
    seg = (torch.rand(2, 159, 64, 64, generator=torch.Generator().manual_seed(5)) > 0.9).float()
    dec_o, diff_o, idx_o = O.vqbase_forward(sd, dd, seg)
    lo = O.bce_loss_with_quant(diff_o, seg, dec_o)
    lo.backward()
    pw = torch.ones(159)
    pw[153:158] = 20
    cb = m.quantize
    idx_ref = idx_o.view(-1)

    def fwd(z):                        # the quantiser's decision pinned to the oracle's, as in the GPU test
        zq, loss = ops.VQGivenFn.apply(z, cb.embedding.weight, cb.beta, idx_ref)
        return zq, loss, idx_ref
    cb.forward = fwd
    dec, diff = m(seg)
    assert dec.shape == (2, 159, 64, 64) and ops._cl_pitch(dec) == 160
    loss = ops.BCELogitsFn.apply(dec, seg, pw) + diff
    loss.backward()
    assert rel_err(dec, dec_o) < 2e-3
    assert abs(float(loss.detach()) - float(lo.detach())) < 2e-3 * abs(float(lo.detach()))
    named = dict(m.named_parameters())
    for k, pr in params.items():
        assert rel_err(named[k].grad, pr.grad) < 1e-2, k
    n = vq_emu.names
    assert n.count("mas_bce_cl_forward") == 1 and n.count("mas_bce_cl_backward") == 1 and n.count("mas_nchw_to_nhwc_pad") == 1
    assert "mas_edge_small_cin_fprop" not in n and "mas_edge_small_cout_fprop" not in n      # both edge layers on the padded tensor route


def test_whole_model_modes_host_logic_against_reference_fixture(vq_emu):
    """The codebook's warm-up bypass (q_counter < q_init: no quantisation, zero loss, modules.py:482-484) and eval mode (running
    BatchNorm statistics, no counters / reservoir) above the emulated C-ABI, against the REAL reference (vqbase_tiny_modes.pt)."""
    from conftest import rel_err
    from models import VQBASE
    g = torch.load(os.path.join(GOLDEN, "vqbase_tiny.pt"), weights_only=False)
    mo = torch.load(os.path.join(GOLDEN, "vqbase_tiny_modes.pt"), weights_only=False)
    m = VQBASE(g["ddconfig"], g["n_embed"], g["embed_dim"], 10, 100)
    m.load_state_dict(g["state_dict"])
    m.train()
    dec, diff = m(g["x"])                      # q_counter = 1 < q_init: warm-up bypass
    assert float(diff) == 0.0 and rel_err(dec, mo["dec_bypass"]) < 1e-5
    assert "mas_vq_forward" not in vq_emu.names
    m.load_state_dict(g["state_dict"])
    m.eval()
    with torch.no_grad():
        dec, diff = m(g["x"])
    assert rel_err(dec, mo["dec_eval"]) < 1e-5
    assert abs(float(diff) - float(mo["diff_eval"])) < 1e-5 * abs(float(mo["diff_eval"]))
    assert "mas_bn_invstd" in vq_emu.names and vq_emu.names.count("mas_vq_forward") == 1


def test_codebook_schedule_host_logic_against_the_reference(vq_emu):
    """Codebook's training-time side paths (modules.py:474-499): step counter, reservoir sampling (10 latents per image, the
    same two torch.randperm draws per step), warm-up bypass - step by step IDENTICAL to the real reference's Codebook under the
    same seed up to the first re-initialisation; then our k-means replacement (the reference calls the absent
    fast_pytorch_kmeans there): triggered on the reference's schedule, lowers the quantisation error, and the following steps
    quantise against the new centres. The reference's per-step results are tests/golden/codebook_schedule.pt
    (oracle/make_golden.py --only=codebook)."""
    from models import modules as M
    g = torch.load(os.path.join(GOLDEN, "codebook_schedule.pt"), weights_only=False)
    K, D, init_steps = 16, 8, 4                                  # collect from step 5, quantise from step 12, re-init every 2 steps
    assert (g["K"], g["D"], g["init_steps"], g["reservoir_size"]) == (K, D, init_steps, 60)
    torch.manual_seed(3)
    ours = M.Codebook(K, D, 0.25, init_steps, 60)
    assert torch.equal(ours.embedding.weight.detach(), g["weight"])    # same initial codes as the reference's under that seed
    ours.train()
    gz = torch.Generator().manual_seed(11)
    zs = [torch.randn(3, D, 4, 4, generator=gz) for _ in range(16)]
    for step, z in enumerate(zs[:11], start=1):                  # steps 1 .. q_init - 1: both bypass, both collect from step 5 on
        torch.manual_seed(100 + step)
        a = ours(z)
        b = g["steps"][step - 1]
        assert ours.q_counter == b["q_counter"] == step
        assert a[2] is None and b["idx"] is None and float(a[1]) == 0.0 == b["loss"] and torch.equal(a[0], b["z_q"])
        if step > init_steps:
            assert torch.equal(ours.reservoir, b["reservoir"]) and ours.reservoir.shape[0] == min(60, 30 * (step - init_steps))
        else:
            assert ours.reservoir is None and b["reservoir"] is None
    assert "mas_vq_forward" not in vq_emu.names
    # step q_init = 12: the first re-initialisation from the reservoir, then quantisation
    e0 = ours.embedding.weight.detach().clone()
    res = ours.reservoir.clone()
    err = lambda E: float(((res[:, None, :] - E[None]) ** 2).sum(-1).min(1).values.mean())
    zq, loss, idx = ours(zs[11])
    assert ours.q_counter == 12 and vq_emu.names.count("mas_kmeans_update") >= 1
    e1 = ours.embedding.weight.detach()
    assert not torch.equal(e0, e1) and err(e1) < 0.5 * err(e0)                 # U(+-1/K) initial codes vs centres of the latents
    d = ((zs[11].permute(0, 2, 3, 1).reshape(-1, D)[:, None, :] - e1[None]) ** 2).sum(-1)
    assert torch.equal(idx.view(-1), d.argmin(1)) and torch.allclose(zq.permute(0, 2, 3, 1).reshape(-1, D), e1[idx.view(-1)])
    n_re = vq_emu.names.count("mas_kmeans_update")
    ours(zs[12])                                                  # step 13: (13 - 12) % 2 != 0 -> no re-initialisation
    assert vq_emu.names.count("mas_kmeans_update") == n_re
    ours(zs[13])                                                  # step 14: on the schedule again
    assert vq_emu.names.count("mas_kmeans_update") > n_re
    # eval mode: no counters, no reservoir updates
    ours.eval()
    q, r = ours.q_counter, ours.reservoir.clone()
    ours(zs[14])
    assert ours.q_counter == q and torch.equal(ours.reservoir, r)
    assert torch.equal(ours.get_codebook_entry(idx.view(-1), (3, 4, 4, D)), ours.embedding.weight.detach()[idx.view(-1)].view(3, 4, 4, D).permute(0, 3, 1, 2))
