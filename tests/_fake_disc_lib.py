"""CPU stand-in for the libkvae entry points the discriminator's host layer calls.  TEST INFRASTRUCTURE ONLY.

The build container has no GPU, so the autograd orchestration of kalle_audio_b200/discriminators.py (forward chain,
hand-written backward chain, weight / input folding, gradient bookkeeping) is checked here against the reference's
recorded autograd gradients by running it over this stand-in: every entry point restates its documented contract
(include/kvae.h) with torch CPU ops on the raw pointers it is handed -- the fold / unfold index formulas literally as
csrc/disc.cuh writes them.  The CUDA kernels themselves are checked on the GPU (tests/test_gpu_discriminator.py)."""
import ctypes

import numpy as np
import torch
import torch.nn.functional as F


def T(ptr, *shape):
    n = int(np.prod(shape))
    buf = (ctypes.c_float * n).from_address(int(ptr))
    return torch.from_numpy(np.ctypeslib.as_array(buf)).view(*shape)


class FakeLib:
    def __init__(self):
        self.calls = []

    def kvae_last_error(self):
        return b"fake"

    # ---- existing layer-level entry points
    def kvae_weight_norm_fold(self, v, g, w, dim0, inner, st):
        vv, gg = T(v, dim0, inner), T(g, dim0, 1)
        T(w, dim0, inner).copy_(vv * (gg / vv.norm(dim=1, keepdim=True)))
        return 0

    def kvae_weight_norm_bwd(self, v, g, dw, dv, dg, dim0, inner, st):
        vv, gg, d = T(v, dim0, inner), T(g, dim0, 1), T(dw, dim0, inner)
        n = vv.norm(dim=1, keepdim=True)
        dot = (d * vv).sum(1, keepdim=True)
        T(dg, dim0).copy_((dot / n).view(-1))
        T(dv, dim0, inner).copy_((gg / n) * (d - vv * dot / (n * n)))
        return 0

    def kvae_conv1d_scratch_bytes(self, Cin, Cout, K):
        return 1024

    def kvae_conv1d_fwd(self, x, y, w, bias, transposed, B, Cin, Cout, Tn, K, stride, dil, pad, dtype, scratch, ns, st):
        assert not transposed and dtype == 0
        xx, ww = T(x, B, Cin, Tn), T(w, Cout, Cin, K)
        out = F.conv1d(xx, ww, None if bias is None else T(bias, Cout), stride=stride, padding=pad, dilation=dil)
        T(y, *out.shape).copy_(out)
        self.calls.append(("conv_fwd", Cin, Cout, K))
        return 0

    def kvae_conv1d_win_bwd_scratch_bytes(self, transposed, B, Cin, Cout, Tn, T_gy, K, stride, engine):
        return 1024

    def kvae_conv1d_win_bwd(self, x, gy, T_gy, w, v, g, gx, dv, dg, dbias, transposed, B, Cin, Cout, Tn, K, stride, dil,
                            pad, dtype, engine, scratch, ns, st):
        assert not transposed and dtype == 0 and engine == 0 and v is None and g is None
        with torch.enable_grad():
            xx = T(x, B, Cin, Tn).clone().requires_grad_(True)
            ww = T(w, Cout, Cin, K).clone().requires_grad_(True)
            out = F.conv1d(xx, ww, None, stride=stride, padding=pad, dilation=dil)
            assert out.shape[2] == T_gy
            gr = T(gy, *out.shape)
            gxx, gww = torch.autograd.grad(out, (xx, ww), gr)
        if gx is not None:
            T(gx, B, Cin, Tn).copy_(gxx)
        if dv is not None:
            T(dv, Cout, Cin, K).copy_(gww)
        if dbias is not None:
            T(dbias, Cout).copy_(gr.sum((0, 2)))
        self.calls.append(("conv_bwd", gx is not None, dv is not None))
        return 0

    def kvae_disc_conv15_supported(self, K, stride, pad):
        return int(K == 15 and stride == 4 and pad == 7)

    def kvae_disc_conv15_fwd(self, x, y, w, bias, N, Cin, Cout, Tn, scratch, ns, st):
        return self.kvae_conv1d_fwd(x, y, w, bias, 0, N, Cin, Cout, Tn, 15, 4, 1, 7, 0, scratch, ns, st)

    def kvae_disc_conv15_bwd(self, x, gy, w, gx, dw, dbias, N, Cin, Cout, Tn, scratch, ns, st):
        return self.kvae_conv1d_win_bwd(x, gy, (Tn - 1) // 4 + 1, w, None, None, gx, dw, None, dbias, 0, N, Cin, Cout, Tn,
                                        15, 4, 1, 7, 0, 0, scratch, ns, st)

    def kvae_disc_conv1x1_supported(self, K, stride, pad, Cout):
        return int(K == 1 and stride == 1 and pad == 0 and 1 <= Cout <= 8)

    def kvae_disc_conv1x1_fwd(self, x, y, w, bias, N, Cin, Cout, Tn, st):
        return self.kvae_conv1d_fwd(x, y, w, bias, 0, N, Cin, Cout, Tn, 1, 1, 1, 0, 0, None, 0, st)

    def kvae_disc_conv1x1_bwd(self, x, gy, w, gx, dw, dbias, N, Cin, Cout, Tn, st):
        return self.kvae_conv1d_win_bwd(x, gy, Tn, w, None, None, gx, dw, None, dbias, 0, N, Cin, Cout, Tn, 1, 1, 1, 0, 0, 0,
                                        None, 0, st)

    # ---- csrc/disc.cuh
    def kvae_disc_period_fold(self, x, y, N, Cc, Tn, n, backward, st):
        H = (Tn + n - 1) // n
        if not backward:
            xx = F.pad(T(x, N, Cc, Tn), (0, H * n - Tn)).view(N, Cc, H, n)
            T(y, N, Cc, n, H).copy_(xx.transpose(2, 3))            # y[b, c n + w, h] = x[b, c, h n + w]
        else:
            g = T(x, N, Cc, n, H).transpose(2, 3).reshape(N, Cc, H * n)
            T(y, N, Cc, Tn).copy_(g[:, :, :Tn])
        return 0

    def kvae_disc_avg_pool2(self, x, y, rows, Tn, backward, st):
        To = Tn // 2
        if not backward:
            xx = T(x, rows, Tn)
            T(y, rows, To).copy_((xx[:, 0:2 * To:2] + xx[:, 1:2 * To:2]) * 0.5)
        else:
            g = T(x, rows, To)
            out = T(y, rows, Tn)
            out.zero_()
            out[:, :2 * To] = 0.5 * g.repeat_interleave(2, dim=1)
        return 0

    def kvae_disc_folded_width(self, W, K, stride, pad):
        if W <= 0 or K <= 0 or stride <= 0 or pad < 0 or W + 2 * pad < K:
            return 0
        return (W + 2 * pad - K) // stride + 1

    def kvae_disc_fold_weight2d(self, w, bias, wf, bias_f, Cout, Cin, K, stride, pad, W, backward, st):
        Wo = self.kvae_disc_folded_width(W, K, stride, pad)
        ww = T(w, Cout, Cin, K, K)
        wff = T(wf, Cout, Wo, Cin, W, K)
        if not backward:
            wff.zero_()
            for wo in range(Wo):
                for wi in range(W):
                    kw = wi - stride * wo + pad
                    if 0 <= kw < K:
                        wff[:, wo, :, wi, :] = ww[:, :, :, kw]
            if bias is not None:
                T(bias_f, Cout, Wo).copy_(T(bias, Cout, 1).expand(Cout, Wo))
        else:
            ww.zero_()
            for kw in range(K):
                for wo in range(Wo):
                    wi = kw + stride * wo - pad
                    if 0 <= wi < W:
                        ww[:, :, :, kw] += wff[:, wo, :, wi, :]
            if bias is not None:
                T(bias, Cout).copy_(T(bias_f, Cout, Wo).sum(1))
        return 0

    def kvae_disc_silu_fwd(self, f, a, n, st):
        T(a, n).copy_(F.silu(T(f, n)))
        return 0

    def kvae_disc_silu_bwd(self, f, ga, gfeat, gf, n, st):
        ff = T(f, n)
        s = torch.sigmoid(ff)
        g = T(ga, n) * (s * (1 + ff * (1 - s)))
        if gfeat is not None:
            g = g + T(gfeat, n)
        T(gf, n).copy_(g)
        return 0

    def kvae_disc_score(self, y, score, N, inner, accumulate, st):
        m = T(y, N, inner).mean(1)
        s = T(score, N)
        s.copy_(s + m if accumulate else m)
        return 0

    def kvae_disc_score_bwd(self, gscore, gfeat, gy, N, inner, st):
        g = torch.zeros(N, inner)
        if gscore is not None:
            g = g + T(gscore, N, 1) / inner
        if gfeat is not None:
            g = g + T(gfeat, N, inner)
        T(gy, N, inner).copy_(g)
        return 0

    def kvae_disc_hinge(self, score, B, losses, g_losses, g_score, st):
        s = T(score, 2 * B)
        if g_losses is None:
            out = T(losses, 2)
            out[0] = torch.relu(1 - s[:B]).mean() + torch.relu(1 + s[B:]).mean()
            out[1] = -s[B:].mean()
        else:
            gl = T(g_losses, 2)
            g = T(g_score, 2 * B)
            g[:B] = torch.where(1 - s[:B] > 0, -gl[0] / B, torch.zeros(()))
            g[B:] = torch.where(1 + s[B:] > 0, gl[0] / B, torch.zeros(())) - gl[1] / B
        return 0

    def kvae_disc_feature_match_scratch_bytes(self, half, n):
        return 1024

    def kvae_disc_feature_match(self, feats, half, n, loss, g_loss, grads, scratch, ns, st):
        if g_loss is None:
            tot = torch.zeros(())
            for k in range(n):
                f = T(feats[k], 2, half[k])
                tot = tot + (f[0] - f[1]).abs().sum() / half[k]
            T(loss, 1)[0] = tot
        else:
            g = T(g_loss, 1)[0].clone()
            for k in range(n):
                f = T(feats[k], 2, half[k])
                v = torch.sign(f[0] - f[1]) * g / half[k]
                out = T(grads[k], 2, half[k])
                out[0] = v
                out[1] = -v
        return 0
