"""BigVGANFlowVAE's kernels against float64 references of the same operations, at the bench config's shapes:

  * every tensor-core conv of the model (and three geometries the configs do not reach) on all three engines, with
    per-element bounds from the rounding model of each engine, at the M-tile edges and every stride residue;
  * the whole model against the float64 oracle (oracle/bigvgan_oracle.py), encode and decode, causal and not, with
    the equalities between the whole-clip, ragged and streaming calls at lengths that are not whole frames;
  * the fused anti-aliased activation (kvae_aa_act_fwd / kvae_aa_act_win_fwd) across its 1024-output tiles.

The other BigVGAN tests mostly check that two of the library's own paths agree bit for bit; these check that the shared
path is right."""
import pytest
import torch
import torch.nn.functional as F

import helpers as H
import kalle_audio_b200 as k
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.layers import TC_MIN_ROWS, WNConv1d
from oracle import alias_free_restated as AF
from oracle import bigvgan_oracle as BO

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


class AttrDict(dict):
    __getattr__ = dict.__getitem__


BENCH = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
                 downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
                 resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                 upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
                 activation="snakebeta", snake_logscale=True)
PRECISIONS = (None, "fp32", "bf16")
ENGINE = {None: 0, "bf16": 1, "fp32": 2}

# Per-element error bounds in units of A = conv(|x|, |w|) (float64, no bias), from the rounding model of each engine.
# Engine 1 multiplies bf16 operands exactly and sums in fp32; engine 2 adds the products hi.hi + hi.lo + lo.hi of the
# bf16 splits (the dropped lo.lo and the split residues are < 2^-16 of each product); engine 0 sums fp32 products.  A
# misplaced tap or a dropped 64-channel chunk is off by about A / (K Cin) or more, far above every bound.
BOUND_OWN = {0: 2.0 ** -18, 1: 2.0 ** -16, 2: 2.0 ** -16}      # against the engine's own operands
BOUND_EXACT = {0: 2.0 ** -18, 1: 2.0 ** -7, 2: 2.0 ** -14}     # against the exact conv of the fp32 operands
FP32_ULP = 2.0 ** -23                                          # the stored output and its bias add: one fp32 ulp


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _model(h, dev, seed=0):
    torch.manual_seed(seed)
    m = BV.BigVGANFlowVAE(AttrDict(h)).eval()
    for n, p in m.named_parameters():               # snake parameters away from their init
        if n.endswith(("alpha", "beta")):
            p.data = 0.2 * torch.randn_like(p) if m.h.snake_logscale else 1.0 + 0.3 * torch.rand_like(p)
    return m.to(dev)


def _bf16_ulp(r):
    """One bf16 ulp of |r| (8 significant bits)."""
    _, e = torch.frexp(r.abs())
    return torch.ldexp(torch.ones_like(r), e - 8)


def _split(t):
    """(hi, lo) of an fp32 tensor as split_pack_kernel / cf_to_cl_bf16_kernel split it, in float64."""
    hi = t.float().bfloat16()
    return hi.double(), (t.float() - hi.float()).bfloat16().double()


# ------------------------------------------------------------------------------------------------- a. layer sweep
def _conv64(m, x, w, bias):
    """The layer ``m`` in float64, sliced as oracle.bigvgan_oracle.conv / conv_transpose: a causal Conv1d keeps the
    first T rows of the symmetric-padded conv, a causal ConvTranspose1d drops its last ``stride`` rows."""
    K, s, d, p = m.kernel_size[0], m.stride[0], m.dilation[0], m.padding[0]
    if m.transposed:
        y = F.conv_transpose1d(x, w, bias, stride=s, padding=p)
        drop = getattr(m, "_drop", 0)
        return y[:, :, :-drop] if drop else y
    y = F.conv1d(x, w, bias, stride=s, padding=p, dilation=d)
    return y[:, :, :x.shape[2]] if getattr(m, "causal", False) and K > 1 else y


def _q_rows(m, T):
    """Output rows per stride phase that the tcgen05 kernel tiles (Tq_out) for an input of T rows."""
    K, s, d, p = m.kernel_size[0], m.stride[0], m.dilation[0], m.padding[0]
    if m.transposed:
        keep = T * s if getattr(m, "_drop", 0) else (T - 1) * s - 2 * p + K
        return -(-keep // s)
    if getattr(m, "causal", False) and K > 1:
        return T
    return (T + 2 * p - d * (K - 1) - 1) // s + 1


def _lengths(m):
    """Input lengths: the 64-row threshold, Tq_out of 127 / 128 / 129 and 255 / 256 / 257 (one vs. two 128-row M
    tiles), one long odd length; a strided conv cycles the residues of T mod s at the tile edges and takes every
    residue at the long length."""
    s_in = 1 if m.transposed else m.stride[0]
    out = [TC_MIN_ROWS]
    for i, tq in enumerate((127, 128, 129, 255, 256, 257)):
        cands = [T for T in range(TC_MIN_ROWS, (tq + 4) * s_in + 16) if _q_rows(m, T) == tq]
        out.append(cands[i % len(cands)])
    out += [1001 + r for r in range(s_in)] if s_in > 1 else [1001]
    return out


def _layer_case(m, x, tag, worst, fails):
    """m(x[:B]) for B in (1, 3) under every precision against the float64 references of the same conv."""
    w = m.folded_weight()
    b = None if m.bias is None else m.bias.detach().double()
    xd, wd = x.double(), w.double()
    exact = _conv64(m, xd, wd, b)
    A = _conv64(m, xd.abs(), wd.abs(), None)
    xh, xl = _split(x)
    wh, wl = _split(w)
    own = {0: exact, 1: _conv64(m, x.bfloat16().double(), w.bfloat16().double(), b),
           2: _conv64(m, xh, wh + wl, b) + _conv64(m, xl, wh, None)}       # hi.hi + hi.lo + lo.hi
    out_tol = FP32_ULP * exact.abs() if x.dtype == torch.float32 else _bf16_ulp(exact)
    Ad = A.clamp_min(1e-300)
    for prec in PRECISIONS:
        m.tc_precision = prec
        e = ENGINE[prec]
        for B in (1, 3):
            case = f"{tag} T={x.shape[2]} B={B} {prec}"
            try:
                y = m(x[:B]).double()
            except _lib.KvaeError as err:
                fails.append(f"{case}: {err}")
                continue
            if y.shape != exact[:B].shape:
                fails.append(f"{case}: shape {tuple(y.shape)} != {tuple(exact[:B].shape)}")
                continue
            for name, ref, bound in (("own", own[e], BOUND_OWN[e]), ("exact", exact, BOUND_EXACT[e])):
                err = (y - ref[:B]).abs()
                ratio = float(((err - out_tol[:B]).clamp_min(0) / Ad[:B]).max())
                if ratio > worst.get((e, name), (0.0, ""))[0]:
                    worst[(e, name)] = (ratio, case)
                if not bool((err <= bound * A[:B] + out_tol[:B]).all()):
                    fails.append(f"{case}: err / A {ratio:.3e} against the {name} reference > {bound:.3e}")
    m.tc_precision = "fp32"


def _tc_modules(model, encoder):
    """The distinct tensor-core conv geometries of the model's op list: one module per geometry."""
    ops, _ = BV._encoder_program(model.h) if encoder else BV._program(model.h)
    model.set_precision("fp32")
    mods = {}
    for op in ops:
        if op.kind not in ("conv", "convT"):
            continue
        m = BV._module(model, op.module)
        key = (m.transposed, m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0], m.dilation[0],
               m.padding[0], getattr(m, "causal", False))
        if m.tc_layer() and key not in mods:
            mods[key] = (op.module, m)
    return list(mods.values())


def _check_fold(m, tag, fails):
    """folded_weight() (kvae_weight_norm_fold) against the float64 fold: per element within 2^-18 relative (fp32 sum
    of <= 64 squares per thread and a 10-level tree, a square root, a division and a product)."""
    v, g = m.weight_v.detach().double(), m.weight_g.detach().double()
    ref = v * (g / v.flatten(1).norm(dim=1).view(-1, *([1] * (v.dim() - 1))))
    if not bool(((m.folded_weight().double() - ref).abs() <= 2.0 ** -18 * ref.abs()).all()):
        fails.append(f"{tag}: folded weight off the float64 fold")


def _sweep(mods, dev, label):
    worst, fails = {}, []
    gen = torch.Generator(device=dev).manual_seed(5)
    for tag, m in mods:
        _check_fold(m, tag, fails)
        for T in _lengths(m):
            x = torch.randn(3, m.in_channels, T, device=dev, generator=gen)
            _layer_case(m, x, tag, worst, fails)
    for (e, name), (ratio, case) in sorted(worst.items()):
        H.report(f"BigVGAN tc-layer sweep {label}: engine {e} max err/A vs {name} conv "
                 f"(bound {(BOUND_OWN if name == 'own' else BOUND_EXACT)[e]:.1e})", f"{ratio:.3e} at {case}")
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:40])


@pytest.mark.parametrize("part", ["decoder_causal", "decoder_noncausal", "encoder"])
def test_tensor_core_layers_vs_float64(dev, part):
    """Every tensor-core conv of the bench config: the whole-layer call ``module(x)`` (causal truncation and the
    transposed convs' stride-group rounding included) on engines 0 / 1 / 2 against float64 convs."""
    model = _model(dict(BENCH, causal=part != "decoder_noncausal"), dev)
    mods = _tc_modules(model, part == "encoder")
    assert len(mods) >= (20 if part == "encoder" else 40)
    _sweep(mods, dev, part)


def test_tensor_core_layers_outside_the_configs(dev):
    """Geometries the configs do not reach: Cout = 192 (three 64-wide N tiles), K = 32 (kMaxTaps) and a stride-8
    strided conv (kMaxPhases)."""
    torch.manual_seed(11)
    mods = [("c64-192 k3", WNConv1d(64, 192, 3, padding=1)), ("c64-128 k32", WNConv1d(64, 128, 32, padding=16)),
            ("c64-128 k16 s8", WNConv1d(64, 128, 16, stride=8, padding=7))]
    for _, m in mods:
        m.to(dev).tc_precision = "fp32"
        assert m.tc_layer()
    _sweep(mods, dev, "synthetic")


@pytest.mark.parametrize("engine", [1, 2])
def test_pitched_bf16_window_conv_vs_float64(dev, engine):
    """kvae_conv1d_win_fwd straight: bf16 input at a row pitch wider than T, bf16 output rows [o0, o1) inside the
    layer, against the float64 conv of the same bf16 values (plus one bf16 ulp of the stored output)."""
    torch.manual_seed(engine)
    Cin, Cout, K, d, p, T, o0, o1 = 128, 256, 7, 3, 9, 700, 3, 611
    L = _lib.lib()
    w = 0.05 * torch.randn(Cout, Cin, K, device=dev)
    bias = torch.randn(Cout, device=dev)
    xbuf = torch.randn(2, Cin, T + 13, device=dev).bfloat16()
    x = xbuf[:, :, :T]
    nb = L.kvae_conv1d_packed_bytes(Cin, Cout, K, engine)
    packed = torch.empty(nb, dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_pack(w.data_ptr(), 0, Cin, Cout, K, engine, packed.data_ptr(), nb, 0))
    y = torch.empty(2, Cout, o1 - o0, dtype=torch.bfloat16, device=dev)
    ns = L.kvae_conv1d_win_scratch_bytes(2, Cin, T, engine)
    sc = torch.empty(ns, dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_win_fwd(xbuf.data_ptr(), T + 13, y.data_ptr(), o1 - o0, packed.data_ptr(), bias.data_ptr(),
                                     0, 2, Cin, Cout, T, K, 1, d, p, o0, o1, _lib.KVAE_BF16, engine, sc.data_ptr(), ns, 0))
    xd = x.double()
    ref = F.conv1d(xd, w.double(), bias.double(), padding=p, dilation=d)[:, :, o0:o1]
    A = F.conv1d(xd.abs(), w.double().abs(), padding=p, dilation=d)[:, :, o0:o1]
    if engine == 1:
        own = F.conv1d(xd, w.bfloat16().double(), bias.double(), padding=p, dilation=d)[:, :, o0:o1]
    else:                                            # bf16 input: its lo half is 0
        wh, wl = _split(w)
        own = F.conv1d(xd, wh + wl, bias.double(), padding=p, dilation=d)[:, :, o0:o1]
    err = (y.double() - own).abs()
    assert bool((err <= BOUND_OWN[engine] * A + _bf16_ulp(own)).all())
    assert bool(((y.double() - ref).abs() <= BOUND_EXACT[engine] * A + _bf16_ulp(ref)).all())
    H.report(f"pitched bf16 window conv engine {engine}: max |err| / (A + ulp)",
             float((err / (A + _bf16_ulp(own))).max()))


# ------------------------------------------------------------------------------------------------- b. whole model
def _oracle(fn, m, x, *args):
    """fn (oracle.bigvgan_oracle) in float64 on x's device; the alias-free filters follow the default dtype."""
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.device(x.device):
            sd = {n: p.detach().double() for n, p in m.state_dict().items()}
            return fn(sd, dict(m.h), x.double(), *args)
    finally:
        torch.set_default_dtype(prev)


@pytest.fixture(scope="module")
def decode_cases(dev):
    """(model, latents, float64 oracle output) of a 70-frame decode (ups.0 on the tensor cores), causal and not."""
    out = {}
    for causal in (True, False):
        m = _model(dict(BENCH, causal=causal), dev, seed=1)
        z = torch.randn(2, 512, 70, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
        out[causal] = (m, z, _oracle(BO.inference_from_latents, m, z))
    return out


@pytest.fixture(scope="module")
def encode_cases(dev):
    """(model, audio, float64 oracle latents) for 113 000 samples (not whole frames), 1280 x 80 samples, and bf16
    audio of 113 000 samples."""
    m = _model(BENCH, dev, seed=3)
    gen = torch.Generator(device=dev).manual_seed(4)
    out = {}
    for tag, L, dt in (("113000", 113000, torch.float32), ("102400", 1280 * 80, torch.float32),
                       ("113000_bf16", 113000, torch.bfloat16)):
        x = (0.3 * torch.randn(1, 1, L, device=dev, generator=gen)).to(dt)
        out[tag] = (m, x, _oracle(BO.extract_latents, m, x))
    return out


def _model_errors(run, ref, label):
    errs = {}
    for prec in PRECISIONS:
        y = run(prec)
        assert y.shape == ref.shape
        errs[prec] = float((y.double() - ref).abs().max())
    scale = max(1.0, float(ref.abs().max()))
    H.report(f"{label}: CUDA-core / tensor-core fp32 / bf16 max err (max |ref| {float(ref.abs().max()):.2f})",
             " / ".join(f"{v:.2e}" for v in errs.values()))
    return errs, scale


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
def test_bench_decode_vs_oracle(dev, decode_cases, causal):
    m, z, ref = decode_cases[causal]
    errs, scale = _model_errors(lambda prec: m.set_precision(prec).inference_from_latents(z, do_sample=False), ref,
                                f"BigVGAN bench decode 70 frames ({'causal' if causal else 'non-causal'})")
    assert errs[None] <= 2e-5 * scale and errs["fp32"] <= 2e-5 * scale and errs["bf16"] <= 5e-3 * scale
    assert errs["bf16"] > errs["fp32"]
    if not causal:                                   # the stream's flush of the odd K - s layers (ups.1, K 10 rate 5)
        m.set_precision("bf16")
        whole = m.inference_from_latents(z, do_sample=False)
        sd = k.BigVGANStreamingDecoder(m)
        outs = [sd.push(z[:, :, a:b]) for a, b in ((0, 1), (1, 17), (17, 17), (17, 37), (37, 70))]
        y = torch.cat(outs + [sd.flush()], dim=2)
        assert y.shape == whole.shape and torch.equal(y, whole)


@pytest.mark.parametrize("tag", ["113000", "102400"])
def test_bench_encode_vs_oracle(dev, encode_cases, tag):
    m, x, ref = encode_cases[tag]
    errs, scale = _model_errors(lambda prec: m.set_precision(prec).extract_latents(x), ref,
                                f"BigVGAN bench encode {tag} samples")
    assert errs[None] <= 2e-5 * scale and errs["fp32"] <= 2e-5 * scale and errs["bf16"] <= 5e-3 * scale
    assert errs["bf16"] > errs["fp32"]


def test_bench_encode_bf16_audio_vs_oracle(dev, encode_cases):
    """bf16 audio: every layer of the call stores bf16, so all three precisions are held to the bf16 criterion, against
    the oracle on the same bf16 samples."""
    m, x, ref = encode_cases["113000_bf16"]
    errs, scale = _model_errors(lambda prec: m.set_precision(prec).extract_latents(x), ref,
                                "BigVGAN bench encode 113000 bf16 samples")
    assert all(e <= 5e-3 * scale for e in errs.values())


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_non_frame_encode_equals_ragged_and_stream(dev, encode_cases, prec):
    """113 000 samples (not whole frames): the whole-clip call, the ragged call on the clip padded to whole frames and
    the streaming encoder give the same latents bit for bit."""
    m, x, _ = encode_cases["113000"]
    L = x.shape[2]
    m.set_precision(prec)
    y = m.extract_latents(x)
    assert y.shape[2] == m.latent_length(L)
    yr = m.extract_latents(F.pad(x, (0, -L % 1280)), valid_len=[L])[:, :, :m.latent_length(L)]
    assert torch.equal(y, yr)
    se = k.BigVGANStreamingEncoder(m)
    outs = [se.push(x[:, :, a:b]) for a, b in ((0, 20000), (20000, 20001), (20001, 53333), (53333, L))]
    ys = torch.cat(outs + [se.flush()], dim=2)
    assert ys.shape == y.shape and torch.equal(ys, y)


# ------------------------------------------------------------------------------------------------- c. activation
def _aa_ref(act, x):
    """UpSample1d -> snake -> DownSample1d in float64 with the module's own filter buffers."""
    up, down = AF.UpSample1d(2, 12).to(x.device), AF.DownSample1d(2, 12).to(x.device)
    up.filter = act.upsample.filter.double()
    down.lowpass.filter = act.downsample.lowpass.filter.double()
    beta = getattr(act.act, "beta", None)
    v = BO.snake(up(x.double()), act.act.alpha.double(), None if beta is None else beta.double(),
                 act.act.alpha_logscale)
    return down(v)


def _act(cls, C, logscale, dev):
    act = BV.Activation1d(cls(C, alpha_logscale=logscale))
    act.act.alpha.data = (0.3 * torch.randn(C)) if logscale else (1.0 + 0.3 * torch.rand(C))
    if hasattr(act.act, "beta"):
        act.act.beta.data = (0.3 * torch.randn(C)) if logscale else (1.0 + 0.3 * torch.rand(C))
    return act.to(dev)


@pytest.mark.parametrize("T", [1023, 1024, 1025, 2048 + 37, 5000])
@pytest.mark.parametrize("C", [6, 96])
def test_anti_aliased_activation_across_tiles(dev, T, C):
    """kvae_aa_act_fwd over several 1024-output tiles (the halo of each read across the tile edges), fp32 and bf16
    input, Snake and SnakeBeta, logscale on and off."""
    torch.manual_seed(T + C)
    worst = 0.0
    for cls in (BV.Snake, BV.SnakeBeta):
        for logscale in (False, True):
            act = _act(cls, C, logscale, dev)
            x = torch.randn(2, C, T, device=dev)
            ref = _aa_ref(act, x)
            tol = 5e-6 * max(1.0, float(ref.abs().max()))
            err = float((act(x).double() - ref).abs().max())
            worst = max(worst, err)
            assert err <= tol, (cls.__name__, logscale, err)
            xb = x.bfloat16()
            refb = _aa_ref(act, xb)
            yb = act(xb)
            assert yb.dtype == torch.bfloat16
            assert bool(((yb.double() - refb).abs() <= 5e-6 * max(1.0, float(refb.abs().max())) +
                         _bf16_ulp(refb)).all()), (cls.__name__, logscale, "bf16")
    H.report(f"anti-aliased activation C={C} T={T}: max err (fp32 input)", worst)


def test_anti_aliased_activation_window_across_a_tile_edge(dev):
    """kvae_aa_act_win_fwd: windows whose first output is not a multiple of 1024 and which cross tile edges, inside
    the stream and at its end, against the same slice of the float64 reference."""
    torch.manual_seed(7)
    T = 5000
    act = _act(BV.SnakeBeta, 96, True, dev)
    x = torch.randn(2, 96, T, device=dev)
    ref = _aa_ref(act, x)
    tol = 5e-6 * max(1.0, float(ref.abs().max()))
    for o0, o1, end in ((1000, 2100, False), (1500, 1600, False), (3001, T, True)):
        x0, x1 = o0 - 5, T if end else o1 + 5
        buf = torch.full((2, 96, x1 - x0 + 7), float("nan"), device=dev)      # pitched
        buf[:, :, :x1 - x0] = x[:, :, x0:x1]
        y = act.window(buf[:, :, :x1 - x0], x0, o0, o1, T if end else -1)
        assert float((y.double() - ref[:, :, o0:o1]).abs().max()) <= tol, (o0, o1)
