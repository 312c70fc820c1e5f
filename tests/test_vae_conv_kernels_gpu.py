"""The VAE conv kernels one launch at a time, at the shapes that reach them, against a plain fp64 reference.

Most of a Wan VAE decode runs in the CTA-pair conv kernels (csrc/conv2_sm100.cuh) with the fused RMS_norm + SiLU epilogue.  The
dispatcher (csrc/vae_ops.cu::conv_cl_impl) takes the pair kernels only when a launch has T * ceil(H / ROWS) * ceil(W / 128) >= 2 * #SMs
row tiles, far above the unit shapes of test_vae_gpu.py, and the decode tests hold whole frames to loose tolerances that a few
percent of error in one tile column would pass.  Here every case of the table below runs one entry point and checks:

  (a) dispatch:    the profiler sees exactly the expected conv instance (and no other conv instance)
  (b) raw output:  every element vs the fp64 implicit GEMM, |d| <= 2^-8 |ref| + 2^-12 rms(ref), and rel-L2 < 4e-3
  (c) norm output: per-pixel rel-L2 over the channels < 1e-2 and global rel-L2 < 4e-3 vs silu(rms_norm(bf16(ref)) * gamma) in fp64
  (d) consistency: the fused kernel's raw output is bit-identical to the plain kernel's, its norm output is within 1 bf16 ulp of
                   rms_silu(plain output) and bit-identical to it almost everywhere (only the order of the sum of squares differs)
  (e) coverage:    outputs live inside larger buffers filled with a sentinel bit pattern: the guard bands stay untouched and no
                   sentinel survives inside the output (every pixel written, by all four parity launches of the up-sampling conv)

Inputs make statistics bugs loud: per-pixel magnitudes spread over 2^-3..2^3, the upper half of the output channels 4x larger (a
missing exchange of the two epilogue warpgroups' sums of squares), gamma and bias different for every channel.  Shapes are chosen
for the B200's 148 SMs -- ragged last row tiles, odd H (masked second row), odd tile counts (an all-out-of-range tile in the last
CTA pair) -- and grown in H when the device has more SMs."""
import math
import os
import re
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import psnr, rel_l2

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

bf16, f32, f64 = torch.bfloat16, torch.float32, torch.float64
ROW_TILE = 128              # pixels per row tile (CONVR_BW)
SENTINEL = 0x7FA5           # a NaN payload: the kernels never produce it
GUARD = 40                  # sentinel elements in front of an output: 80 bytes keeps 16-byte alignment, breaks 128-byte alignment
# fraction of norm outputs allowed to differ (by 1 ulp) from rms_silu of the plain output: the two sum the squares in a different
# fp32 order, which moves 1/rms by a few fp32 ulps and flips a bf16 rounding in ~1e-4 of the elements
NORM_FLIP_FRAC = 2e-3


@dataclass(frozen=True)
class Case:
    label: str
    entry: str              # conv_norm | upconv_norm | stream_norm | conv | repconv | timeconv
    kernel: tuple           # expected instance: (kernel name, template arguments)
    T: int
    H: int
    W: int
    cin: int
    cout: int
    k: tuple = (3, 3, 3)
    pair: object = True     # True: CTA-pair side of the threshold, False: single-CTA side, None: not a row-tiled conv
    residual: bool = False
    raw: bool = True        # the fused call also writes the un-normalised output


def _v2(*a):
    return ("conv_row2_tcgen05_kernel", a)


def _v1(*a):
    return ("conv_row_tcgen05_kernel", a)


CASES = [
    Case("wan 96 fused", "conv_norm", _v2(96, 2, 32, 1, 3, 9), 3, 29, 832, 96, 96),
    Case("wan 96 fused norm_only", "conv_norm", _v2(96, 2, 32, 1, 3, 9), 3, 29, 832, 96, 96, raw=False),
    Case("wan 96 fused +residual", "conv_norm", _v2(96, 2, 32, 1, 3, 9), 3, 29, 832, 96, 96, residual=True),
    Case("wan 192 fused 480p", "conv_norm", _v2(192, 1, 64, 1, 3, 3), 3, 25, 416, 192, 192, residual=True),
    Case("wan 192 fused odd tiles", "conv_norm", _v2(192, 1, 64, 1, 3, 3), 3, 33, 330, 192, 192),
    Case("wan up 192->96 fused", "upconv_norm", _v2(96, 2, 64, 1, 2, 4), 3, 50, 416, 192, 96),
    Case("wan up 192->96 fused odd tiles", "upconv_norm", _v2(96, 2, 64, 1, 2, 4), 5, 41, 330, 192, 96),
    Case("wan up 384->192 fused", "upconv_norm", _v2(192, 1, 64, 1, 2, 4), 3, 50, 208, 384, 192),
    Case("wan 96 fused single-CTA", "conv_norm", _v1(96, 2, 32, 1, 0), 2, 5, 104, 96, 96, pair=False, residual=True),
    Case("wan 192 fused single-CTA", "conv_norm", _v1(192, 1, 64, 1, 0), 2, 5, 230, 192, 192, pair=False, residual=True),
    Case("wan up 192->96 fused single-CTA", "upconv_norm", _v1(96, 2, 64, 1, 0), 2, 5, 110, 192, 96, pair=False),
    Case("wan 96 plain +residual", "conv", _v2(96, 2, 32, 0, 3, 9), 3, 29, 832, 96, 96, residual=True),
    Case("hy 128 replicate", "repconv", _v2(128, 2, 64, 0, 3, 3), 3, 50, 424, 128, 128, residual=True),
    Case("hy 256 replicate", "repconv", _v2(256, 1, 64, 0, 3, 3), 3, 50, 212, 256, 256),
    Case("stream 96 fused +residual", "stream_norm", _v2(96, 2, 32, 1, 3, 9), 3, 29, 832, 96, 96, residual=True),
    Case("stream 96 fused single-CTA", "stream_norm", _v1(96, 2, 32, 1, 0), 2, 5, 104, 96, 96, pair=False),
    Case("time_conv interleave 384->768", "timeconv", ("gemm_tcgen05_kernel", (256, 0, 64, 1, 0)), 5, 6, 10, 384, 768, k=(3, 1, 1),
         pair=None),
]


def _s():
    return torch.cuda.current_stream().cuda_stream


def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tiles(c, H):
    rows = 2 if c.cout <= 128 else 1                 # ROWS of the row kernel for BN = Cout (conv_row_rows)
    return c.T * -(-H // rows) * -(-c.W // ROW_TILE)


def _shape_h(c):
    """H of the case on this device: the table's H (chosen for 148 SMs), grown by 2 rows at a time (keeping its parity) until a
    CTA-pair case reaches the pair threshold."""
    H, need = c.H, 2 * _num_sms()
    if c.pair is True:
        while _tiles(c, H) < need:
            H += 2
    elif c.pair is False:
        assert _tiles(c, H) < need, f"{c.label}: {_tiles(c, H)} tiles reach the CTA-pair threshold {need}"
    return H


# ---------------------------------------------------------------------------------------------------------------- inputs
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _act(shape, seed):
    """bf16 activations whose pixels have magnitudes spread over 2^-3..2^3 (every pixel's sum of squares is different)."""
    g = _gen(seed)
    x = torch.randn(*shape, generator=g, device="cuda")
    scale = torch.exp2(torch.rand(*shape[:-1], 1, generator=g, device="cuda") * 6 - 3)
    return (x * scale).to(bf16).contiguous()


def _weights(cout, cin, k, seed):
    """fp32 conv weights [Cout, Cin, *k]; the upper half of the output channels 4x larger."""
    g = _gen(seed)
    w = torch.randn(cout, cin, *k, generator=g, device="cuda") * (cin * math.prod(k)) ** -0.5
    w[cout // 2:] *= 4
    return w


def _per_channel(c, seed, lo, hi):
    g = _gen(seed)
    return (lo + (hi - lo) * torch.rand(c, generator=g, device="cuda")).contiguous()


# ---------------------------------------------------------------------------------------------------------------- fp64 references
def conv_ref(x, w, bias, k, pad="zeros", t_front=None):
    """Causal-in-time, centred-in-space conv as an implicit GEMM in fp64: sum over the taps of [P, Cin] @ [Cin, Cout].
    x bf16 [Ti, H, W, Cin]; w the packed operand [Cout, taps (t, h, w), Cin]; t_front frames of padding in front (default kt - 1;
    0 when x carries its own history frames).  pad: "zeros" or "replicate" (time and space).  -> fp64 [Ti + t_front - kt + 1, H, W, Cout]."""
    kt, kh, kw = k
    t_front = kt - 1 if t_front is None else t_front
    xd = x.double().permute(3, 0, 1, 2)[None]                                             # [1, C, T, H, W]
    pads = (kw // 2, kw // 2, kh // 2, kh // 2, t_front, 0)
    xp = (F.pad(xd, pads, mode="replicate") if pad == "replicate" else F.pad(xd, pads))[0].permute(1, 2, 3, 0)
    T, H, W = xp.shape[0] - kt + 1, x.shape[1], x.shape[2]
    wd = w.double()
    out = torch.zeros(T * H * W, w.shape[0], device=x.device, dtype=f64)
    for dt in range(kt):
        for dh in range(kh):
            for dw in range(kw):
                win = xp[dt:dt + T, dh:dh + H, dw:dw + W].reshape(-1, x.shape[3])
                out += win @ wd[:, (dt * kh + dh) * kw + dw].t()
    return (out + bias.double()).reshape(T, H, W, -1)


def upconv_ref(x, w4, bias):
    """nearest 2x + 3x3 conv as the four 2x2 sub-pixel convs of the folded operand w4 [4 (2 py + px), Cout, 4 taps (a, b), Cin], fp64:
    out[t, 2h + py, 2w + px] = sum_ab x[t, h + a - 1 + py, w + b - 1 + px] @ w4[2 py + px, :, 2 a + b]^T + bias (zero outside)."""
    T, H, W, C = x.shape
    xp = F.pad(x.double(), (0, 0, 1, 1, 1, 1))                                            # [T, H+2, W+2, C]
    out = torch.empty(T, H, 2, W, 2, w4.shape[1], device=x.device, dtype=f64)
    for py in range(2):
        for px in range(2):
            acc = torch.zeros(T * H * W, w4.shape[1], device=x.device, dtype=f64)
            for a in range(2):
                for b in range(2):
                    win = xp[:, a + py:a + py + H, b + px:b + px + W].reshape(-1, C)
                    acc += win @ w4[2 * py + px, :, 2 * a + b].double().t()
            out[:, :, py, :, px] = (acc + bias.double()).reshape(T, H, W, -1)
    return out.reshape(T, 2 * H, 2 * W, -1)


def norm_ref(raw, gamma):
    """silu(r / max(|r|, 1e-12) * sqrt(C) * gamma) in fp64 over the channels of r = raw rounded to bf16 (the kernel normalises the
    values it stores)."""
    r = raw.to(bf16).double()
    y = r / r.norm(dim=-1, keepdim=True).clamp_min(1e-12) * math.sqrt(r.shape[-1]) * gamma.double()
    return y * torch.sigmoid(y)


# ---------------------------------------------------------------------------------------------------------------- checks
def _elementwise_ratio(got, ref):
    """max over the elements of |got - ref| / (2^-8 |ref| + 2^-12 rms(ref)): one bf16 rounding (at most half an ulp = 2^-8 of the
    value) plus a floor for the fp32 accumulation where terms cancel; must be <= 1."""
    ref = ref.double()
    bound = ref.abs() * 2.0 ** -8 + float(ref.pow(2).mean().sqrt()) * 2.0 ** -12
    return float(((got.double() - ref).abs() / bound).max())


def _pixel_rel(got, ref):
    ref = ref.double()
    return float(((got.double() - ref).norm(dim=-1) / ref.norm(dim=-1).clamp_min(1e-30)).max())


def _ulp_key(t):
    """bf16 bit patterns as integers ordered like the values (+0 and -0 both 0): adjacent bf16 values differ by 1."""
    i = t.contiguous().view(torch.int16).int()
    return torch.where(i < 0, -(i & 0x7FFF), i)


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))


class _Guarded:
    """A bf16 tensor of `shape` inside a larger sentinel-filled buffer: GUARD elements in front, `tail` elements behind."""

    def __init__(self, shape, tail):
        n = math.prod(shape)
        self.n, self.tail = n, tail
        self.buf = torch.full((GUARD + n + tail,), SENTINEL, device="cuda", dtype=torch.int16)
        self.t = self.buf[GUARD:GUARD + n].view(bf16).view(shape)
        assert self.t.data_ptr() % 16 == 0 and self.t.data_ptr() % 128 != 0

    def check(self, label, untouched=None):
        """Guard bands bit-for-bit intact; no sentinel inside the tensor except where `untouched` (a bool mask) says it must stay."""
        b = self.buf
        assert bool((b[:GUARD] == SENTINEL).all()) and bool((b[GUARD + self.n:] == SENTINEL).all()), f"{label}: store outside the output"
        inside = self.t.view(torch.int16) == SENTINEL
        if untouched is None:
            assert not bool(inside.any()), f"{label}: {int(inside.sum())} output elements never written"
        else:
            assert torch.equal(inside, untouched), f"{label}: written elements differ from the expected ones"


_KERNEL_RE = re.compile(r"(\w+_tcgen05_kernel)<([^<>]*)>")


def _instances(names):
    """{(kernel, template args)} of the tcgen05 conv / GEMM kernels among demangled kernel names; bool arguments as 0 / 1."""
    out = set()
    for n in names:
        for m in _KERNEL_RE.finditer(n):
            args = tuple(int({"true": "1", "false": "0"}.get(a.strip(), a.strip())) for a in m.group(2).split(","))
            out.add((m.group(1), args))
    return out


def _profiled(fn):
    """Run fn under the CUDA profiler -> names of the launched kernels (the run must record some)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    names += [e.name() for e in prof.profiler.kineto_results.events() if e.device_type() == torch.autograd.DeviceType.CUDA]
    assert names, "the profiler recorded no CUDA kernel: dispatch cannot be checked"
    return names


def _ab_flags():
    return sorted(k for k in os.environ if k.startswith(("B200_CONV_", "B200_VAE_")))


# ---------------------------------------------------------------------------------------------------------------- the reference itself
def test_references_match_torch():
    """conv_ref against F.conv3d (zero / replicate padding) and upconv_ref + the _UpConv weight fold against nearest-exact 2x +
    F.conv2d, in fp64 on small shapes.  The up-sampling weights are multiples of 1/8 so the folded bf16 operand is exact."""
    from wan2gp_b200.wan.vae import _UpConv
    g = _gen(3)
    T, H, W, ci, co, k = 3, 5, 7, 16, 32, (3, 3, 3)
    x = torch.randn(T, H, W, ci, generator=g, device="cuda").to(bf16)
    w = torch.randn(co, ci, *k, generator=g, device="cuda").to(bf16)
    b = torch.randn(co, generator=g, device="cuda")
    wp = w.permute(0, 2, 3, 4, 1).reshape(co, 27, ci)
    xc = x.double().permute(3, 0, 1, 2)[None]
    for mode in ("zeros", "replicate"):
        xp = F.pad(xc, (1, 1, 1, 1, 2, 0), mode="replicate" if mode == "replicate" else "constant")
        ref = F.conv3d(xp, w.double(), b.double())[0].permute(1, 2, 3, 0)
        assert float((conv_ref(x, wp, b, k, mode) - ref).abs().max()) < 1e-9, mode
    xh = torch.randn(T + 2, H, W, ci, generator=g, device="cuda").to(bf16)             # history frames in front: valid in time
    ref = F.conv3d(F.pad(xh.double().permute(3, 0, 1, 2)[None], (1, 1, 1, 1, 0, 0)), w.double(), b.double())[0].permute(1, 2, 3, 0)
    assert float((conv_ref(xh, wp, b, k, t_front=0) - ref).abs().max()) < 1e-9
    w2 = torch.randint(-8, 9, (co, ci, 3, 3), generator=g, device="cuda").float() / 8
    up = _UpConv(w2, b, "cuda")
    ref = F.conv2d(F.interpolate(x.double().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest-exact"), w2.double(), b.double(), padding=1)
    assert float((upconv_ref(x, up.w4, b) - ref.permute(0, 2, 3, 1)).abs().max()) < 1e-9


# ---------------------------------------------------------------------------------------------------------------- the case table
@pytest.mark.parametrize("c", CASES, ids=[c.label.replace(" ", "_") for c in CASES])
def test_conv_kernel(c):
    from wan2gp_b200 import _lib
    from wan2gp_b200.hyvideo.vae import _RepConv
    from wan2gp_b200.wan.vae import _Conv, _UpConv, rms_silu
    H = _shape_h(c)
    T, W, ci, co = c.T, c.W, c.cin, c.cout
    seed = sum(map(ord, c.label))
    norm = c.entry.endswith("_norm")
    gamma = _per_channel(co, seed + 1, 0.25, 2.0)
    bias = _per_channel(co, seed + 2, -1.0, 1.0)
    r = _act((T, H, W, co), seed + 3) if c.residual else None
    rp = 0 if r is None else r.data_ptr()

    # ---- operands and the launch
    if c.entry == "upconv_norm":
        conv = _UpConv(_weights(co, ci, (3, 3), seed + 4), bias, "cuda")
        x = _act((T, H, W, ci), seed + 5)
        oshape = (T, 2 * H, 2 * W, co)
    elif c.entry == "timeconv":
        conv = _Conv(_weights(co, ci, c.k, seed + 4), bias, "cuda")
        x = _act((T, H, W, ci), seed + 5)
        oshape = (2 * T - 1, H, W, co // 2)
    else:
        conv = (_RepConv if c.entry == "repconv" else _Conv)(_weights(co, ci, c.k, seed + 4), bias, "cuda")
        x = _act((T + 2 if c.entry == "stream_norm" else T, H, W, ci), seed + 5)      # streaming: 2 non-zero history frames
        oshape = (T, H, W, co)
    tail = 2 * oshape[2] * oshape[3] * 2 + 4096                                        # more than one band of row tiles
    out = _Guarded(oshape, tail) if c.raw else None
    nrm = _Guarded(oshape, tail) if norm else None
    op, np_ = (0 if out is None else out.t.data_ptr()), (0 if nrm is None else nrm.t.data_ptr())
    xp = None
    if c.entry == "repconv":
        xp = torch.empty(T + 2, H + 2, W + 2, ci, device="cuda", dtype=bf16)
        _lib.call("b200_pad_replicate_cl", x.data_ptr(), xp.data_ptr(), T, H, W, ci, 2, 1, 1, _s())

    def launch():
        if c.entry == "conv_norm":
            _lib.call("b200_conv3d_cl_norm", x.data_ptr(), conv.w.data_ptr(), conv.b.data_ptr(), rp, op, np_, gamma.data_ptr(),
                      T, H, W, ci, co, *c.k, _s())
        elif c.entry == "upconv_norm":
            _lib.call("b200_upconv2x_cl_norm", x.data_ptr(), conv.w4.data_ptr(), conv.b.data_ptr(), op, np_, gamma.data_ptr(),
                      T, H, W, ci, co, _s())
        elif c.entry == "stream_norm":
            _lib.call("b200_conv3d_cl_stream", x.data_ptr(), conv.w.data_ptr(), conv.b.data_ptr(), rp, op, np_, gamma.data_ptr(),
                      T, H, W, ci, co, *c.k, 0, 0, _s())
        elif c.entry == "conv":
            conv(x, residual=r, out=out.t)
        elif c.entry == "repconv":
            conv.prepadded(xp, T, H, W, r, out.t, 0)
        elif c.entry == "timeconv":
            conv(x[1:], out=out.t, out_mode=1, t_off=1)                               # wan/vae.py _up: frame 0 is copied, not convolved

    names = _profiled(launch)
    got_inst = _instances(names)
    line = f"{c.label}: T={T} H={H} W={W} {ci}->{co}, {_tiles(c, H)} row tiles (pair threshold {2 * _num_sms()}), launched {sorted(got_inst)}"

    # ---- (a) dispatch
    flags = _ab_flags()
    if flags:
        print(f"{line}; dispatch not checked under {flags}")
    else:
        assert got_inst == {c.kernel}, f"{c.label}: expected {c.kernel}, launched {sorted(got_inst)}"

    # ---- (e) every output element written, nothing outside
    if out is not None:
        if c.entry == "timeconv":
            untouched = torch.zeros(oshape, dtype=torch.bool, device="cuda")
            untouched[0] = True
            out.check(c.label + " out", untouched)
        else:
            out.check(c.label + " out")
    if nrm is not None:
        nrm.check(c.label + " norm_out")

    # ---- (b) raw output vs fp64
    if c.entry == "upconv_norm":
        ref = upconv_ref(x, conv.w4, conv.b)
    elif c.entry == "timeconv":
        y = conv_ref(x[1:], conv.w, conv.b, c.k)                                       # [T-1, H, W, 2C], zero history
        C = co // 2
        ref = torch.stack([y[..., :C], y[..., C:]], 1).reshape(2 * T - 2, H, W, C)    # conv frame i -> frames 2i+1 ([0,C)), 2i+2 ([C,2C))
    else:
        ref = conv_ref(x, conv.w, conv.b, c.k, "replicate" if c.entry == "repconv" else "zeros",
                       t_front=0 if c.entry == "stream_norm" else None)
        if r is not None:
            ref = ref + r.double()
    if out is not None:
        got = out.t[1:] if c.entry == "timeconv" else out.t
        ratio, e = _elementwise_ratio(got, ref), rel_l2(got, ref)
        line += f"; raw: max |d|/bound {ratio:.3f}, rel-L2 {e:.3e}"

    # ---- (c) fused norm vs fp64
    if norm:
        nref = norm_ref(ref, gamma)
        pmax, ne = _pixel_rel(nrm.t, nref), rel_l2(nrm.t, nref)
        line += f"; norm: max per-pixel rel-L2 {pmax:.3e}, rel-L2 {ne:.3e}"

    # ---- (d) the fused kernel against the plain kernel + the separate norm pass
    if norm:
        if c.entry == "conv_norm":
            plain = conv(x, residual=r)
        elif c.entry == "upconv_norm":
            plain = conv(x)
        else:
            plain = torch.empty(oshape, device="cuda", dtype=bf16)
            _lib.call("b200_conv3d_cl_stream", x.data_ptr(), conv.w.data_ptr(), conv.b.data_ptr(), rp, plain.data_ptr(), 0, 0,
                      T, H, W, ci, co, *c.k, 0, 0, _s())
        sep = rms_silu(plain, gamma)
        dk = (_ulp_key(nrm.t) - _ulp_key(sep)).abs()
        ulp, flip = int(dk.max()), float((dk != 0).double().mean())
        same_raw = None if out is None else _bits_equal(out.t, plain)
        line += f"; vs plain: raw bit-identical {same_raw}, norm max {ulp} ulp, {flip:.2e} of elements differ"
    print(line)

    if out is not None:
        assert ratio <= 1.0 and e < 4e-3, line
    if norm:
        assert pmax < 1e-2 and ne < 4e-3, line
        assert same_raw is not False, line
        assert ulp <= 1 and flip < NORM_FLIP_FRAC, line


# ---------------------------------------------------------------------------------------------------------------- whole decode
def test_wanvae_decode_480p_9frames():
    """Whole Wan VAE decode of a [16,3,60,104] latent (9 frames at 480 x 832) vs the oracle evaluated on the GPU: the decode whose
    96- and 192-channel fused stages (widths 832 / 416) all have a ragged last row tile."""
    from oracle import vae_oracle
    from wan2gp_b200 import synth
    from wan2gp_b200.wan import WanVAE
    sd = synth.make_vae_state_dict(synth.VAE_CFG, 0)
    z = synth._normal((16, 3, 60, 104), 1.0, 7, "input.z480", "cpu")
    vae = WanVAE(device="cuda", state_dict=sd)
    got = vae.model.decode_frames(z.cuda(), vae.mean, vae.std)
    torch.cuda.synchronize()
    sdg = {k: v.cuda() for k, v in sd.items()}
    with torch.no_grad():
        mean, std = torch.tensor(synth.VAE_MEAN, device="cuda"), torch.tensor(synth.VAE_STD, device="cuda")
        ref_bf = vae_oracle.vae_decode(sdg, z.cuda(), mean, std, emulate_bf16=True)
        ref_32 = vae_oracle.vae_decode(sdg, z.cuda(), mean, std, emulate_bf16=False)
    assert got.shape == ref_32.shape == (3, 9, 480, 832)
    e_bf, p32 = rel_l2(got, ref_bf), psnr(got.clamp(-1, 1), ref_32.clamp(-1, 1), 2.0)
    u8 = (vae_oracle.frames_to_uint8(got).int() - vae_oracle.frames_to_uint8(ref_32).int()).abs()
    print(f"WanVAE decode 480p x 9f: rel-L2 vs bf16-emulating oracle {e_bf:.3e}, PSNR vs fp32 oracle {p32:.1f} dB, mean |d uint8| {float(u8.float().mean()):.3f}, max {int(u8.max())}")
    assert e_bf < 2.5e-2 and p32 > 35.0 and float(u8.float().mean()) < 1.5
