"""Every compiled gemm_s8_kernel instantiation (and the stem's conv_rows_s8_kernel), in every operand mode that can
reach it, against an evaluation that shares nothing with the kernels:

    acc = float64 matmul / conv2d of the int8 operands on the GPU, rounded to int64       exact: |acc| < 2^53
    y   = clamp(clamp(RightShift(acc, rs)) + b) [ReLU], fp32 = y / 2^ob                   new_quantity_op.py:11-44,124-133
    add = clamp(y / 2^ob + sc / 2^sbit, -128, 127) [ReLU] exactly; int16 = add * 2^o_bit, int8 = Quantity(q_bit)(add)

Each row of ROWS names the C entry point, the geometry and the instantiation the launch must land on (checked with
torch.profiler); every row runs every epilogue variant its kernel can select (folded bias with and without the fused
ReLU, classic shift, rs <= 0, the generic fp32 / unstaged int8 body, the fused add at its bit limits).  Every output is
written into the middle of a sentinel-filled buffer, and the bytes around it must survive.
"""
import ctypes
import re
import shutil
import subprocess
import zlib

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

# ------------------------------------------------------------------------------------------ instantiation table
# (BN, BK, STAGES, ADDK, BSLOTS) of every gemm_s8_kernel the library compiles (pq_gemm_s8.cu: launch_bn, conv_impl).
PLAIN = [(bn, bk, st, 0, st) for bn, row in ((32, (8, 9, 9)), (64, (8, 9, 9)), (128, (6, 9, 9)), (256, (4, 8, 9)))
         for bk, st in zip((128, 64, 32), row)]
DEEP_A = (64, 64, 18, 0, 9)          # short-K 3x3 im2col (C = 64, N <= 64), and the patch windows of C = 64
WIN128 = (128, 128, 3, 0, 9)         # patch windows of C = 128
ADDK = [(bn, bk, st, 1, st) for bn, row in ((64, (6, 8, 8)), (128, (4, 8, 8)), (256, (3, 6, 8)))
        for bk, st in zip((128, 64, 32), row)]
INSTANTIATIONS = sorted(PLAIN + [DEEP_A, WIN128] + ADDK)
ROWS_KERNEL = "conv_rows_s8_kernel"

# One row per reachable (instantiation, operand mode) pair.  Fields: entry point, operand mode, instantiation, geometry:
#   gemm:   pq_gemm_s8 [M][K] x [N][K]; M is the smallest ragged M (128 * m_tiles - 37) for which pick_bn chooses BN
#   conv:   pq_conv2d_s8 over NHWC (C, N filters, R x R, stride, pad R // 2, H = W = hw); the batch is the smallest for
#           which pick_bn chooses BN; stride 2 (or C % 64 != 0) keeps 3x3 layers off the patch windows
#   add:    pq_conv2d_s8_add, the same geometry (1x1 stride 1 = its GEMM form, H = W = 1); the add needs BN >= 64
#   win:    pq_conv2d_s8 3x3 / stride 1 / pad 1 patch windows (no pick_bn: C = 64 -> DEEP_A, C = 128 -> WIN128)
#   smallc: pq_conv2d_smallc_s8 (8-byte pixels, BK = 64): stride_w 4 takes the window kernel (a_im2col == 2, B never
#           resident), stride_w 2 the row kernel
# Unreachable pairs: DEEP_A needs im2col taps (a_im2col == 1) or patch windows, so it has no GEMM / small-channel row;
# WIN128 exists only for patch windows; the small-channel window kernel always has BK = 64 and no fused add; patch
# windows never fuse the add (conv_impl skips them when an add is requested).
ROWS = [
    # GEMM (A is a plain 2-D tile source)
    ("gemm", "gemm", (32, 128, 8, 0, 8), dict(N=32, K=1152)),          # num_kb 9 > BSLOTS: B streamed
    ("gemm", "gemm", (32, 64, 9, 0, 9), dict(N=32, K=96)),
    ("gemm", "gemm", (32, 32, 9, 0, 9), dict(N=16, K=48)),             # second K block half outside K
    ("gemm", "gemm", (64, 128, 8, 0, 8), dict(N=48, K=256)),
    ("gemm", "gemm", (64, 64, 9, 0, 9), dict(N=64, K=64)),
    ("gemm", "gemm", (64, 32, 9, 0, 9), dict(N=48, K=32)),
    ("gemm", "gemm", (128, 128, 6, 0, 6), dict(N=112, K=896)),         # num_kb 7 > 6
    ("gemm", "gemm", (128, 64, 9, 0, 9), dict(N=128, K=80)),
    ("gemm", "gemm", (128, 32, 9, 0, 9), dict(N=96, K=32)),
    ("gemm", "gemm", (256, 128, 4, 0, 4), dict(N=272, K=128)),         # two n tiles, the second ragged
    ("gemm", "gemm", (256, 64, 8, 0, 8), dict(N=256, K=64)),
    ("gemm", "gemm", (256, 32, 9, 0, 9), dict(N=208, K=16)),
    ("gemm", "gemm", (64, 128, 8, 0, 8), dict(N=40, K=128)),           # N % 16 != 0: no staged store, no fold
    ("add", "gemm", (64, 128, 6, 1, 6), dict(C=128, N=48, R=1, stride=1, hw=1)),
    ("add", "gemm", (64, 64, 8, 1, 8), dict(C=64, N=64, R=1, stride=1, hw=1)),
    ("add", "gemm", (64, 32, 8, 1, 8), dict(C=32, N=32, R=1, stride=1, hw=1)),
    ("add", "gemm", (128, 128, 4, 1, 4), dict(C=640, N=128, R=1, stride=1, hw=1)),   # num_kb 5 > 4
    ("add", "gemm", (128, 64, 8, 1, 8), dict(C=64, N=96, R=1, stride=1, hw=1)),
    ("add", "gemm", (128, 32, 8, 1, 8), dict(C=48, N=112, R=1, stride=1, hw=1)),
    ("add", "gemm", (256, 128, 3, 1, 3), dict(C=256, N=272, R=1, stride=1, hw=1)),   # N > BN
    ("add", "gemm", (256, 64, 6, 1, 6), dict(C=96, N=256, R=1, stride=1, hw=1)),
    ("add", "gemm", (256, 32, 8, 1, 8), dict(C=32, N=176, R=1, stride=1, hw=1)),
    # im2col-TMA
    ("conv", "im2col", (32, 128, 8, 0, 8), dict(C=128, N=32, R=3, stride=2, hw=26)),  # num_kb 9 > 8
    ("conv", "im2col", (32, 64, 9, 0, 9), dict(C=64, N=32, R=3, stride=2, hw=26)),
    ("conv", "im2col", (32, 32, 9, 0, 9), dict(C=32, N=16, R=5, stride=2, hw=26)),    # num_kb 25 > 9
    ("conv", "im2col", (32, 32, 9, 0, 9), dict(C=32, N=24, R=3, stride=1, hw=13)),    # N % 16 != 0
    ("conv", "im2col", (64, 128, 8, 0, 8), dict(C=256, N=64, R=1, stride=2, hw=26)),
    ("conv", "im2col", (64, 64, 9, 0, 9), dict(C=64, N=96, R=3, stride=2, hw=26)),    # N > 64: not deep-A
    ("conv", "im2col", (64, 32, 9, 0, 9), dict(C=96, N=48, R=3, stride=2, hw=26)),
    ("conv", "im2col", DEEP_A, dict(C=64, N=48, R=3, stride=2, hw=26)),
    ("conv", "im2col", (128, 128, 6, 0, 6), dict(C=128, N=128, R=3, stride=2, hw=26)),  # num_kb 9 > 6
    ("conv", "im2col", (128, 64, 9, 0, 9), dict(C=64, N=112, R=1, stride=2, hw=26)),
    ("conv", "im2col", (128, 32, 9, 0, 9), dict(C=32, N=80, R=3, stride=1, hw=13)),
    ("conv", "im2col", (256, 128, 4, 0, 4), dict(C=128, N=256, R=1, stride=2, hw=26)),
    ("conv", "im2col", (256, 64, 8, 0, 8), dict(C=64, N=208, R=3, stride=2, hw=26)),
    ("conv", "im2col", (256, 32, 9, 0, 9), dict(C=32, N=256, R=3, stride=2, hw=26)),
    ("add", "im2col", (64, 128, 6, 1, 6), dict(C=128, N=64, R=3, stride=2, hw=26)),   # num_kb 9 > 6
    ("add", "im2col", (64, 64, 8, 1, 8), dict(C=64, N=48, R=3, stride=1, hw=13)),
    ("add", "im2col", (64, 32, 8, 1, 8), dict(C=32, N=32, R=1, stride=2, hw=26)),
    ("add", "im2col", (128, 128, 4, 1, 4), dict(C=128, N=128, R=1, stride=2, hw=26)),
    ("add", "im2col", (128, 64, 8, 1, 8), dict(C=64, N=96, R=3, stride=2, hw=26)),
    ("add", "im2col", (128, 32, 8, 1, 8), dict(C=96, N=128, R=3, stride=2, hw=26)),
    ("add", "im2col", (256, 128, 3, 1, 3), dict(C=256, N=256, R=1, stride=2, hw=26)),
    ("add", "im2col", (256, 64, 6, 1, 6), dict(C=64, N=272, R=3, stride=2, hw=26)),   # N > BN
    ("add", "im2col", (256, 32, 8, 1, 8), dict(C=32, N=144, R=3, stride=2, hw=26)),
    # small-channel windows (a_im2col == 2): P x Q = 20 x 24 output pixels = 3 x 2 ragged 8 x 16 patches per image
    ("smallc", "smallc", (32, 64, 9, 0, 9), dict(N=32, R=3, S=3, stride=(1, 4))),
    ("smallc", "smallc", (64, 64, 9, 0, 9), dict(N=64, R=3, S=5, stride=(1, 4))),
    ("smallc", "smallc", (128, 64, 9, 0, 9), dict(N=128, R=2, S=8, stride=(2, 4))),
    ("smallc", "smallc", (256, 64, 8, 0, 8), dict(N=256, R=3, S=3, stride=(1, 4))),
    # patch windows (a_im2col == 3)
    ("conv", "win", DEEP_A, dict(C=64, N=64, R=3, stride=1, hw=(21, 30), batch=2)),
    ("conv", "win", WIN128, dict(C=128, N=80, R=3, stride=1, hw=(13, 9), batch=3)),
    # the stem's row kernel
    ("smallc", "rows", ROWS_KERNEL, dict(N=64, R=7, S=7, stride=(2, 2))),
]


def row_id(r):
    inst = r[2] if isinstance(r[2], str) else "bn%d_bk%d_s%d%s_b%d" % (r[2][0], r[2][1], r[2][2], "_add" if r[2][3] else "",
                                                                        r[2][4])
    g = r[3]
    return "%s-%s-%s-n%d" % (r[1], r[0], inst, g["N"]) + ("-r%d" % g["R"] if "R" in g else "")


def pick_bn(m, n, sms):
    """pq_gemm_s8.cu pick_bn: the widest tile that leaves every SM two tiles, never wider than N needs."""
    mt = -(-m // 128)
    cap = 256 if n > 128 else (128 if n > 64 else (64 if n > 32 else 32))
    bn = cap
    while bn > 32:
        if mt * -(-n // bn) >= 2 * sms:
            return bn
        bn //= 2
    return 64 if cap > 32 and mt * -(-n // 64) >= sms else 32


def parse_instantiation(name):
    """(BN, BK, STAGES, ADDK, BSLOTS) from a demangled gemm_s8_kernel name, either spelling ("(int)128, (bool)1" as
    cu++filt prints it, or "128, true")."""
    m = re.search(r"gemm_s8_kernel<([^>]*)>", name)
    if not m:
        return None
    vals = []
    for a in m.group(1).split(","):
        a = re.sub(r"\((int|bool)\)", "", a).strip()
        vals.append({"true": 1, "false": 0}[a] if a in ("true", "false") else int(a))
    return tuple(vals)


# ------------------------------------------------------------------------------------------ the exact reference
def right_shift(acc, rs):
    """new_quantity_op.py:11-44 on int64 accumulators: round half away from zero for rs >= 1, else clamp then scale."""
    if rs >= 1:
        half = 1 << (rs - 1)
        r = torch.where(acc >= 0, (acc + half) >> rs, -((half - acc) >> rs))
    else:
        r = acc.clamp(-128, 127) << (-rs)
    return r.clamp(-128, 127)


def epilogue_ref(acc, bias, rs, relu):
    """int64 [M][N] accumulators, int64 [N] bias -> the int8-valued layer output (RightShift, BiasAdd, Sp[, ReLU])."""
    y = (right_shift(acc, rs) + bias.view(1, -1)).clamp(-128, 127)
    return y.clamp(min=0) if relu else y


def dequant_ref(y, ob):
    return (y.double() * 2.0 ** -ob).float()          # exact: |y| <= 128 and 2^-ob is a normal float for |ob| <= 100


def round_half_even_shift(v, d):
    """round_half_even(v / 2^d) for int64 v and d >= 1."""
    t = v >> d
    rem = v - (t << d)
    half = 1 << (d - 1)
    return t + ((rem > half) | ((rem == half) & ((t & 1) == 1))).long()


def add_ref(y, ob, sc, sbit, sc_relu, out_relu, q_bit):
    """NewAdd (+ the nn.ReLU after it) of the convolution output y at bit ob and the shortcut sc at bit sbit, exactly:
    (int16 sum at o_bit = max(ob, sbit), int8 Quantity(q_bit) of it)."""
    o = max(ob, sbit)
    s = sc.clamp(min=0) if sc_relu else sc
    total = ((y << (o - ob)) + (s << (o - sbit))).clamp(-128 << o, 127 << o)
    if out_relu:
        total = total.clamp(min=0)
    q8 = total << (q_bit - o) if q_bit >= o else round_half_even_shift(total, o - q_bit)
    return total, q8.clamp(-128, 127)


def exact_gemm(a, w):
    acc = F.linear(a.double(), w.double())
    assert float(acc.abs().max()) < 2.0 ** 53
    return torch.round(acc).long()


def exact_conv(x_nhwc, w_krsc, stride, pad):
    acc = F.conv2d(x_nhwc.permute(0, 3, 1, 2).double(), w_krsc.permute(0, 3, 1, 2).double(), None, stride, pad)
    assert float(acc.abs().max()) < 2.0 ** 53
    return torch.round(acc).long().permute(0, 2, 3, 1).reshape(-1, w_krsc.shape[0])


# ------------------------------------------------------------------------------------------ launches through ctypes
SENTINEL = 0xA5
GUARD = 512                    # bytes on either side; a multiple of 16, so the output keeps the staged store's alignment


class Guarded:
    """An output tensor in the middle of a sentinel-filled buffer (skew: extra bytes in front, breaking alignment)."""

    def __init__(self, shape, dtype, skew=0):
        n = 1
        for s in shape:
            n *= s
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        self.buf = torch.full((nbytes + 2 * GUARD + 16,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.lo, self.hi = GUARD + skew, GUARD + skew + nbytes
        self.t = self.buf[self.lo:self.hi].view(dtype).view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        assert bool((self.buf[:self.lo] == SENTINEL).all()), "%s: bytes before the output were overwritten" % what
        assert bool((self.buf[self.hi:] == SENTINEL).all()), "%s: bytes after the output were overwritten" % what


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _flags(bias, n, relu):
    from common.quantity import _native
    return (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias.numel() == 3 * n else 0)


class Case:
    """Operands, exact accumulator and output geometry of one row."""

    def __init__(self, row, sms):
        from common.quantity import _native
        self.entry, self.mode, self.inst, g = row
        self.N = g["N"]
        gen = torch.Generator(device="cuda").manual_seed(zlib.crc32(row_id(row).encode()))
        self.gen = gen
        if self.entry == "gemm":
            K, bn = g["K"], self.inst[0]
            self.M = next(m for m in (128 * t - 37 if t > 1 else 91 for t in range(1, 8 * sms))
                          if pick_bn(m, self.N, sms) == bn)
            self.a = self._activations((self.M, K))
            self.w = self._weights(self.N, K)
            self.acc = exact_gemm(self.a, self.w)
            self.hw = 1
        elif self.entry in ("conv", "add"):
            C, R, st = g["C"], g["R"], g["stride"]
            pad = R // 2
            H, W = (g["hw"], g["hw"]) if isinstance(g["hw"], int) else g["hw"]
            P, Q = _native.conv_out_size((H, W), (R, R), (st, st), (pad, pad))
            if "batch" in g:
                B = g["batch"]
            else:
                bn = self.inst[0]
                fits = (lambda m: max(pick_bn(m, self.N, sms), 64) == bn) if self.entry == "add" else \
                    (lambda m: pick_bn(m, self.N, sms) == bn)
                B = next(b for b in range(-(-91 // (P * Q)), 1 << 20) if fits(b * P * Q))
            self.x = self._activations((B, H, W, C))
            self.w = self._weights(self.N, R * R * C).view(self.N, R, R, C)
            self.acc = exact_conv(self.x, self.w, st, pad)
            self.desc = lambda rs, ob: _native.ConvDesc(B, H, W, C, self.N, R, R, st, st, pad, pad, P, Q, rs, ob, 1, 1)
            self.M, self.nchw, self.hw = B * P * Q, (B, self.N, P, Q), P * Q
        else:                                        # smallc: the padded 8-byte-pixel image itself is the operand
            R, S, (sh, sw) = g["R"], g["S"], g["stride"]
            if self.mode == "rows":
                B, P, Q = 2, 20, 20
            else:
                P, Q = 20, 24
                per_img = -(-P // 8) * -(-Q // 16)
                B = next(b for b in range(1, 1 << 20) if pick_bn(b * per_img * 128, self.N, sms) == self.inst[0])
            Hp = -(-((P - 1) * sh + R) // sh) * sh
            Wp = ((Q - 1) * sw + 8 + 1) // 2 * 2
            self.xp = self._activations((B, Hp, Wp, 8))
            wk = self._weights(self.N, R * 64).view(self.N, R, 8, 8)         # [K][R][pixel slot s][channel]
            wk[:, :, S:, :] = 0                                              # slots s >= S are zero by contract
            self.w = wk.reshape(self.N, R, 64).contiguous()
            acc = F.conv2d(self.xp.permute(0, 3, 1, 2).double(), wk.permute(0, 3, 1, 2).double(), None, (sh, sw))
            acc = torch.round(acc[:, :, :P, :Q]).long()
            self.acc = acc.permute(0, 2, 3, 1).reshape(-1, self.N)
            # image = the padded image without padding: H = Hp, W chosen so that nn.Conv2d arithmetic gives Q
            H, W = Hp, (Q - 1) * sw + S
            self.Hp, self.Wp = Hp, Wp
            self.desc = lambda rs, ob: _native.ConvDesc(B, H, W, 8, self.N, R, S, sh, sw, 0, 0, P, Q, rs, ob, 1, 1)
            self.M, self.nchw, self.hw = B * P * Q, (B, self.N, P, Q), P * Q
        b = torch.randint(-128, 128, (self.N,), generator=gen, device="cuda", dtype=torch.int32)
        b[:4] = torch.tensor([-128, -1, 0, 127], dtype=torch.int32)
        self.bias = b
        self.max_acc = int(self.acc.abs().max())

    def _activations(self, shape):
        x = torch.randint(-128, 128, shape, generator=self.gen, device="cuda", dtype=torch.int8)
        px = x.view(-1, shape[-1])                    # one row per pixel
        k = max(1, px.shape[0] // 16)
        px[:k] = 127                                  # coherent extremes: the largest accumulators of the layer
        px[k:2 * k] = -128
        px[2 * k:3 * k] = 0
        return x

    def _weights(self, n, k):
        """Per-channel magnitude (0 .. 127), sign coherence and sparsity, so |acc| spans 0 .. max across channels."""
        w = torch.randint(-128, 128, (n, k), generator=self.gen, device="cuda", dtype=torch.int32)
        mags = torch.tensor([0, 1, 3, 15, 127, 128, 40, 7], device="cuda", dtype=torch.int32)
        ch = torch.arange(n, device="cuda")
        w = torch.div(w * mags[ch % 8].view(-1, 1), 128, rounding_mode="floor")
        coherent = (ch % 3 == 1).view(-1, 1)
        w = torch.where(coherent, w.abs().clamp(max=127), w)
        sparse = (ch % 5 == 2).view(-1, 1) & (torch.arange(k, device="cuda").view(1, -1) > 0)
        w = torch.where(sparse, torch.zeros_like(w), w)
        return w.to(torch.int8).contiguous()

    # -------------------------------------------------------------------------------------- launches
    def run(self, rs, ob, bias, relu, out):
        """One launch of the row's entry point; returns (fp32 as [M][N] or None, int8 [M][N] or None)."""
        from common.quantity import _native
        lib = _native.lib()
        f32 = Guarded(self.nchw if self.hw > 1 else (self.M, self.N), torch.float32) if out in ("f32", "both") else None
        s8 = Guarded((self.M, self.N), torch.int8, skew=1 if out == "s8u" else 0) if out in ("s8", "s8u", "both") else None
        fp = f32.ptr() if f32 else None
        sp = s8.ptr() if s8 else None
        flags = _flags(bias, self.N, relu)
        if self.entry == "gemm":
            rc = lib.pq_gemm_s8(self.a.data_ptr(), self.w.data_ptr(), bias.data_ptr(), self.M, self.N, self.a.shape[1],
                                rs, ob, 1, flags, fp, sp, _stream())
        elif self.entry == "conv":
            d = self.desc(rs, ob)
            flags |= _native.FLAG_NO_WINDOWS if self.mode == "im2col" else 0
            rc = lib.pq_conv2d_s8(self.x.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(d), flags, fp, sp,
                                  _stream())
        else:
            d = self.desc(rs, ob)
            rc = lib.pq_conv2d_smallc_s8(self.xp.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(d),
                                         self.Hp, self.Wp, flags, fp, sp, _stream())
        assert rc == 0, "launch failed: %s" % lib.pq_error_string(rc).decode()
        torch.cuda.synchronize()
        for g, name in ((f32, "fp32"), (s8, "int8")):
            if g is not None:
                g.check(name)
        f = None
        if f32 is not None:
            f = f32.t.permute(0, 2, 3, 1).reshape(self.M, self.N) if self.hw > 1 else f32.t
        return f, (s8.t if s8 is not None else None)

    def run_add(self, rs, ob, bias, sc, sbit, sc_relu, q_bit, out_relu, want16):
        from common.quantity import _native
        lib = _native.lib()
        o16 = Guarded((self.M, self.N), torch.int16) if want16 else None
        o8 = Guarded((self.M, self.N), torch.int8)
        add = _native.AddDesc(sc.data_ptr(), 1 if sc.dtype == torch.int16 else 0, sbit, int(sc_relu), int(out_relu), q_bit,
                              o16.ptr() if o16 else None, o8.ptr())
        d = self.desc(rs, ob)
        rc = lib.pq_conv2d_s8_add(self.x.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(d),
                                  ctypes.byref(add), _flags(bias, self.N, False), _stream())
        assert rc == 0, "launch failed: %s" % lib.pq_error_string(rc).decode()
        torch.cuda.synchronize()
        o8.check("int8")
        if o16:
            o16.check("int16")
        return (o16.t if o16 else None), o8.t

    def bias_for(self, kind, rs):
        """'plain': int32 [N]; 'fold': the [3N] folded buffer (PQ_FLAG_BIAS_FOLDED).  Outside 1 <= rs <= 20 the library
        ignores the fold and reads the plain bias at the front of the buffer, which is what rs in 21..24 checks."""
        from common.quantity import _native
        if kind == "plain":
            return self.bias
        return _native.bias_fold(self.bias, min(max(rs, 1), 20))


def launched_kernels(fn):
    """Names of the gemm_s8 / conv_rows kernels that ran during fn()."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "gemm_s8_kernel" in e.name or ROWS_KERNEL in e.name]


def check_landing(case, fn):
    names = launched_kernels(fn)
    assert len(names) == 1, names
    if case.inst == ROWS_KERNEL:
        assert ROWS_KERNEL in names[0], names
    else:
        assert parse_instantiation(names[0]) == case.inst, (names[0], case.inst)


def assert_not_degenerate(case, rs, y, relu, what):
    """The variant exercised its shift and both saturations: the int8 output has interior values and (without a ReLU)
    both -128 and 127, the shift itself is not all zero wherever the accumulators reach 2^rs, and not everything
    saturates."""
    interior = (y > -128) & (y < 127)
    assert bool(interior.any()), what
    if not relu:
        assert bool((y == -128).any()) and bool((y == 127).any()), what
    r = right_shift(case.acc, rs)
    if rs >= 1 and case.max_acc >= 1 << rs:
        assert bool(((r != 0) & (r > -128) & (r < 127)).any()), what
    if rs <= 0:                                    # the clamp before the scaling: zero and both saturations
        assert bool((r == 0).any()) and bool((r == 127).any()) and bool((r == -128).any()), what
    assert float((~interior).float().mean()) < 0.9, what


# (rs, ob, bias, relu, outputs): 's8' int8 only (staged TMA store when N % 16 == 0), 's8u' int8 only from an address
# one byte off 16-byte alignment (unstaged, the generic body), 'f32' fp32 only, 'both' fp32 + int8 (generic body).
# Every rs class of the epilogue dispatch appears, every ob appears with an fp32 output (int8 does not depend on ob).
PLAIN_VARIANTS = [
    (1, 0, "fold", False, "s8"),         # FOLD = 1
    (7, 0, "fold", True, "s8"),          # FOLD = 2
    (13, 0, "fold", False, "s8"),
    (20, 0, "fold", True, "s8"),
    (2, 0, "plain", False, "s8"),        # classic POS, FAST
    (21, 0, "fold", False, "s8"),        # the fold is ignored above rs 20: classic POS, FAST
    (24, 0, "fold", True, "s8"),
    (0, 0, "plain", False, "s8"),        # POS = false, FAST
    (-1, 0, "fold", True, "s8"),
    (-8, -100, "plain", False, "f32"),   # generic body
    (-24, -3, "plain", False, "both"),
    (7, 0, "fold", False, "f32"),
    (13, 4, "plain", True, "both"),
    (24, 100, "plain", False, "both"),
    (1, 100, "fold", False, "f32"),
    (2, 4, "plain", False, "s8u"),
    (-1, 4, "plain", True, "s8u"),
    (20, -100, "fold", True, "s8u"),
]

# (rs, bias, conv ob, shortcut bit, q_bit, int16 shortcut, shortcut ReLU, output ReLU, want int16).  o_bit = max(ob, sbit)
# must be 0..7 with a span <= 7, so the plain epilogue's ob = +-100 has no fused-add counterpart.
ADD_VARIANTS = [
    (7, "fold", 4, 4, 4, False, False, True, True),       # same bit: packed folded saturation, FASTQ
    (13, "fold", 0, 0, 0, True, False, False, True),      # o_bit 0
    (1, "fold", 7, 7, 7, False, True, False, False),      # o_bit 7
    (20, "fold", 7, 0, 22, True, False, False, True),     # span 7, conv finer; q - o = 15
    (2, "fold", 0, 7, -8, False, False, True, True),      # span 7, shortcut finer (conv scaled by 2^7); q - o = -15
    (7, "fold", -3, 4, 3, True, True, True, True),        # negative conv ob; q - o = -1
    (7, "plain", 5, 3, 6, False, False, False, True),     # POS with a plain bias; q - o = 1
    (21, "fold", 3, 3, 3, True, False, True, False),      # fold ignored above rs 20
    (24, "fold", 3, 5, 5, False, True, False, True),
    (0, "plain", 4, 6, 6, False, False, False, True),     # POS = false
    (-1, "plain", 6, 2, 6, True, True, True, True),
    (-8, "plain", 2, 2, 2, False, False, False, False),
    (-24, "plain", 7, 1, 0, True, False, False, True),
]


def shortcut(case, is16, sbit):
    if is16:
        sc = torch.randint(-128 << sbit, (127 << sbit) + 1, (case.M, case.N), generator=case.gen, device="cuda",
                           dtype=torch.int32).to(torch.int16)
    else:
        sc = torch.randint(-128, 128, (case.M, case.N), generator=case.gen, device="cuda", dtype=torch.int8)
    lim = (127 << sbit) if is16 else 127
    sc.view(-1)[:4] = torch.tensor([-lim - (1 << sbit if is16 else 1), lim, 0, -1], dtype=sc.dtype)
    return sc


_SMS = []


def sms():
    if not _SMS:
        _SMS.append(torch.cuda.get_device_properties(0).multi_processor_count)
    return _SMS[0]


@gpu
@pytest.mark.parametrize("row", ROWS, ids=[row_id(r) for r in ROWS])
def test_every_instantiation_and_epilogue_vs_exact_evaluation(row):
    case = Case(row, sms())
    if case.entry != "add":
        check_landing(case, lambda: case.run(7, 0, case.bias, False, "s8"))
        for rs, ob, kind, relu, out in PLAIN_VARIANTS:
            what = "rs=%d ob=%d %s relu=%s %s" % (rs, ob, kind, relu, out)
            want = epilogue_ref(case.acc, case.bias.long(), rs, relu)
            f32, s8 = case.run(rs, ob, case.bias_for(kind, rs), relu, out)
            if s8 is not None:
                assert torch.equal(s8.long(), want), what
            if f32 is not None:
                assert torch.equal(f32, dequant_ref(want, ob)), what
            assert_not_degenerate(case, rs, want, relu, what)
        return
    sc_cache = {}
    for i, (rs, kind, ob, sbit, q, is16, sc_relu, out_relu, want16) in enumerate(ADD_VARIANTS):
        what = "rs=%d %s ob=%d sbit=%d q=%d sc16=%s sc_relu=%s relu=%s want16=%s" % (
            rs, kind, ob, sbit, q, is16, sc_relu, out_relu, want16)
        sc = sc_cache.setdefault((is16, sbit), shortcut(case, is16, sbit))
        bias = case.bias_for(kind, rs)
        if i == 0:
            check_landing(case, lambda: case.run_add(rs, ob, bias, sc, sbit, sc_relu, q, out_relu, want16))
        y = epilogue_ref(case.acc, case.bias.long(), rs, False)
        want16_, want8 = add_ref(y, ob, sc.long(), sbit, sc_relu, out_relu, q)
        o16, o8 = case.run_add(rs, ob, bias, sc, sbit, sc_relu, q, out_relu, want16)
        assert torch.equal(o8.long(), want8), what
        if want16:
            assert torch.equal(o16.long(), want16_), what
        assert_not_degenerate(case, rs, y, False, what)


# ------------------------------------------------------------------------------------------ crafted ties
TIE_K, TIE_N = 16384, 16
TIE_LIMIT = (TIE_K - 2) * 127 * 127                 # largest |acc| the construction below reaches


def tie_operands(rs):
    """A GEMM whose accumulators sit exactly at (j + 1/2) * 2^rs (and one either side) for j near 0 and at both
    saturation edges, both signs, as far as |acc| <= TIE_LIMIT allows.  Every filter is 127 x (K - 1) then 1, so an
    activation row of q // 127 entries of +-127, one entry of +-(q % 127) and a last entry r gives 127 q + r."""
    targets = []
    for j in (-3, -2, -1, 0, 1, 2, 125, 126, 127, 128, -126, -127, -128, -129):
        t = (2 * j + 1) << (rs - 1)
        for d in ((0,) if rs == 1 else (-1, 0, 1)):
            if abs(t + d) <= TIE_LIMIT:
                targets.append(t + d)
    a = torch.zeros((len(targets), TIE_K), dtype=torch.int8)
    for i, t in enumerate(targets):
        q, r = divmod(t, 127)
        sgn, mag = (1 if q >= 0 else -1), abs(q)
        n127 = mag // 127
        a[i, :n127] = 127 * sgn
        a[i, n127] = (mag % 127) * sgn
        a[i, TIE_K - 1] = r
    w = torch.full((TIE_N, TIE_K), 127, dtype=torch.int8)
    w[:, TIE_K - 1] = 1
    return a.cuda(), w.cuda(), torch.tensor(targets, dtype=torch.int64, device="cuda")


@gpu
@pytest.mark.parametrize("rs", range(1, 25))
def test_crafted_ties_and_folded_bounds(rs):
    """Round half away from zero at exact ties of both signs, the saturation edges around 127.5 and -128.5 * 2^rs, and
    the folded bounds h = 127 + min(b, 0), l = -128 + max(b, 0) for b in {-128, -1, 0, 127}: through the plain epilogue
    (classic, folded, folded + ReLU, fp32) and the fused-add epilogue (folded with and without the conv-side scaling,
    classic)."""
    from common.quantity import _native
    lib = _native.lib()
    a, w, targets = tie_operands(rs)
    M = a.shape[0]
    acc = exact_gemm(a, w)
    assert torch.equal(acc, targets.view(-1, 1).expand(M, TIE_N))
    bias = torch.tensor([-128, -1, 0, 127] * (TIE_N // 4), dtype=torch.int32, device="cuda")
    kinds = [("plain", bias)] + [("fold", _native.bias_fold(bias, min(rs, 20)))]
    for kind, bq in kinds:
        for relu in (False, True):
            want = epilogue_ref(acc, bias.long(), rs, relu)
            for out in ("s8", "f32"):
                g = Guarded((M, TIE_N), torch.int8 if out == "s8" else torch.float32)
                rc = lib.pq_gemm_s8(a.data_ptr(), w.data_ptr(), bq.data_ptr(), M, TIE_N, TIE_K, rs, -2, 1,
                                    _flags(bq, TIE_N, relu), g.ptr() if out == "f32" else None,
                                    g.ptr() if out == "s8" else None, _stream())
                assert rc == 0
                torch.cuda.synchronize()
                g.check(out)
                got = g.t.long() if out == "s8" else g.t
                assert torch.equal(got, want if out == "s8" else dequant_ref(want, -2)), (kind, relu, out)
        # fused add with a zero shortcut: the int16 sum is the convolution result itself, scaled to o_bit
        y = epilogue_ref(acc, bias.long(), rs, False)
        x = a.view(M, 1, 1, TIE_K)
        wk = w.view(TIE_N, 1, 1, TIE_K)
        for ob, sbit in ((4, 4), (0, 3)):                 # add_cshift 0 (packed saturation) and 3
            sc = torch.zeros((M, TIE_N), dtype=torch.int8, device="cuda")
            o16, o8 = Guarded((M, TIE_N), torch.int16), Guarded((M, TIE_N), torch.int8)
            add = _native.AddDesc(sc.data_ptr(), 0, sbit, 0, 0, max(ob, sbit), o16.ptr(), o8.ptr())
            d = _native.ConvDesc(M, 1, 1, TIE_K, TIE_N, 1, 1, 1, 1, 0, 0, 1, 1, rs, ob, 1, 1)
            rc = lib.pq_conv2d_s8_add(x.data_ptr(), wk.data_ptr(), bq.data_ptr(), ctypes.byref(d), ctypes.byref(add),
                                      _flags(bq, TIE_N, False), _stream())
            assert rc == 0
            torch.cuda.synchronize()
            o16.check("int16"), o8.check("int8")
            w16, w8 = add_ref(y, ob, sc.long(), sbit, False, False, max(ob, sbit))
            assert torch.equal(o16.t.long(), w16), (kind, ob, sbit)
            assert torch.equal(o8.t.long(), w8), (kind, ob, sbit)


# ------------------------------------------------------------------------------------------ argument limits
@gpu
def test_one_step_beyond_each_limit_is_unsupported_and_writes_nothing():
    """The fused add's bit limits (o_bit 0..7, span <= 7, |q_bit - o_bit| <= 15) and the epilogue's (|rs| <= 24,
    |ob| <= 100) are argument checks: one step beyond returns PQ_EUNSUPPORTED before any launch, on every entry point
    and operand mode, and the outputs stay untouched.  One step inside is accepted."""
    from common.quantity import _native
    lib = _native.lib()
    EUNSUPPORTED = -2
    g = torch.Generator(device="cuda").manual_seed(5)
    x3 = torch.randint(-128, 128, (2, 9, 9, 64), generator=g, device="cuda", dtype=torch.int8)
    w3 = torch.randint(-128, 128, (32, 3, 3, 64), generator=g, device="cuda", dtype=torch.int8)
    w1 = torch.randint(-128, 128, (32, 1, 1, 64), generator=g, device="cuda", dtype=torch.int8)
    bias = torch.zeros(32, dtype=torch.int32, device="cuda")
    xp = torch.randint(-128, 128, (1, 12, 24, 8), generator=g, device="cuda", dtype=torch.int8)
    ws = torch.randint(-128, 128, (32, 3, 64), generator=g, device="cuda", dtype=torch.int8)

    def conv_desc(R, rs, ob):
        return _native.ConvDesc(2, 9, 9, 64, 32, R, R, 1, 1, R // 2, R // 2, 9, 9, rs, ob, 1, 1)

    def add_call(R, ob, sbit, q):
        sc = torch.zeros((2, 9, 9, 32), dtype=torch.int8, device="cuda")
        o16, o8 = Guarded((2 * 81, 32), torch.int16), Guarded((2 * 81, 32), torch.int8)
        add = _native.AddDesc(sc.data_ptr(), 0, sbit, 0, 0, q, o16.ptr(), o8.ptr())
        rc = lib.pq_conv2d_s8_add((x3 if R == 3 else x3).data_ptr(), (w3 if R == 3 else w1).data_ptr(), bias.data_ptr(),
                                  ctypes.byref(conv_desc(R, 7, ob)), ctypes.byref(add), 0, _stream())
        torch.cuda.synchronize()
        return rc, (o16, o8)

    for R in (1, 3):                                   # GEMM form and im2col form of the fused add
        for ob, sbit, q in ((-1, 7, 7), (-1, -1, -1), (8, 8, 8), (4, 4, 20), (4, 4, -12), (7, -1, 7)):
            rc, outs = add_call(R, ob, sbit, q)
            assert rc == EUNSUPPORTED, (R, ob, sbit, q)
            for o in outs:
                assert bool((o.buf == SENTINEL).all())
        for ob, sbit, q in ((0, 7, 7), (0, 0, 0), (7, 7, 7), (4, 4, 19), (4, 4, -11)):
            assert add_call(R, ob, sbit, q)[0] == 0, (R, ob, sbit, q)
    sc = torch.zeros((2, 9, 9, 32), dtype=torch.int8, device="cuda")
    for rs, ob, want in ((25, 0, EUNSUPPORTED), (-25, 0, EUNSUPPORTED), (7, 101, EUNSUPPORTED), (7, -101, EUNSUPPORTED),
                         (24, 0, 0), (-24, 0, 0), (7, 100, 0), (7, -100, 0)):
        outs = []
        out = Guarded((2 * 81, 32), torch.int8)
        outs.append(out)
        assert lib.pq_gemm_s8(x3.data_ptr(), w1.data_ptr(), bias.data_ptr(), 2 * 81, 32, 64, rs, ob, 1, 0, None,
                              out.ptr(), _stream()) == want, (rs, ob)
        for R, w in ((1, w1), (3, w3)):
            out = Guarded((2 * 81, 32), torch.int8)
            outs.append(out)
            assert lib.pq_conv2d_s8(x3.data_ptr(), w.data_ptr(), bias.data_ptr(), ctypes.byref(conv_desc(R, rs, ob)), 0,
                                    None, out.ptr(), _stream()) == want, (R, rs, ob)
            if abs(ob) <= 7:                           # (the add's own limits bound ob more tightly)
                out = Guarded((2 * 81, 32), torch.int8)
                outs.append(out)
                add = _native.AddDesc(sc.data_ptr(), 0, 4, 0, 0, 4, None, out.ptr())
                assert lib.pq_conv2d_s8_add(x3.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                            ctypes.byref(conv_desc(R, rs, ob)), ctypes.byref(add), 0, _stream()) == want
        out = Guarded((10 * 5, 32), torch.int8)
        outs.append(out)
        d = _native.ConvDesc(1, 12, 19, 8, 32, 3, 3, 1, 4, 0, 0, 10, 5, rs, ob, 1, 1)
        assert lib.pq_conv2d_smallc_s8(xp.data_ptr(), ws.data_ptr(), bias.data_ptr(), ctypes.byref(d), 12, 24, 0, None,
                                       out.ptr(), _stream()) == want, (rs, ob)
        torch.cuda.synchronize()
        for o in outs:
            if want == 0:
                o.check("int8")
                assert not bool((o.t.view(torch.uint8) == SENTINEL).all()), "accepted launch wrote nothing"
            else:
                assert bool((o.buf == SENTINEL).all())


# ------------------------------------------------------------------------------------------ pipeline fall-back
@gpu
def test_pipeline_falls_back_outside_the_fused_add_ranges(tmp_path):
    """Bits outside the add kernels' ranges (o_bit 8, o_bit -1, span 8, |q_bit - o_bit| 16) make those Eltwises fall
    back to the fp32-boundary arithmetic: the int8 pipeline still equals the fp32-boundary model, with fewer add
    kernels than Eltwises."""
    import tools
    from bench_sim import build, configs
    from common.quantity import NewAdd, _native, enable_int8_pipeline, merge_bn
    cfg, user = configs(str(tmp_path / "wd"), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build("r18"), "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(2)])
        q.weight_quantize()
        path = cfg["OUTPUT"]["FEAT_BIT_TABLE"]
        lines = [ln.split(" ") for ln in open(path).read().splitlines() if ln.strip()]
        table = {f[0]: f for f in lines}
        rewrite = {"layer1.0.left.3": 8,                                  # o_bit 8 (the shortcut is lower)
                   "layer2.0.left.3": -1, "layer2.0.shortcut.0": -1,      # o_bit -1
                   "layer3.0.left.3": 7, "layer3.0.shortcut.0": -1,       # span 8
                   "layer4.1.Eltwise": int(table["layer4.0.Eltwise"][1]) + 16}   # q_bit - o_bit >= 16
        for name, bit in rewrite.items():
            assert name in table, sorted(table)
            table[name][1] = str(bit)
        open(path, "w").write("\n".join(" ".join(f) for f in lines) + "\n")
        r = tools.Reconstruction(build("r18"), config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), None).cuda().eval()
        x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(7)).cuda()
        ref = model(x)
        enable_int8_pipeline(model)
        model(x)                                                          # first forward: payload census

        def add_kernels():
            return _native.LAUNCHES.get("add_requant", 0) + _native.LAUNCHES.get("conv_add_s8", 0)
        before = add_kernels()
        out = model(x)
        launched = add_kernels() - before
    n_adds = sum(1 for m in model.modules() if isinstance(m, NewAdd))
    assert torch.equal(out, ref)
    assert 0 < launched <= n_adds - 4, (launched, n_adds)


# ------------------------------------------------------------------------------------------ CPU checks
def test_reference_helper_equals_oracle(oracle):
    """The exact evaluation above against the oracle's NewConv2d (int_conv_layer) on integer-valued operands, for
    every rs class and both signs of ob."""
    import numpy as np
    g = torch.Generator().manual_seed(3)
    x = torch.randint(-128, 128, (2, 7, 6, 32), generator=g, dtype=torch.int8)
    w = torch.randint(-128, 128, (24, 3, 3, 32), generator=g, dtype=torch.int8)
    b = torch.randint(-128, 128, (24,), generator=g, dtype=torch.int32)
    b[:4] = torch.tensor([-128, -1, 0, 127], dtype=torch.int32)
    acc = exact_conv(x, w, 1, 1)
    for wb, ib, ob in ((9, 7, -4), (7, 7, 1), (5, 3, 0), (2, 1, 3), (0, 0, 8), (6, 6, -12), (8, 8, -8)):
        info = {"weight_bit": wb, "input_bit": ib, "output_bit": ob, "bias_bit": 2}
        rs = wb + ib - ob
        xf = (x.permute(0, 3, 1, 2).double() * 2.0 ** -ib).float().numpy()
        wf = (w.permute(0, 3, 1, 2).double() * 2.0 ** -wb).float().numpy()
        bf = (b.double() * 2.0 ** -2).float().numpy()
        f32, y = oracle.int_conv_layer(xf, wf, bf, info, stride=1, padding=1)
        want = epilogue_ref(acc, b.long(), rs, False)
        assert np.array_equal(want.view(2, 7, 6, 24).permute(0, 3, 1, 2).numpy(), y), rs
        assert np.array_equal(dequant_ref(want, ob).view(2, 7, 6, 24).permute(0, 3, 1, 2).numpy(), f32), rs


def test_instantiation_table_equals_library_symbols():
    """The gemm_s8_kernel entry symbols of the built library are exactly INSTANTIATIONS, and ROWS reaches each of them
    (plus the row kernel): a new instantiation without an epilogue case fails here."""
    from common.quantity import _native
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    sym = subprocess.run(["cuobjdump", "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run(["cu++filt"], input=sym, check=True, capture_output=True, text=True).stdout
    found = {parse_instantiation(line) for line in names.splitlines() if "STO_ENTRY" in line and "gemm_s8_kernel<" in line}
    assert sorted(found) == INSTANTIATIONS
    assert any(ROWS_KERNEL in line for line in names.splitlines())
    assert {r[2] for r in ROWS} == set(INSTANTIATIONS) | {ROWS_KERNEL}
    pairs = {(r[1], r[2]) for r in ROWS}
    assert len(pairs) == 21 + 22 + 4 + 2 + 1
    assert parse_instantiation("void pq::gemm_s8_kernel<128, 64, 8, true, 8>(CUtensorMap)") == (128, 64, 8, 1, 8)
