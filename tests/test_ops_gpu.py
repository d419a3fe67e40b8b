"""GPU parity of each CUDA operator against the oracle's torch-CPU fp32 arithmetic, called
through the C ABI.  Tolerances are absolute on O(1) data; fp32 accumulation order differs from
MKL-DNN's so bit-exactness is not expected (stated per test)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import svc_oracle as O
from tests.util import max_abs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from whisper_vits_svc_b200 import ops as o
    return o


CONV_CASES = [
    # B, Cin, Cout, T, K, stride, dil, pad
    (2, 192, 192, 300, 1, 1, 1, 0),
    (2, 192, 384, 301, 5, 1, 1, 2),
    (1, 160, 160, 1000, 11, 1, 5, 25),
    (2, 20, 20, 777, 7, 1, 3, 9),
    (2, 10, 10, 1500, 3, 1, 1, 1),
    (1, 10, 1, 640, 7, 1, 1, 3),
    (2, 1, 40, 4096, 8, 4, 1, 2),
    (1, 1, 160, 12800, 128, 64, 1, 32),
    (1, 80, 1280, 200, 3, 1, 1, 1),
    (1, 96, 64, 201, 3, 2, 1, 1),
    (3, 7, 13, 50, 2, 1, 1, 0),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv1d(ops, case):
    B, Cin, Cout, T, K, s, d, p = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, Cin, T, generator=g)
    w = torch.randn(Cout, Cin, K, generator=g) / (Cin * K) ** 0.5
    b = torch.randn(Cout, generator=g)
    ref = F.conv1d(x, w, b, stride=s, padding=p, dilation=d)
    got = ops.conv1d(x.cuda(), w, b.cuda(), stride=s, padding=p, dilation=d)
    assert got.shape == ref.shape
    assert max_abs(got, ref) <= 2e-5  # fp32, different summation order


@pytest.mark.parametrize("act,fn", [(1, torch.relu), (2, lambda v: v * torch.tanh(F.softplus(v))),
                                    (3, F.gelu), (4, torch.tanh)])
def test_conv1d_activations(ops, act, fn):
    g = torch.Generator().manual_seed(act)
    x = torch.randn(2, 24, 100, generator=g) * 3
    w = torch.randn(16, 24, 3, generator=g) / 4
    b = torch.randn(16, generator=g)
    # float64 reference: the host's fp32 conv kernel (and its summation order) differs from box to box,
    # and with pre-activations of magnitude ~25 that alone is ~1e-5
    ref = fn(F.conv1d(x.double(), w.double(), b.double(), padding=1)).float()
    got = ops.conv1d(x.cuda(), w, b.cuda(), padding=1, act=act)
    assert max_abs(got, ref) <= 4e-5   # ~1.5 ulp at |v| = 25 from the 72-term fp32 sum + the activation


@pytest.mark.parametrize("C,L", [(10, 3000), (160, 1024), (3, 1), (5, 7), (20, 2049)])
def test_snake_alias(ops, sd, C, L):
    g = torch.Generator().manual_seed(C + L)
    x = torch.randn(2, C, L, generator=g) * 2
    fake = {"a.act.alpha": torch.randn(C, generator=g) * 0.5, "a.act.beta": torch.randn(C, generator=g) * 0.5,
            "a.upsample.filter": sd["dec.activation_post.upsample.filter"],
            "a.downsample.lowpass.filter": sd["dec.activation_post.downsample.lowpass.filter"]}
    ref = O.snake_alias(fake, "a", x)
    got = ops.snake_alias(x.cuda(), fake["a.act.alpha"], fake["a.act.beta"], fake["a.upsample.filter"],
                          fake["a.downsample.lowpass.filter"])
    assert max_abs(got, ref) <= 1e-5


@pytest.mark.parametrize("C,T,per_batch", [(192, 333, False), (192, 64, True), (80, 31, True)])
def test_layernorm_c(ops, C, T, per_batch):
    g = torch.Generator().manual_seed(C + T)
    x = torch.randn(3, C, T, generator=g) * 2 + 0.5
    r = torch.randn(3, C, T, generator=g)
    if per_batch:
        gamma, beta = torch.randn(3, C, generator=g), torch.randn(3, C, generator=g)
        xt = x.transpose(1, -1)
        mean = xt.mean(-1, keepdim=True)
        var = ((xt - mean) ** 2).mean(-1, keepdim=True)
        ref = (((xt - mean) / (var + 1e-5).sqrt()) * gamma.unsqueeze(1) + beta.unsqueeze(1)).transpose(1, -1)
        got = ops.layernorm_c(x.cuda(), None, gamma.cuda(), beta.cuda())
    else:
        gamma, beta = torch.randn(C, generator=g), torch.randn(C, generator=g)
        ref = O.channel_layer_norm(x + r, gamma, beta)
        got = ops.layernorm_c(x.cuda(), r.cuda(), gamma.cuda(), beta.cuda())
    assert max_abs(got, ref) <= 2e-5


@pytest.mark.parametrize("T,lens,tc", [(150, [150, 97], False), (64, [64, 64], False), (65, [65, 1], False), (300, [300, 201], False),
                                       (150, [150, 97], True), (64, [64, 64], True), (65, [65, 1], True), (300, [300, 201], True),
                                       (5, [5, 3], True), (129, [129, 64], True), (1000, [1000, 777, 1], True), (2520, [2520], True)])
def test_rel_attention(ops, T, lens, tc):
    """fp32 CUDA-core kernel (precision 0) and the tcgen05 kernel (bf16x3 split operands, precision 1 / 3)
    against the oracle's dense pad/reshape formulation in float64, fed the same float32 q, k, v.  Lengths:
    ragged masks, a fully valid item, tiles with a ragged last query / key tile, fewer keys than the relative
    window, the longest chunk (2520).  Worst seen on an NVIDIA B200 (1000 W power limit): 4.3e-6 for the fp32
    kernel, 6.9e-5 for the bf16x3 one (T = 2520, peak 3.7)."""
    g = torch.Generator().manual_seed(T)
    H, heads, w = 192, 2, 4
    B = len(lens)
    x = torch.randn(B, H, T, generator=g)
    fake = {}
    for n in "qkvo":
        fake[f"a.conv_{n}.weight"] = torch.randn(H, H, 1, generator=g) / H ** 0.5 * 1.5
        fake[f"a.conv_{n}.bias"] = torch.randn(H, generator=g) * 0.1
    fake["a.emb_rel_k"] = torch.randn(1, 9, H // heads, generator=g) * (H // heads) ** -0.5
    fake["a.emb_rel_v"] = torch.randn(1, 9, H // heads, generator=g) * (H // heads) ** -0.5
    lengths = torch.tensor(lens)
    mask = O.sequence_mask(lengths, T).unsqueeze(1).double()
    attn_mask = mask.unsqueeze(2) * mask.unsqueeze(-1)
    qkv = torch.cat([F.conv1d(x, fake[f"a.conv_{n}.weight"], fake[f"a.conv_{n}.bias"]) for n in "qkv"], 1)
    # the float64 oracle reads the kernel's own float32 q, k, v: its conv_q/k/v select the rows of qkv
    # (exact in float64) and its conv_o is the identity
    sel = torch.eye(3 * H, dtype=torch.float64).unsqueeze(-1)
    ref64 = {f"a.conv_{n}.weight": sel[j * H:(j + 1) * H] for j, n in enumerate("qkv")}
    ref64.update({f"a.conv_{n}.bias": torch.zeros(H, dtype=torch.float64) for n in "qkvo"})
    ref64["a.conv_o.weight"] = torch.eye(H, dtype=torch.float64).unsqueeze(-1)
    ref64["a.emb_rel_k"], ref64["a.emb_rel_v"] = fake["a.emb_rel_k"].double(), fake["a.emb_rel_v"].double()
    ref = O.rel_attention(ref64, "a", qkv.double(), attn_mask)
    got = ops.rel_attention(qkv.cuda(), fake["a.emb_rel_k"].cuda(), fake["a.emb_rel_v"].cuda(), lengths, tc=tc)
    err = float((got.cpu().double() - ref).abs().max())
    print(f"rel_attention T={T} tc={tc}: max-abs {err:.3e} (peak {float(ref.abs().max()):.2f})")
    assert err <= (1e-4 if tc else 1.5e-5)


@pytest.mark.parametrize("N,K,shift,R", [(160, 160, 0, 128), (160, 160, 7, 178), (80, 80, 25, 160), (48, 48, 3, 140),
                                         (32, 32, 1, 130), (16, 16, 0, 128), (256, 64, 9, 137)])
def test_tcgen05_gemm_selftest(N, K, shift, R):
    """tcgen05.mma + TMEM + row-shifted K-major SWIZZLE_NONE descriptors (the conv-tap trick):
    bf16 inputs, fp32 accumulate -> exact up to fp32 summation order."""
    import ctypes
    from whisper_vits_svc_b200 import _lib
    g = torch.Generator().manual_seed(N + K + shift)
    A = torch.randn(R, K, generator=g).bfloat16()
    Bm = torch.randn(N, K, generator=g).bfloat16()
    ref = A[shift:shift + 128].float() @ Bm.float().t()
    Ad, Bd = A.cuda(), Bm.cuda()
    D = torch.zeros(128, N, device="cuda")
    st = _lib.load().svcb_op_tc_gemm_selftest(Ad.data_ptr(), Bd.data_ptr(), D.data_ptr(), R, N, K, shift,
                                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(st, "svcb_op_tc_gemm_selftest")
    torch.cuda.synchronize()
    assert max_abs(D, ref) <= 1e-3 * K ** 0.5


@pytest.mark.parametrize("C,L,K,dil,nsplit,tol", [
    (160, 700, 11, 5, 3, 2e-4), (160, 300, 3, 1, 3, 2e-4), (80, 1000, 7, 3, 3, 2e-4), (40, 513, 11, 1, 3, 2e-4),
    (20, 1024, 7, 5, 3, 2e-4), (10, 2000, 3, 3, 3, 2e-4), (80, 640, 7, 1, 1, 5e-2), (10, 127, 11, 5, 3, 2e-4)])
def test_amp_conv_tc(ops, sd, C, L, K, dil, nsplit, tol):
    """Fused SnakeAlias -> Conv1d (+bias +residual) on tcgen05 vs the oracle's two torch ops.
    bf16x3 split operands: expected error ~1e-5 on O(1) data; plain bf16 ~1e-2 (reported, loose)."""
    g = torch.Generator().manual_seed(C * 7 + L + K + dil)
    B = 2
    x = torch.randn(B, C, L, generator=g) * 1.5
    w = torch.randn(C, C, K, generator=g) / (C * K) ** 0.5
    b = torch.randn(C, generator=g) * 0.1
    res = torch.randn(B, C, L, generator=g)
    fake = {"a.act.alpha": torch.randn(C, generator=g) * 0.4, "a.act.beta": torch.randn(C, generator=g) * 0.4,
            "a.upsample.filter": sd["dec.activation_post.upsample.filter"],
            "a.downsample.lowpass.filter": sd["dec.activation_post.downsample.lowpass.filter"]}
    ref = F.conv1d(O.snake_alias(fake, "a", x), w, b, dilation=dil, padding=dil * (K - 1) // 2) + res
    got = ops.amp_conv_tc(x.cuda(), fake["a.act.alpha"], fake["a.act.beta"], fake["a.upsample.filter"],
                          fake["a.downsample.lowpass.filter"], w, b.cuda(), dilation=dil, res=res.cuda(), nsplit=nsplit)
    err = max_abs(got, ref)
    print(f"amp_conv_tc C={C} L={L} K={K} d={dil} nsplit={nsplit}: max-abs {err:.3e}")
    assert err <= tol


@pytest.mark.parametrize("Cin,Cout,T,K,dil,nsplit,tol", [
    (192, 384, 1000, 5, 1, 3, 2e-4), (192, 576, 300, 1, 1, 3, 2e-4), (640, 192, 257, 3, 1, 3, 2e-4),
    (96, 192, 130, 1, 1, 3, 2e-4), (192, 640, 500, 3, 1, 3, 2e-4), (192, 320, 64, 7, 1, 3, 2e-4),
    (1280, 192, 200, 5, 1, 3, 3e-4), (192, 96, 77, 1, 1, 1, 5e-2)])
def test_conv_tc(ops, Cin, Cout, T, K, dil, nsplit, tol):
    """General implicit-GEMM Conv1d on tcgen05 vs F.conv1d (fp32 CPU)."""
    g = torch.Generator().manual_seed(Cin + Cout + T + K)
    x = torch.randn(2, Cin, T, generator=g)
    w = torch.randn(Cout, Cin, K, generator=g) / (Cin * K) ** 0.5
    b = torch.randn(Cout, generator=g) * 0.1
    ref = F.conv1d(x, w, b, dilation=dil, padding=dil * (K - 1) // 2)
    got = ops.conv_tc(x.cuda(), w, b.cuda(), dilation=dil, nsplit=nsplit)
    err = max_abs(got, ref)
    print(f"conv_tc {Cin}->{Cout} T={T} K={K} nsplit={nsplit}: max-abs {err:.3e}")
    assert err <= tol


def test_conv_tc_epilogues(ops):
    """masks, gate on interleaved pairs, residual, ReLU — the flags the prior/flow pipelines use."""
    g = torch.Generator().manual_seed(99)
    B, C, T = 2, 192, 150
    x = torch.randn(B, C, T, generator=g)
    lengths = torch.tensor([150, 101])
    mask = O.sequence_mask(lengths, T).unsqueeze(1).float()
    w = torch.randn(2 * C, C, 5, generator=g) / (C * 5) ** 0.5
    b = torch.randn(2 * C, generator=g) * 0.1
    a = F.conv1d(x, w, b, padding=2)
    ref = torch.tanh(a[:, :C]) * torch.sigmoid(a[:, C:])
    idx = torch.stack([torch.arange(C), torch.arange(C) + C], 1).reshape(-1)
    got = ops.conv_tc(x.cuda(), w[idx], b[idx].cuda(), flags=4)
    assert max_abs(got, ref) <= 2e-4
    w2 = torch.randn(C, C, 3, generator=g) / (C * 3) ** 0.5
    b2 = torch.randn(C, generator=g) * 0.1
    res = torch.randn(B, C, T, generator=g)
    ref2 = torch.relu(F.conv1d(x * mask, w2, b2, padding=1)) * mask + res
    got2 = ops.conv_tc(x.cuda(), w2, b2.cuda(), res=res.cuda(), lengths=lengths, flags=1 | 2, act=1)
    assert max_abs(got2, ref2) <= 2e-4


@pytest.mark.parametrize("C,L,K,dil", [(20, 8 * 126 * 2, 3, 1), (20, 8 * 300, 11, 5), (20, 8 * 126, 7, 3), (20, 8 * 5, 11, 3),
                                       (20, 8, 3, 1), (20, 8 * 1000, 11, 1), (10, 16 * 126, 3, 1), (10, 16 * 200, 11, 5),
                                       (10, 16 * 3, 7, 5), (10, 16 * 257, 7, 1), (40, 4 * 124 * 2, 3, 1), (40, 4 * 500, 11, 5),
                                       (40, 8, 7, 3), (40, 4 * 126, 11, 1), (40, 4 * 1002, 7, 5)])
def test_amp_s2d_link(ops, sd, C, L, K, dil):
    """One AMP-block link of the narrow stages in space-to-depth form (csrc/amp_s2d.cu): block-Toeplitz
    tcgen05 conv (bf16x3) with bias + residual, and the NEXT SnakeAlias computed in the epilogue — both
    against the oracle's torch ops.  Lengths cover: whole tiles (126 useful rows), ragged last tiles, a
    single row, items shorter than the Snake / conv reach (sequence-end clamps on both sides at once)."""
    g = torch.Generator().manual_seed(C * 11 + L + K + dil)
    B = 2
    x = torch.randn(B, C, L, generator=g) * 1.5
    w = torch.randn(C, C, K, generator=g) / (C * K) ** 0.5
    b = torch.randn(C, generator=g) * 0.1
    res = torch.randn(B, C, L, generator=g)
    filt = {"upsample.filter": sd["dec.activation_post.upsample.filter"],
            "downsample.lowpass.filter": sd["dec.activation_post.downsample.lowpass.filter"]}
    fa = {"a.act.alpha": torch.randn(C, generator=g) * 0.4, "a.act.beta": torch.randn(C, generator=g) * 0.4,
          **{"a." + k: v for k, v in filt.items()}}
    fb = {"b.act.alpha": torch.randn(C, generator=g) * 0.4, "b.act.beta": torch.randn(C, generator=g) * 0.4,
          **{"b." + k: v for k, v in filt.items()}}
    ref = F.conv1d(O.snake_alias(fa, "a", x), w, b, dilation=dil, padding=dil * (K - 1) // 2) + res
    ref_act = O.snake_alias(fb, "b", ref)
    got, got_act = ops.amp_s2d_link(x.cuda(), fa["a.act.alpha"], fa["a.act.beta"], filt["upsample.filter"],
                                    filt["downsample.lowpass.filter"], w, b.cuda(), dilation=dil, res=res.cuda(),
                                    alpha_out=fb["b.act.alpha"], beta_out=fb["b.act.beta"])
    e1, e2 = max_abs(got, ref), max_abs(got_act, ref_act)
    print(f"amp_s2d_link C={C} L={L} K={K} d={dil}: conv max-abs {e1:.3e}, next-snake image max-abs {e2:.3e}")
    assert e1 <= 2e-4 and e2 <= 3e-4
