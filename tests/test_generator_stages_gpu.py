"""Every generator stage of every precision mode on its own, against the float64 oracle.

`SynthesizerInfer.generator(..., taps=...)` returns all generator taps.  Each tap is compared with the float64
oracle stage (oracle/svc_oracle.py: gen_pre, gen_up, gen_amp_stage, gen_post) fed with the DEVICE's own previous
tap, so each comparison sees only the error of the kernels that compute that stage, not the error carried in
from upstream.  The waveform hides a stage error (a stage change reaches the wave 7-20x smaller), so a bound on
the wave alone lets a stage be wrong by ~1e-3 unnoticed.

Which kernels compute each tap (csrc/api.cu: run_generator / run_amp_stage) for the default generator
(channels 320 -> 160/80/40/20/10, rates 5,4,4,2,2); `test_dispatch_kernel_sets` holds the runs to it:

  tap          precision 0                      precision 1 (bf16) / 3 (bf16x3)
  gen_pre      layernorm_c + conv1d              layernorm_c + conv_tc
  gen_up0      conv1d phases + ups_finalize      conv_tc phases + ups_finalize + noise conv as conv_tc (noise_tc)
               + conv1d noise conv
  gen_up1, 2   (same as gen_up0; ups_finalize    comb_up: one conv_tc with the interleaved store (ilv) and the
               adds the short noise conv at 2)   source gather (x2)
  gen_up3, 4   conv1d phases + ups_finalize      ups_fused (fp32)
  gen_stage0,1 snake_alias + conv1d              snake_pack + amp_conv_tc
  gen_stage2   snake_alias + conv1d              p3: amp_s2d_link chain;  p1: snake_pack + amp_conv_tc
  gen_stage3,4 snake_alias + conv1d              p3: amp_s2d_link chain (accum / out_div fold the stage mean);
                                                 p1: amp_block_fused (fp32)
  wave         post_fused (fp32)                 post_fused (fp32)

The 80-input geometry (`gen80`) runs the same kernels.  The 256-wide generator (`w256`, channels 128/64/32/16/8)
misses every specialised kernel: precision 1 and 3 run snake_pack + amp_conv_tc in all five stages, and conv_tc
polyphase phases + ups_finalize (with the short noise conv fused) at the rate-2 stages 3 and 4.

Bounds (max|got - ref| <= bound * max|ref|), one per kernel family and precision, set at >= 3x the worst error
observed over the whole sweep below (3 configurations x 16 (B, T) x 3 precisions; NVIDIA B200, 1000 W power
limit).  Worst observed, relative to the stage peak (peaks are 2.5-7):

  family              precision  observed  bound
  conv1d              0          1.6e-6    5e-6
  conv1d_ups          0          1.4e-6    5e-6
  snake_alias_conv1d  0          4.3e-7    2e-6
  post_fused          0 / 1 / 3  6.0e-7    2e-6
  ups_fused           1 / 3      4.4e-7    2e-6
  amp_block_fused     1          2.3e-7    1e-6
  conv_tc             3          8.2e-6    3e-5
  conv_tc_ups         3          8.1e-6    3e-5
  comb_up             3          6.2e-6    2e-5
  amp_conv_tc         3          5.4e-6    2e-5
  amp_s2d             3          5.1e-6    2e-5
  conv_tc             1          3.4e-3    1.2e-2
  conv_tc_ups         1          3.3e-3    1e-2
  comb_up             1          2.9e-3    1e-2
  amp_conv_tc         1          2.0e-3    6e-3

Plain bf16 (precision 1) rounds both operands to 8 significant bits (unit roundoff 2^-8 = 3.9e-3), so an error
near one rounding unit of the peak is its nature, not a defect; the conv_tc bound is 3.6x its worst case.
"""
import os

import numpy as np
import pytest
import torch

from oracle import svc_oracle as O
from tests.util import GOLDEN, launched_kernels, make_inputs, max_abs
from whisper_vits_svc_b200 import hparams, synth

pytestmark = pytest.mark.gpu

N_UPS = 5
TAPS = ["gen_pre"] + [f"gen_{s}{i}" for i in range(N_UPS) for s in ("up", "stage")]
CONFIGS = {
    "base": {},
    "gen80": dict(gen__upsample_input=80, data__sampling_rate=24000),
    "w256": dict(gen__upsample_initial_channel=256),
}


def stage_families(cfg: str, precision: int) -> dict:
    """tap -> kernel family (the module docstring's table)."""
    if precision == 0:
        fam = {"gen_pre": "conv1d", "wave": "post_fused"}
        for i in range(N_UPS):
            fam[f"gen_up{i}"] = "conv1d_ups"
            fam[f"gen_stage{i}"] = "snake_alias_conv1d"
        return fam
    fam = {"gen_pre": "conv_tc", "gen_up0": "conv_tc_ups", "gen_up1": "comb_up", "gen_up2": "comb_up",
           "wave": "post_fused"}
    for i in range(N_UPS):
        fam[f"gen_stage{i}"] = "amp_conv_tc"
    if cfg == "w256":
        fam["gen_up3"] = fam["gen_up4"] = "conv_tc_ups"
        return fam
    fam["gen_up3"] = fam["gen_up4"] = "ups_fused"
    if precision == 3:
        fam["gen_stage2"] = fam["gen_stage3"] = fam["gen_stage4"] = "amp_s2d"
    else:
        fam["gen_stage3"] = fam["gen_stage4"] = "amp_block_fused"
    return fam


# (family, precision) -> bound relative to the stage peak
BOUNDS = {
    ("conv1d", 0): 5e-6, ("conv1d_ups", 0): 5e-6, ("snake_alias_conv1d", 0): 2e-6,
    **{("post_fused", p): 2e-6 for p in (0, 1, 3)}, **{("ups_fused", p): 2e-6 for p in (1, 3)},
    ("amp_block_fused", 1): 1e-6,
    ("conv_tc", 3): 3e-5, ("conv_tc_ups", 3): 3e-5, ("comb_up", 3): 2e-5, ("amp_conv_tc", 3): 2e-5, ("amp_s2d", 3): 2e-5,
    ("conv_tc", 1): 1.2e-2, ("conv_tc_ups", 1): 1e-2, ("comb_up", 1): 1e-2, ("amp_conv_tc", 1): 6e-3,
}


def bound(cfg, precision, tap):
    return BOUNDS[(stage_families(cfg, precision)[tap], precision)]


# ------------------------------------------------------------------------------------------------ fixtures
_HP, _SD, _MODELS, _CASES = {}, {}, {}, {}
_WORST = {}   # (family, precision) -> (worst relative error, where)


def _hp(cfg):
    if cfg not in _HP:
        base = hparams.load_hparams(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                 "configs", "base.yaml"))
        _HP[cfg] = hparams.override(base, **CONFIGS[cfg])
    return _HP[cfg]


def _sd(cfg):
    if cfg not in _SD:
        sd = synth.svc_state_dict(_hp(cfg), 1234)
        _SD[cfg] = (sd, {k: v.double() for k, v in sd.items()})
    return _SD[cfg]


def _new_model(hpx, sd, precision):
    from whisper_vits_svc_b200 import models
    m = models.SynthesizerInfer(hpx.data.filter_length // 2 + 1, hpx.data.segment_size // hpx.data.hop_length, hpx,
                                precision=precision)
    m.load_state_dict(sd)
    m.eval()
    return m.to("cuda")


def _model(cfg, precision):
    if (cfg, precision) not in _MODELS:
        _MODELS[(cfg, precision)] = _new_model(_hp(cfg), _sd(cfg)[0], precision)
    return _MODELS[(cfg, precision)]


def _case(cfg, B, T):
    """Seeded generator inputs (float32 and float64) and the oracle's float64 gen_pre, cached per (cfg, B, T)."""
    key = (cfg, B, T)
    if key not in _CASES:
        hpx = _hp(cfg)
        sd, sd64 = _sd(cfg)
        d = make_inputs(100 + 7 * T + B, B, T, hpx, gen_only=True)
        src = O.pitch2source(sd, hpx, d["pit"], d["rand_ini"], d["noise"])
        c = dict(spk=d["spk"], z=d["z"], src=src, spk64=d["spk"].double(), z64=d["z"].double(), src64=src.double())
        with torch.no_grad():
            c["pre64"] = O.gen_pre(sd64, c["spk64"], c["z64"])
        _CASES[key] = c
    return _CASES[key]


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if _WORST:
        print("\nworst stage error per kernel family (relative to the stage peak):")
        for (fam, p), (e, where) in sorted(_WORST.items(), key=lambda kv: (kv[0][1], kv[0][0])):
            print(f"  {fam:20s} precision {p}  {e:.2e}  ({where})  bound {BOUNDS[(fam, p)]:.0e}")
    _MODELS.clear()


def run_device(m, c, B, T, hpx):
    """All generator taps + the wave from one svcb_generator call."""
    ch0 = int(hpx.gen.upsample_initial_channel)
    rates = [int(r) for r in hpx.gen.upsample_rates]
    taps = {"gen_pre": torch.zeros(B, ch0, T, device="cuda")}
    L = T
    for i in range(N_UPS):
        L *= rates[i]
        for s in ("up", "stage"):
            taps[f"gen_{s}{i}"] = torch.zeros(B, ch0 >> (i + 1), L, device="cuda")
    wave = m.generator(c["spk"], c["z"], c["src"], taps=taps)
    torch.cuda.synchronize()
    out = {k: v.cpu().double() for k, v in taps.items()}
    out["wave"] = wave.cpu().double()
    return out


def stage_errors(hpx, sd64, c, got, upto=None):
    """[(tap, max-abs error, peak)] of each device tap against the float64 oracle stage fed with the device's
    previous tap, in pipeline order, stopping after `upto`."""
    rows = []

    def add(name, ref):
        rows.append((name, float((got[name] - ref).abs().max()), float(ref.abs().max())))
        return name == upto

    with torch.no_grad():
        if add("gen_pre", c["pre64"]):
            return rows
        prev = got["gen_pre"]
        for i in range(N_UPS):
            if add(f"gen_up{i}", O.gen_up(sd64, hpx, i, prev, c["src64"])):
                return rows
            if add(f"gen_stage{i}", O.gen_amp_stage(sd64, hpx, i, got[f"gen_up{i}"])):
                return rows
            prev = got[f"gen_stage{i}"]
        add("wave", O.gen_post(sd64, prev))
    return rows


# ------------------------------------------------------------------------------------------------ the sweep
# T around the tile edges of each kernel (rows of one tile; the stage lengths are L = T * 5, 20, 80, 160, 320):
#   amp_conv_tc: 128 rows -> stage 0 (L = 5T) full at T = 25.6 (T = 26); stage 1 (L = 20T) at T = 6.4 (6 / 7, 13)
#   amp_s2d_link: 20T rows of r samples against 126 useful rows per tile -> T = 6 / 7, 13
#   ups_fused: 80T output pairs at stage 3 against 256 per block -> T = 3 / 4
#   post_fused: 254 x 8 = 2032 samples per block, L = 320T -> T = 6 / 7, 13
#   conv_tc: 128 output rows per tile -> conv_pre / stage-0 phases at T = 64 / 129
SWEEP = ([("base", 2, T) for T in (1, 3, 4, 6, 7, 13, 26, 64, 129)] + [("base", 3, 13)] +
         [("gen80", 2, 7), ("gen80", 2, 36)] +
         [("w256", 2, T) for T in (1, 4, 7, 13, 64)])


@pytest.mark.parametrize("precision", [0, 1, 3])
@pytest.mark.parametrize("cfg,B,T", SWEEP)
def test_generator_stage_vs_float64(cfg, B, T, precision):
    hpx = _hp(cfg)
    c = _case(cfg, B, T)
    got = run_device(_model(cfg, precision), c, B, T, hpx)
    fam = stage_families(cfg, precision)
    report, bad = [], []
    for tap, e, peak in stage_errors(hpx, _sd(cfg)[1], c, got):
        rel = e / peak
        b = BOUNDS[(fam[tap], precision)]
        key = (fam[tap], precision)
        if rel > _WORST.get(key, (-1.0, ""))[0]:
            _WORST[key] = (rel, f"{cfg} B={B} T={T} {tap}")
        report.append(f"  {tap:11s} {fam[tap]:20s} max-abs {e:.2e}  peak {peak:5.2f}  rel {rel:.2e}  bound {b:.0e}")
        if not e <= b * peak:
            bad.append(tap)
    print(f"\n{cfg} B={B} T={T} precision {precision}\n" + "\n".join(report))
    assert not bad, f"stages out of bound: {bad}\n" + "\n".join(report)


# ------------------------------------------------------------------------------------------------ dispatch
def _amp(prefix, ch, ks=(3, 7, 11), suffix=""):
    return {f"{prefix}_c{ch}k{k}{suffix}" for k in ks}


COMMON = {"linear_small", "layernorm_c"}


def _base_tc(mode, cin):
    """Default widths, either tensor-core mode: stage 0 = conv_tc phases (320 -> 160, 3 taps) + ups_finalize +
    noise_tc (64 source channels, 2 taps); stages 1-2 = comb_up (rate * Cout outputs, 3 taps); 3-4 = ups_fused."""
    return (COMMON | {
        "pad_source", f"conv_tc_{mode}_{cin}to320_k7_o1", f"conv_tc_{mode}_320to160_k3_o1", "ups_finalize",
        f"conv_tc_{mode}_64to160_k2_o1", "snake_pack_c160", "snake_pack_c80", f"conv_tc_{mode}_160to320_k3_o1",
        f"conv_tc_{mode}_80to160_k3_o1", "ups_fused_40to20", "ups_fused_20to10", "post_fused"}
        | _amp(f"amp_conv_tc_{mode}", 160) | _amp(f"amp_conv_tc_{mode}", 80))


def _base_p3(cin):
    return (_base_tc("bf16x3", cin)
            | {"s2d_image_clear", "snake_pack_s2d_c40", "snake_pack_s2d_c20", "snake_pack_s2d_c10"}
            | _amp("amp_s2d_link", 40, suffix="r4") | _amp("amp_s2d_link", 20, suffix="r8")
            | _amp("amp_s2d_link", 10, suffix="r16"))


def _base_p1(cin):
    return (_base_tc("bf16", cin) | {"snake_pack_c40"} | _amp("amp_conv_tc_bf16", 40)
            | _amp("amp_block_fused", 20) | _amp("amp_block_fused", 10))


def _w256(mode):
    """256 wide: amp_conv_tc in every stage; stages 3-4 as conv_tc phases (rate 2, 2 taps) + ups_finalize."""
    return (COMMON | {
        "pad_source", f"conv_tc_{mode}_192to256_k7_o1", f"conv_tc_{mode}_256to128_k3_o1", "ups_finalize",
        f"conv_tc_{mode}_64to128_k2_o1", f"conv_tc_{mode}_128to256_k3_o1", f"conv_tc_{mode}_64to128_k3_o1",
        f"conv_tc_{mode}_32to16_k2_o1", f"conv_tc_{mode}_16to8_k2_o1", "post_fused"}
        | {f"snake_pack_c{ch}" for ch in (128, 64, 32, 16, 8)}
        | set().union(*(_amp(f"amp_conv_tc_{mode}", ch) for ch in (128, 64, 32, 16, 8))))


def _p0(cin, ch0):
    """precision 0: every conv on conv1d_fp32 (phases with out_mul 1, the long noise convs as accumulate passes)."""
    s = COMMON | {f"conv1d_fp32_{cin}to{ch0}_k7_o1", "ups_finalize", "snake_alias", "post_fused"}
    taps = [3, 2, 2, 2, 2]
    noise_k = [128, 32]
    ch = ch0
    for i in range(N_UPS):
        s.add(f"conv1d_fp32_{ch}to{ch // 2}_k{taps[i]}_o1")
        ch //= 2
        if i < 2:
            s.add(f"conv1d_fp32_1to{ch}_k{noise_k[i]}_o1")
        s |= {f"conv1d_fp32_{ch}to{ch}_k{k}_o1" for k in (3, 7, 11)}
    return s


KERNELS = {
    ("base", 3): _base_p3(192), ("gen80", 3): _base_p3(80), ("w256", 3): _w256("bf16x3"),
    ("base", 1): _base_p1(192), ("gen80", 1): _base_p1(80), ("w256", 1): _w256("bf16"),
    ("base", 0): _p0(192, 320), ("gen80", 0): _p0(80, 320), ("w256", 0): _p0(192, 256),
}


@pytest.mark.parametrize("precision", [0, 1, 3])
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_dispatch_kernel_sets(cfg, precision):
    """The exact set of kernels one generator call launches, so that a changed dispatch predicate
    (ups_fused_supported, amp_block_fused_supported, post_fused_supported, the comb_up / noise_tc conditions,
    s2d_link_factor) cannot move a stage to another kernel without the stage table above changing with it."""
    hpx = _hp(cfg)
    B, T = 2, 13
    got = launched_kernels(lambda: run_device(_model(cfg, precision), _case(cfg, B, T), B, T, hpx))
    print(f"\n{cfg} precision {precision}: {sorted(got)}")
    assert got == KERNELS[(cfg, precision)], (f"missing {sorted(KERNELS[(cfg, precision)] - got)}, "
                                              f"unexpected {sorted(got - KERNELS[(cfg, precision)])}")
    if precision != 0:
        assert not any(k.startswith("conv1d_fp32_") or k == "snake_alias" for k in got)
    if cfg == "base" and precision == 3:
        assert not any(k.startswith("amp_block_fused_") for k in got)
        assert sum(k == "ups_finalize" for k in got) == 1
    if cfg == "w256":
        assert not any(k.startswith(("amp_s2d_link", "snake_pack_s2d", "ups_fused", "amp_block_fused")) for k in got)


# ------------------------------------------------------------------------------------------------ the bounds see a bug
def _shift_noise(sd, stage):
    """noise_convs[stage] filter moved by one source sample (an off-by-one in the kernel's source index)."""
    k = f"dec.noise_convs.{stage}.weight"
    w = torch.zeros_like(sd[k])
    w[..., 1:] = sd[k][..., :-1]
    return {k: w}


PERTURBATIONS = [
    # (name, precision, stage tap it must show in)
    ("noise_shift0", 3, "gen_up0"), ("noise_shift1", 3, "gen_up1"), ("noise_shift3", 3, "gen_up3"),
    ("noise_shift3", 1, "gen_up3"),
    ("bias2", 3, "gen_stage2"), ("bias3", 3, "gen_stage3"), ("bias4", 3, "gen_stage4"),
    ("bias3", 1, "gen_stage3"), ("bias4", 1, "gen_stage4"),
    ("post_alpha", 3, "wave"), ("post_alpha", 1, "wave"),
]


def _oracle_chain(cfg, B, T):
    """The float64 oracle's own stages (cached): the inputs on which a perturbation's size is computed."""
    c = _case(cfg, B, T)
    if "chain64" not in c:
        st = {}
        with torch.no_grad():
            c["wave64"] = O.generator(_sd(cfg)[1], _hp(cfg), c["spk64"], c["z64"], c["src64"], stages=st)
        c["chain64"] = st
    return c


def _perturb(name, cfg, precision, B, T):
    """State-dict entries to replace.  Bias and alpha shifts are sized so that the float64 oracle's stage moves
    by 3x that stage's bound (computed here, not by hand)."""
    hpx, (sd, sd64) = _hp(cfg), _sd(cfg)
    if name.startswith("noise_shift"):
        return _shift_noise(sd, int(name[-1]))
    c = _oracle_chain(cfg, B, T)
    if name.startswith("bias"):
        i = int(name[-1])
        tap = f"gen_stage{i}"
        key = f"dec.resblocks.{i * len(hpx.gen.resblock_kernel_sizes) + 1}.convs2.2.bias"
        x, ref = c["chain64"][f"gen_up{i}"], c["chain64"][tap]

        def change(delta):
            b = sd64[key].clone()
            b[0] += delta
            with torch.no_grad():
                return float((O.gen_amp_stage({**sd64, key: b}, hpx, i, x) - ref).abs().max())
    else:
        tap, key = "wave", "dec.activation_post.act.alpha"
        x, ref = c["chain64"]["gen_stage4"], c["wave64"]

        def change(delta):
            a = sd64[key].clone()
            a[0] += delta
            with torch.no_grad():
                return float((O.gen_post({**sd64, key: a}, x) - ref).abs().max())
    target = 3 * bound(cfg, precision, tap) * float(ref.abs().max())
    delta = 1e-3
    for _ in range(3):   # secant steps on a (near-)linear response
        delta *= target / change(delta)
    assert 2.5 * target / 3 <= change(delta) <= 3.5 * target / 3
    v = sd[key].clone()
    v[0] += delta
    return {key: v}


@pytest.mark.parametrize("name,precision,tap", PERTURBATIONS)
def test_stage_bounds_flag_perturbed_weights(name, precision, tap):
    """A plausible kernel bug emulated in the weights (device model only; the oracle keeps the original state
    dict): the stage comparator must flag the stage it lands in and no stage before it.  Changes weights, not
    kernels: nothing unusual runs on the device."""
    cfg, B, T = "base", 2, 7
    hpx, (sd, sd64) = _hp(cfg), _sd(cfg)
    m = _new_model(hpx, {**sd, **_perturb(name, cfg, precision, B, T)}, precision)
    c = _case(cfg, B, T)
    rows = stage_errors(hpx, sd64, c, run_device(m, c, B, T, hpx), upto=tap)
    flagged = [t for t, e, peak in rows if e > bound(cfg, precision, t) * peak]
    report = "\n".join(f"  {t:11s} max-abs {e:.2e} peak {p:5.2f} bound {bound(cfg, precision, t) * p:.2e}"
                       for t, e, p in rows)
    print(f"\n{name} precision {precision}\n{report}")
    assert flagged == [tap], report


# ------------------------------------------------------------------------------------------------ golden, tensor cores
@pytest.mark.parametrize("name,cfg", [("gen80_b2_t36", "gen80"), ("gen192_b1_t64", "base")])
def test_golden_generator_tensor_core_mode(name, cfg):
    """The two golden generator geometries (waves of the unmodified reference) in the default precision 3."""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    hpx = _hp(cfg)
    m = _model(cfg, 3)
    d = make_inputs(int(g["seed"]), int(g["B"]), int(g["T"]), hpx, gen_only=True)
    wave = m.generator(d["spk"], d["z"], torch.from_numpy(g["source"]))
    err = max_abs(wave, g["wave"])
    print(f"{name} (precision 3): wave max-abs err {err:.3e}")
    assert err <= 2e-4
