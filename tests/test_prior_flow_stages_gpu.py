"""Every prior-encoder layer and flow step of every precision mode on its own, against the float64 oracle.

`SynthesizerInfer.prior(..., taps=...)` returns z_p and fills the encoder taps; `flow_reverse(z_p, ..., taps=...)`
fills the flow taps (pipeline order z_p -> flow3 -> flow2 -> flow1 -> flow0 = z).  Each tap is compared with the
float64 oracle stage (oracle/svc_oracle.py: enc_front, enc_layer, enc_proj, flow_step) fed with the DEVICE's own
previous tap, so each comparison sees only the error of the kernels that compute that stage.  The waveform hides a
stage error several times over, so a bound on the wave alone lets one encoder layer or flow step be off unnoticed.

Which kernels compute each tap (csrc/api.cu: run_prior / run_flow); `test_dispatch_kernel_sets` holds the runs to it:

  tap          precision 0                           precision 1 (bf16) / 3 (bf16x3)
  enc_front    conv1d (pre, hub on time-major input)  conv_tc (the same, float4 loads of time-major input)
               + pitch_embed_add                      + pitch_embed_add
  enc_layer*   conv1d (qkv, o, ffn1, ffn2)            conv_tc (qkv, o, ffn1, ffn2) + rel_attn_pack + rel_attn_tc
               + rel_attention + layernorm_c           + layernorm_c
  z_p          conv1d (proj) + reparam                conv_tc (proj) + reparam
  flow*        conv1d (pre, gated WN in, res/skip,    conv_tc (the same) + linear_small + coupling_pre/post
               post) + linear_small + coupling_pre/    + wn_update
               post + wn_update

enc_front, z_p and the flows are compared on all frames (the device's z_p and flow outputs must be exactly 0 on
padded frames); the encoder layers on valid frames only: their padded frames are don't-care, and the float64
oracle's valid frames do not depend on them (tests/test_oracle_stages_cpu.py::test_padded_frames_do_not_matter).

Bounds (max|got - ref| <= bound * max|ref|), one per (tap kind, precision), set at >= 3x the worst error observed
over the whole sweep below (10 (B, T, lengths) x 3 precisions; NVIDIA B200, 1000 W power limit).  Worst observed,
relative to the stage peak (peaks are 3-15):

  tap kind    precision  observed  bound
  enc_front   0          2.5e-6    8e-6
  enc_layer   0          1.4e-6    5e-6
  z_p         0          7.5e-7    3e-6
  flow        0          1.6e-7    6e-7
  enc_front   3          1.7e-5    6e-5
  enc_layer   3          2.0e-5    7e-5
  z_p         3          6.1e-6    2e-5
  flow        3          1.7e-6    6e-6
  enc_front   1          2.5e-3    8e-3
  enc_layer   1          7.2e-3    2.5e-2
  z_p         1          2.7e-3    1e-2
  flow        1          8.6e-4    3e-3

The errors do not grow at the tile edges: at precision 3 enc_front is 1.2e-5 to 1.7e-5 and the encoder layers
1.0e-5 to 2.0e-5 for every T from 4 to 2520.  bf16x3 keeps about 16 significant bits of each operand, and enc_front
sums 6400 products per output (pre: 1280 channels x 5 taps), hence its ~2e-5.  Plain bf16 (precision 1) keeps 8
(unit roundoff 2^-8 = 3.9e-3), so its errors sit near one or two rounding units of the peak.
"""
import numpy as np
import pytest
import torch

from oracle import svc_oracle as O
from tests.util import launched_kernels, make_inputs

pytestmark = pytest.mark.gpu

N_LAYERS, N_FLOWS = 6, 4
ENC_TAPS = ["enc_front"] + [f"enc_layer{i}" for i in range(N_LAYERS)]
FLOW_TAPS = [f"flow{i}" for i in reversed(range(N_FLOWS))]   # pipeline order: flow3 runs first
TAPS = ENC_TAPS + ["z_p"] + FLOW_TAPS


def kind(tap):
    return "enc_layer" if tap.startswith("enc_layer") else "flow" if tap.startswith("flow") else tap


# (tap kind, precision) -> bound relative to the stage peak
BOUNDS = {
    ("enc_front", 0): 8e-6, ("enc_layer", 0): 5e-6, ("z_p", 0): 3e-6, ("flow", 0): 6e-7,
    ("enc_front", 3): 6e-5, ("enc_layer", 3): 7e-5, ("z_p", 3): 2e-5, ("flow", 3): 6e-6,
    ("enc_front", 1): 8e-3, ("enc_layer", 1): 2.5e-2, ("z_p", 1): 1e-2, ("flow", 1): 3e-3,
}


def bound(precision, tap):
    return BOUNDS[(kind(tap), precision)]


# ------------------------------------------------------------------------------------------------ fixtures
_MODELS, _CASES = {}, {}
_WORST = {}   # (tap kind, precision) -> (worst relative error, where)


@pytest.fixture(scope="module")
def sd64(sd):
    return {k: v.double() for k, v in sd.items()}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if _WORST:
        print("\nworst stage error per tap kind (relative to the stage peak):")
        for (k, p), (e, where) in sorted(_WORST.items(), key=lambda kv: (kv[0][1], kv[0][0])):
            print(f"  {k:10s} precision {p}  {e:.2e}  ({where})  bound {BOUNDS[(k, p)]:.0e}")
    _MODELS.clear()


def _new_model(hp, sd, precision):
    from whisper_vits_svc_b200 import models
    m = models.SynthesizerInfer(hp.data.filter_length // 2 + 1, hp.data.segment_size // hp.data.hop_length, hp,
                                precision=precision)
    m.load_state_dict(sd)
    m.eval()
    return m.to("cuda")


def _model(hp, sd, precision):
    if precision not in _MODELS:
        _MODELS[precision] = _new_model(hp, sd, precision)
    return _MODELS[precision]


def _case(hp, sd64, B, T, lens):
    """Seeded prior inputs with explicit lengths (float32 for the device, float64 for the oracle) and the oracle's
    float64 enc_front, cached per (B, T, lengths)."""
    key = (B, T, tuple(lens))
    if key not in _CASES:
        d = make_inputs(300 + 7 * T + B, B, T, hp)
        c = {k: d[k] for k in ("ppg", "vec", "pit", "eps", "spk")}
        c.update({k + "64": d[k].double() for k in ("ppg", "vec", "pit", "eps", "spk")})
        c["ppg_l"] = torch.tensor(lens)
        c["mask64"] = O.sequence_mask(c["ppg_l"], T).unsqueeze(1).double()
        with torch.no_grad():
            c["front64"] = O.enc_front(sd64, c["ppg64"], c["vec64"], c["pit64"], c["mask64"])
        _CASES[key] = c
    return _CASES[key]


def run_device(m, c, hp):
    """The encoder taps and z_p from one svcb_prior call, then the flow taps from one svcb_flow call on that z_p."""
    B, T = c["pit"].shape
    enc = {k: torch.zeros(B, hp.vits.hidden_channels, T, device="cuda") for k in ENC_TAPS}
    z_p = m.prior(c["ppg"], c["vec"], c["pit"], c["ppg_l"], c["eps"], taps=enc)
    flow = {k: torch.zeros(B, hp.vits.inter_channels, T, device="cuda") for k in FLOW_TAPS}
    z = m.flow_reverse(z_p, c["ppg_l"], c["spk"], taps=flow)
    torch.cuda.synchronize()
    assert torch.equal(z, flow["flow0"])
    return {k: v.cpu().double() for k, v in {**enc, "z_p": z_p, **flow}.items()}


def stage_errors(sd64, c, got, upto=None):
    """[(tap, max-abs error, peak)] of each device tap against the float64 oracle stage fed with the device's
    previous tap, in pipeline order, stopping after `upto`.  Encoder layers count valid frames only."""
    rows = []
    mask = c["mask64"]

    def add(tap, ref):
        diff = got[tap] - ref
        if kind(tap) == "enc_layer":
            valid = mask.bool().expand_as(ref)
            diff, ref = diff[valid], ref[valid]
        rows.append((tap, float(diff.abs().max()), float(ref.abs().max())))
        return tap == upto

    with torch.no_grad():
        if add("enc_front", c["front64"]):
            return rows
        prev = got["enc_front"] * mask
        for i in range(N_LAYERS):
            if add(f"enc_layer{i}", O.enc_layer(sd64, i, prev, mask)):
                return rows
            prev = got[f"enc_layer{i}"]
        if add("z_p", O.enc_proj(sd64, prev, mask, c["eps64"])):
            return rows
        prev = got["z_p"]
        for tap in FLOW_TAPS:
            if add(tap, O.flow_step(sd64, int(tap[-1]), prev, mask, c["spk64"])):
                return rows
            prev = got[tap]
    return rows


# ------------------------------------------------------------------------------------------------ the sweep
# (B, T, lengths) around the tile edges: conv_tc computes 128 output rows per tile; rel_attn_tc 128 queries per CTA
# against 64-key tiles; the relative window reaches +-4 frames (T = 1, 4, 6 have fewer keys than the window).
# T = 2520 is the longest chunk svc_infer makes.
SWEEP = [(1, 1, [1]), (2, 4, [4, 1]), (2, 6, [6, 5]), (2, 64, [64, 63]), (3, 65, [65, 64, 1]), (2, 128, [128, 127]),
         (3, 129, [129, 128, 65]), (2, 257, [257, 129]), (2, 1000, [1000, 777]), (1, 2520, [2520])]


@pytest.mark.parametrize("precision", [0, 1, 3])
@pytest.mark.parametrize("B,T,lens", SWEEP)
def test_prior_flow_stage_vs_float64(hp, sd, sd64, B, T, lens, precision):
    c = _case(hp, sd64, B, T, lens)
    got = run_device(_model(hp, sd, precision), c, hp)
    pad = ~c["mask64"].bool()
    for tap in ["z_p"] + FLOW_TAPS:
        assert (got[tap].masked_select(pad) == 0).all(), f"{tap} is not 0 on padded frames"
    report, bad = [], []
    for tap, e, peak in stage_errors(sd64, c, got):
        rel = e / peak
        b = bound(precision, tap)
        key = (kind(tap), precision)
        if rel > _WORST.get(key, (-1.0, ""))[0]:
            _WORST[key] = (rel, f"B={B} T={T} {tap}")
        report.append(f"  {tap:10s} max-abs {e:.2e}  peak {peak:5.2f}  rel {rel:.2e}  bound {b:.0e}")
        if not e <= b * peak:
            bad.append(tap)
    print(f"\nB={B} T={T} lengths {lens} precision {precision}\n" + "\n".join(report))
    assert not bad, f"stages out of bound: {bad}\n" + "\n".join(report)


# ------------------------------------------------------------------------------------------------ dispatch
def _kernels(precision, convs, extra):
    if precision == 0:
        return {f"conv1d_fp32_{s}_o1" for s in convs} | extra
    mode = "bf16x3" if precision == 3 else "bf16"
    return {f"conv_tc_{mode}_{s}_o1" for s in convs} | extra


def prior_kernels(precision):
    """pre, hub, qkv, o, ffn1, ffn2, proj; attention on rel_attention (fp32) or rel_attn_pack + rel_attn_tc."""
    attn = {"rel_attention"} if precision == 0 else {"rel_attn_pack", "rel_attn_tc"}
    return _kernels(precision, ["1280to192_k5", "256to192_k5", "192to576_k1", "192to192_k1", "192to640_k3",
                                "640to192_k3", "192to384_k1"],
                    attn | {"pitch_embed_add", "mask_mul", "layernorm_c", "reparam"})


def flow_kernels(precision):
    """pre, the gated WN in-convs, res/skip (the last one H wide), post."""
    return _kernels(precision, ["96to192_k1", "192to384_k5", "192to384_k1", "192to192_k1", "192to96_k1"],
                    {"linear_small", "coupling_pre", "coupling_post", "wn_update"})


@pytest.mark.parametrize("precision", [0, 1, 3])
def test_dispatch_kernel_sets(hp, sd, sd64, precision):
    """The exact set of kernels one prior call and one flow call launch, so that a changed routing (run_conv's
    tensor-core predicate, the attention switch) cannot move a stage to another kernel unnoticed."""
    m = _model(hp, sd, precision)
    c = _case(hp, sd64, 3, 129, [129, 128, 65])
    z_p = []
    got_prior = launched_kernels(lambda: z_p.append(m.prior(c["ppg"], c["vec"], c["pit"], c["ppg_l"], c["eps"])))
    got_flow = launched_kernels(lambda: m.flow_reverse(z_p[0], c["ppg_l"], c["spk"]))
    print(f"\nprecision {precision}\n  prior: {sorted(got_prior)}\n  flow:  {sorted(got_flow)}")
    for got, want in ((got_prior, prior_kernels(precision)), (got_flow, flow_kernels(precision))):
        assert got == want, f"missing {sorted(want - got)}, unexpected {sorted(got - want)}"
        if precision != 0:
            assert not any(k.startswith("conv1d_fp32_") or k == "rel_attention" for k in got)


# ------------------------------------------------------------------------------------------------ the bounds see a bug
PERTURB_CASE = (3, 129, [129, 128, 65])


def _oracle_chain(hp, sd64):
    """The float64 oracle's own stages on PERTURB_CASE (cached): the inputs on which a perturbation is sized."""
    c = _case(hp, sd64, *PERTURB_CASE)
    if "chain64" not in c:
        st = {}
        with torch.no_grad():
            st["z_p"], _ = O.prior_encoder(sd64, c["ppg64"], c["ppg_l"], c["vec64"], c["pit64"], c["eps64"], stages=st)
            O.flow_reverse(sd64, st["z_p"], c["mask64"], c["spk64"], stages=st)
        c["chain64"] = st
    return c


def _spec(name, c):
    """(tap, state-dict key, change(weight, a) -> weight, oracle stage(state dict) -> tap value) of a perturbation:
    a plausible kernel bug emulated in one weight, of size a."""
    ch, mask = c["chain64"], c["mask64"]
    if name == "pit_bin":
        # pitch bin off by one: the embedding row of the most used voiced bin moves towards its neighbour's
        voiced = c["mask64"][:, 0].bool() & (c["pit"] > 0)
        k = int(O.f0_to_coarse(c["pit"])[voiced].mode().values)

        def change(w, a):
            w = w.clone()
            w[k] += a * (w[k + 1] - w[k])
            return w
        return ("enc_front", "enc_p.pit.weight", change,
                lambda s: O.enc_front(s, c["ppg64"], c["vec64"], c["pit64"], mask))
    if name.startswith("rel_"):
        # relative-key / -value band shifted by one: the table blended with its one-row roll
        i = int(name[-1])
        x = ch["enc_front"] * mask if i == 0 else ch[f"enc_layer{i - 1}"]
        return (f"enc_layer{i}", f"enc_p.enc.attn_layers.{i}.emb_{name[:5]}", lambda w, a: w + a * (w.roll(1, 1) - w),
                lambda s: O.enc_layer(s, i, x, mask))

    def bias(half=False):
        """a bias's first channel, or every channel of its second half"""
        def change(w, a):
            w = w.clone()
            if half:
                w[w.shape[0] // 2:] += a
            else:
                w[0] += a
            return w
        return change
    if name.startswith("ffn_bias"):
        i = int(name[-1])
        return (f"enc_layer{i}", f"enc_p.enc.ffn_layers.{i}.conv_2.bias", bias(),
                lambda s: O.enc_layer(s, i, ch[f"enc_layer{i - 1}"], mask))
    if name == "logs_bias":   # the logs half of proj
        return ("z_p", "enc_p.proj.bias", bias(half=True),
                lambda s: O.enc_proj(s, ch["enc_layer5"], mask, c["eps64"]))
    if name == "wn_gate_bias":   # the sigmoid (gate) half of flow 1's second WN in-conv
        return ("flow1", "flow.flows.2.enc.in_layers.1.bias", bias(half=True),
                lambda s: O.flow_step(s, 1, ch["flow2"], mask, c["spk64"]))
    assert name == "snac_bias"
    return ("flow0", "flow.flows.0.snac.bias", bias(), lambda s: O.flow_step(s, 0, ch["flow1"], mask, c["spk64"]))


def _perturb(name, precision, hp, sd, sd64):
    """The replaced state-dict entry, sized so that the float64 oracle's stage moves by 3x that stage's bound
    (secant steps on a near-linear response, computed here, not by hand)."""
    c = _oracle_chain(hp, sd64)
    tap, key, change, stage = _spec(name, c)
    ref = c["chain64"][tap]
    keep = c["mask64"].bool().expand_as(ref) if kind(tap) == "enc_layer" else torch.ones_like(ref, dtype=torch.bool)

    def moved(a):
        with torch.no_grad():
            return float((stage({**sd64, key: change(sd64[key], a)}) - ref)[keep].abs().max())
    target = 3 * bound(precision, tap) * float(ref[keep].abs().max())
    a = 1e-3
    for _ in range(4):
        a *= target / moved(a)
    assert 2.5 * target / 3 <= moved(a) <= 3.5 * target / 3
    return tap, {key: change(sd[key], a)}


PERTURBATIONS = ["pit_bin", "rel_k2", "rel_v4", "ffn_bias5", "logs_bias", "wn_gate_bias", "snac_bias"]


@pytest.mark.parametrize("precision", [3, 1])
@pytest.mark.parametrize("name", PERTURBATIONS)
def test_stage_bounds_flag_perturbed_weights(hp, sd, sd64, name, precision):
    """A plausible kernel bug emulated in the weights (device model only; the oracle keeps the original state
    dict): the stage comparator must flag the tap it lands in and no tap before it."""
    tap, new = _perturb(name, precision, hp, sd, sd64)
    m = _new_model(hp, {**sd, **new}, precision)
    c = _case(hp, sd64, *PERTURB_CASE)
    rows = stage_errors(sd64, c, run_device(m, c, hp), upto=tap)
    flagged = [t for t, e, peak in rows if e > bound(precision, t) * peak]
    report = "\n".join(f"  {t:10s} max-abs {e:.2e} peak {p:5.2f} bound {bound(precision, t) * p:.2e}" for t, e, p in rows)
    print(f"\n{name} precision {precision}\n{report}")
    assert flagged == [tap], report


# ------------------------------------------------------------------------------------------------ pitch bins
def _bin_pitches():
    """float32 pitches: every integer Hz 0..1200 shifted by -12..+12 semitones the way hostio.prepare_features
    does it (float64 product, then float32); 0, 50 and 1100 Hz (the clamps) and their float32 neighbours; and the
    float32 values whose float64 mel + 0.5 lies within 1e-4 of an integer, i.e. on the rounding edge of a bin."""
    hz, shift = np.arange(0, 1201)[:, None], np.arange(-12, 13)[None, :]
    shifted = torch.FloatTensor((hz * 2 ** (shift / 12)).reshape(-1))
    edges = torch.tensor([0.0, 50.0, 1100.0])
    clamps = torch.cat([edges, torch.nextafter(edges, torch.tensor(np.inf)), torch.nextafter(edges, torch.tensor(-np.inf))])
    n = torch.arange(2, 256, dtype=torch.float64)   # mel + 0.5 == n at the edge between bins n - 1 and n
    span = O._F0_MEL_MAX - O._F0_MEL_MIN
    f0 = 700 * torch.expm1(((n - 1.5) * span / 254 + O._F0_MEL_MIN) / 1127)
    bits = f0.float().view(torch.int32)[:, None] + torch.arange(-256, 257, dtype=torch.int32)[None, :]
    cand = bits.reshape(-1).view(torch.float32)
    mel = (1127 * torch.log1p(cand.double() / 700) - O._F0_MEL_MIN) * 254 / span + 1 + 0.5
    near = cand[(mel - mel.round()).abs() <= 1e-4]
    assert len(near) > 254
    return torch.cat([shifted, clamps, near])


def test_pitch_bins_on_device(hp, sd):
    """pitch_embed_add bins the pitch on the device (prior_ops.cu:f0_coarse).  With pre / hub zeroed and embedding
    row k = k, enc_front IS the device's bin: it must equal the oracle's float32 f0_to_coarse everywhere."""
    sd0 = dict(sd)
    for k in ("enc_p.pre.weight", "enc_p.pre.bias", "enc_p.hub.weight", "enc_p.hub.bias"):
        sd0[k] = torch.zeros_like(sd[k])
    emb = sd["enc_p.pit.weight"]
    sd0["enc_p.pit.weight"] = torch.arange(emb.shape[0], dtype=torch.float32)[:, None].expand_as(emb).contiguous()
    m = _new_model(hp, sd0, 3)
    pit = _bin_pitches()
    T = 1024
    B = -(-len(pit) // T)
    pit = torch.cat([pit, torch.zeros(B * T - len(pit))]).reshape(B, T)
    H = hp.vits.hidden_channels
    front = torch.zeros(B, H, T, device="cuda")
    m.prior(torch.zeros(B, T, hp.vits.ppg_dim), torch.zeros(B, T, hp.vits.vec_dim), pit, torch.full((B,), T),
            torch.zeros(B, hp.vits.inter_channels, T), taps={"enc_front": front})
    front = front.cpu()
    assert torch.equal(front, front[:, :1].expand_as(front))
    want = O.f0_to_coarse(pit)
    bad = (front[:, 0] != want.float())
    print(f"\n{pit.numel()} pitches, {int(bad.sum())} bins differ from the oracle's")
    assert not bad.any(), [(float(p), int(b), int(w)) for p, b, w in zip(pit[bad], front[:, 0][bad], want[bad])][:10]


# ------------------------------------------------------------------------------------------------ one path, one answer
@pytest.mark.parametrize("precision", [0, 1, 3])
def test_inference_taps_equal_stage_entry_points(hp, sd, sd64, precision):
    """svcb_infer runs the prior and the flow in the arena behind one mark; its taps must be the separate calls'."""
    m = _model(hp, sd, precision)
    c = _case(hp, sd64, *PERTURB_CASE)
    B, T = c["pit"].shape
    sep = run_device(m, c, hp)
    taps = {k: torch.zeros(B, hp.vits.hidden_channels if k in ENC_TAPS else hp.vits.inter_channels, T, device="cuda")
            for k in TAPS}
    m.inference(c["ppg"], c["vec"], c["pit"], c["spk"], c["ppg_l"], torch.zeros(B, 1, T * m.hop), eps=c["eps"],
                taps=taps)
    torch.cuda.synchronize()
    for k in TAPS:
        assert torch.equal(taps[k].cpu().double(), sep[k]), k


def test_ragged_item_equals_item_alone(hp, sd):
    """precision 3: an item of length 70 inside a B=3, T=200 ragged batch (frames past each length zero, as a
    padded batch holds them) gives the valid-frame z_p and z of the same item run alone at T=70."""
    m = _model(hp, sd, 3)
    B, T, lens = 3, 200, [200, 70, 143]
    d = make_inputs(41, B, T, hp)
    for b, n in enumerate(lens):
        d["ppg"][b, n:] = 0
        d["vec"][b, n:] = 0
    ppg_l = torch.tensor(lens)
    z_p = m.prior(d["ppg"], d["vec"], d["pit"], ppg_l, d["eps"])
    z = m.flow_reverse(z_p, ppg_l, d["spk"])
    n = lens[1]
    one = slice(1, 2)
    z_p1 = m.prior(d["ppg"][one, :n], d["vec"][one, :n], d["pit"][one, :n], ppg_l[one], d["eps"][one, :, :n])
    z1 = m.flow_reverse(z_p1, ppg_l[one], d["spk"][one])
    for name, full, alone in (("z_p", z_p, z_p1), ("z", z, z1)):
        full, alone = full[one, :, :n].cpu(), alone.cpu()
        e, peak = float((full - alone).abs().max()), float(alone.abs().max())
        print(f"{name}: item in batch vs alone max-abs {e:.2e} (peak {peak:.2f})")
        assert e <= 1e-6 * peak, name
