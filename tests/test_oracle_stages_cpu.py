"""The oracle generator split into stages (gen_pre, gen_up, gen_amp_stage, gen_post) and the prior encoder and flow
split likewise (enc_front, enc_layer, enc_proj, flow_step), which the per-stage GPU tests in
test_generator_stages_gpu.py and test_prior_flow_stages_gpu.py feed with the device's own taps: each composition is
the whole-path function exactly, and every stage runs in float64 when given a float64 state dict."""
import pytest
import torch

from oracle import svc_oracle as O
from tests.util import make_inputs, max_abs

N_UPS = 5


def _staged(sd, hp, spk, z, src):
    taps = {"gen_pre": O.gen_pre(sd, spk, z)}
    x = taps["gen_pre"]
    for i in range(N_UPS):
        x = taps[f"gen_up{i}"] = O.gen_up(sd, hp, i, x, src)
        x = taps[f"gen_stage{i}"] = O.gen_amp_stage(sd, hp, i, x)
    return O.gen_post(sd, x), taps


@pytest.fixture(scope="module")
def gen_case(hp, sd):
    d = make_inputs(61, 2, 13, hp, gen_only=True)
    src = O.pitch2source(sd, hp, d["pit"], d["rand_ini"], d["noise"])
    return d["spk"], d["z"], src


def test_staged_composition_equals_generator(hp, sd, gen_case):
    spk, z, src = gen_case
    st = {}
    with torch.no_grad():
        wave = O.generator(sd, hp, spk, z, src, stages=st)
        wave_s, taps = _staged(sd, hp, spk, z, src)
    assert len(hp.gen.upsample_rates) == N_UPS
    assert set(taps) == set(st)
    for k in st:
        assert torch.equal(taps[k], st[k]), k
    assert torch.equal(wave_s, wave)


def test_float64_stages_agree_with_float32(hp, sd, gen_case):
    """Each stage of the float64 chain against the float32 one: the float32 oracle's own rounding, a few 1e-6
    (1e-6 at gen_pre to ~6e-6 at gen_stage4 for T=129).  A piece that silently dropped to float32 (a float32
    constant or buffer) would show as an exact match; one that broke would show as a large gap."""
    spk, z, src = gen_case
    sd64 = {k: v.double() for k, v in sd.items()}
    with torch.no_grad():
        wave32, t32 = _staged(sd, hp, spk, z, src)
        wave64, t64 = _staged(sd64, hp, spk.double(), z.double(), src.double())
    assert wave64.dtype == torch.float64 and all(v.dtype == torch.float64 for v in t64.values())
    report = []
    for k in list(t32) + ["wave"]:
        a, b = (wave32, wave64) if k == "wave" else (t32[k], t64[k])
        e = float((a.double() - b).abs().max())
        report.append(f"{k:11s} fp32-vs-fp64 max-abs {e:.2e} (peak {float(b.abs().max()):.2f})")
        assert 0.0 < e <= 2e-5, "\n".join(report)
    print("\n".join(report))
    assert max_abs(wave32, wave64) <= 2e-5


# ------------------------------------------------------------------------------------------------ prior encoder + flow
N_LAYERS, N_FLOWS = 6, 4
PRIOR_CASES = [(2, 90, [90, 54]), (1, 2520, [2520])]


def _prior_inputs(hp, B, T, lens, dtype=torch.float32):
    d = make_inputs(11 + T, B, T, hp)
    d["ppg_l"] = torch.tensor(lens)
    d = {k: v.to(dtype) if v.is_floating_point() else v for k, v in d.items()}
    d["mask"] = O.sequence_mask(d["ppg_l"], T).unsqueeze(1).to(dtype)
    return d


def _staged_prior_flow(sd, d):
    """enc_front -> enc_layer0..5 -> enc_proj (z_p) -> flow_step 3..0, as the per-stage GPU tests chain them."""
    mask = d["mask"]
    taps = {"enc_front": O.enc_front(sd, d["ppg"], d["vec"], d["pit"], mask)}
    x = taps["enc_front"] * mask
    for i in range(N_LAYERS):
        x = taps[f"enc_layer{i}"] = O.enc_layer(sd, i, x, mask)
    x = taps["z_p"] = O.enc_proj(sd, x, mask, d["eps"])
    for i in reversed(range(N_FLOWS)):
        x = taps[f"flow{i}"] = O.flow_step(sd, i, x, mask, d["spk"])
    return taps


def test_staged_composition_equals_prior_and_flow(hp, sd):
    d = _prior_inputs(hp, *PRIOR_CASES[0])
    st = {}
    with torch.no_grad():
        z_p, mask = O.prior_encoder(sd, d["ppg"], d["ppg_l"], d["vec"], d["pit"], d["eps"], stages=st)
        z = O.flow_reverse(sd, z_p, mask, d["spk"], stages=st)
        taps = _staged_prior_flow(sd, d)
    assert torch.equal(mask, d["mask"])
    st["z_p"] = z_p
    assert set(taps) == set(st)
    for k in st:
        assert torch.equal(taps[k], st[k]), k
    assert torch.equal(taps["flow0"], z)


@pytest.mark.parametrize("B,T,lens", PRIOR_CASES)
def test_prior_flow_float64_stages_agree_with_float32(hp, sd, B, T, lens):
    """Each stage of the float64 prior/flow chain against the float32 one, over all frames (the flow steps carry
    z_p's float32 error on): 1.8e-6 to 2.4e-6 at enc_front, 1.9e-6 to 6.4e-6 at the encoder layers, 5e-6 to
    1.0e-5 at z_p and the flows (peaks 3.5 to 14).  An exact match would mean a piece dropped to float32."""
    sd64 = {k: v.double() for k, v in sd.items()}
    with torch.no_grad():
        t32 = _staged_prior_flow(sd, _prior_inputs(hp, B, T, lens))
        t64 = _staged_prior_flow(sd64, _prior_inputs(hp, B, T, lens, torch.float64))
    assert all(v.dtype == torch.float64 for v in t64.values())
    report = []
    for k in t32:
        e = float((t32[k].double() - t64[k]).abs().max())
        report.append(f"{k:10s} fp32-vs-fp64 max-abs {e:.2e} (peak {float(t64[k].abs().max()):.2f})")
        assert 0.0 < e <= 3e-5, "\n".join(report)
    print("\n".join(report))


def test_f0_bin_uses_float32_pitch():
    """enc_front bins a float64 pitch as its float32 value: float32 arithmetic puts 256.29599 Hz in bin 72 and
    float64 in bin 71, and the reference (and the device) bin in float32."""
    p32 = torch.tensor([256.2959899902344])
    assert int(O.f0_to_coarse(p32)) == 72 and int(O.f0_to_coarse(p32.double())) == 71
    sd = {"enc_p.pit.weight": torch.arange(256, dtype=torch.float64)[:, None].expand(256, 4).contiguous(),
          "enc_p.pre.weight": torch.zeros(4, 3, 5, dtype=torch.float64), "enc_p.pre.bias": torch.zeros(4, dtype=torch.float64),
          "enc_p.hub.weight": torch.zeros(4, 2, 5, dtype=torch.float64), "enc_p.hub.bias": torch.zeros(4, dtype=torch.float64)}
    front = O.enc_front(sd, torch.zeros(1, 1, 3, dtype=torch.float64), torch.zeros(1, 1, 2, dtype=torch.float64),
                        p32.double()[None], torch.ones(1, 1, 1, dtype=torch.float64))
    assert torch.equal(front[0, :, 0], torch.full((4,), float(O.f0_to_coarse(p32)), dtype=torch.float64))


def test_padded_frames_do_not_matter(hp, sd):
    """The per-stage GPU tests feed each oracle stage the device's previous tap, whose padded frames hold whatever
    the kernels left there.  In float64 an encoder layer's valid frames are bit-for-bit independent of the padded
    frames of its input (masked keys get exp(-1e4 - max) = 0 weight; the FFN masks its inputs), and z_p and every
    flow output are exactly 0 on padded frames."""
    sd64 = {k: v.double() for k, v in sd.items()}
    d = _prior_inputs(hp, *PRIOR_CASES[0], dtype=torch.float64)
    valid = d["mask"].bool().expand(-1, hp.vits.hidden_channels, -1)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        taps = _staged_prior_flow(sd64, d)
        for i in range(N_LAYERS):
            x = taps["enc_front"] * d["mask"] if i == 0 else taps[f"enc_layer{i - 1}"]
            junk = torch.where(valid, x, 1e3 * torch.randn(x.shape, generator=g, dtype=torch.float64))
            assert not torch.equal(junk, x)
            y = O.enc_layer(sd64, i, junk, d["mask"])
            assert torch.equal(y[valid], taps[f"enc_layer{i}"][valid]), i
        junk = torch.where(valid, taps["enc_layer5"], 1e3 * torch.randn(valid.shape, generator=g, dtype=torch.float64))
        assert torch.equal(O.enc_proj(sd64, junk, d["mask"], d["eps"]), taps["z_p"])
    pad = ~d["mask"].bool()
    assert pad.any()
    for k in ["z_p"] + [f"flow{i}" for i in range(N_FLOWS)]:
        assert (taps[k].masked_select(pad) == 0).all(), k
