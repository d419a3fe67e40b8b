"""The oracle generator split into stages (gen_pre, gen_up, gen_amp_stage, gen_post), which the per-stage GPU
tests in test_generator_stages_gpu.py feed with the device's own taps: the composition is generator() exactly,
and every stage runs in float64 when given a float64 state dict."""
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
