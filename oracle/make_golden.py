"""Generate tests/golden/*.npz by running the UNMODIFIED reference (TEST INFRASTRUCTURE).

Run in the build container only (needs /root/reference):  python oracle/make_golden.py
The reference's internal RNG calls are answered with the seeded tensors of tests/util.make_inputs
(in the order the reference draws them: torch.rand -> rand_ini, torch.randn_like -> noise, then
torch.randn_like -> eps), so the fixtures pin the reference's arithmetic, not its RNG stream.
Also asserts that oracle/svc_oracle.py reproduces every fixture.

`whisper_case` does the same for the PPG extractor: the reference's `Whisper` module is built from a
synthetic checkpoint through the loader surgery of whisper/inference.py:11-20 (decoder deleted, last
quarter of the encoder blocks deleted, strict=False load) and `model.encoder(mel)` is stored next to
the mel; oracle/whisper_oracle.py must reproduce it.
"""
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import, svc_oracle as O  # noqa: E402
from tests.util import GOLDEN, make_inputs  # noqa: E402
from whisper_vits_svc_b200 import hparams, synth  # noqa: E402


class FeedRNG:
    """Answer torch.rand / torch.randn_like with queued tensors."""

    def __init__(self, rand_q, randn_q):
        self.rand_q, self.randn_q = list(rand_q), list(randn_q)

    def __enter__(self):
        self.o = (torch.rand, torch.randn_like)

        def rand(*shape, **kw):
            t = self.rand_q.pop(0)
            assert tuple(t.shape) == tuple(shape), (t.shape, shape)
            return t.clone()

        def randn_like(x, **kw):
            t = self.randn_q.pop(0)
            assert t.shape == x.shape, (t.shape, x.shape)
            return t.clone()

        torch.rand, torch.randn_like = rand, randn_like
        return self

    def __exit__(self, *a):
        torch.rand, torch.randn_like = self.o


def ref_model(hp, sd):
    Syn = ref_import.import_synthesizer()
    m = Syn(hp.data.filter_length // 2 + 1, hp.data.segment_size // hp.data.hop_length,
            ref_import.to_attr(hp)).eval()
    m.load_state_dict(sd)
    return m


def full_case(name, hp, seed, B, T, ragged):
    sd = synth.svc_state_dict(hp, 1234)
    m = ref_model(hp, sd)
    d = make_inputs(seed, B, T, hp, ragged=ragged)
    with torch.no_grad(), FeedRNG([d["rand_ini"]], [d["noise"], d["eps"]]):
        src = m.pitch2source(d["pit"])
        wave = m.inference(d["ppg"], d["vec"], d["pit"], d["spk"], d["ppg_l"], src)
    st = {}
    src_o = O.pitch2source(sd, hp, d["pit"], d["rand_ini"], d["noise"])
    wave_o = O.synthesizer_infer(sd, hp, d["ppg"], d["vec"], d["pit"], d["spk"], d["ppg_l"], src_o, d["eps"], stages=st)
    assert torch.equal(src, src_o) or (src - src_o).abs().max() < 1e-6, "oracle source != reference"
    err = (wave - wave_o).abs().max().item()
    assert err < 1e-5, f"oracle wave != reference ({err})"
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), seed=seed, B=B, T=T, ragged=int(ragged),
                        source=src.numpy(), wave=wave.numpy(), z_p=st["z_p"].numpy(), z=st["z"].numpy(),
                        pcm=m.source2wav(src[:1]))
    print(name, "wave peak %.3f" % wave.abs().max().item(), "oracle-vs-reference max abs", err)


def gen_case(name, hp, seed, B, T):
    """BASELINE config #2 shape family: Generator.inference on a random latent."""
    sd = synth.svc_state_dict(hp, 1234)
    ref_import._ensure_path()
    from vits_decoder.generator import Generator
    g = Generator(ref_import.to_attr(hp))
    torch.nn.Module.eval(g)
    g.load_state_dict({k[4:]: v for k, v in sd.items() if k.startswith("dec.")})
    d = make_inputs(seed, B, T, hp, gen_only=True)
    with torch.no_grad(), FeedRNG([d["rand_ini"]], [d["noise"]]):
        src = g.pitch2source(d["pit"])
        wave = g.inference(d["spk"], d["z"], src)
    wave_o = O.generator(sd, hp, d["spk"], d["z"], O.pitch2source(sd, hp, d["pit"], d["rand_ini"], d["noise"]))
    err = (wave - wave_o).abs().max().item()
    assert err < 1e-5, err
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), seed=seed, B=B, T=T, source=src.numpy(), wave=wave.numpy())
    print(name, "wave peak %.3f" % wave.abs().max().item(), "oracle-vs-reference max abs", err)


WHISPER_CASES = {
    # name: (dims overrides, checkpoint seed, B, n_frames, input seed)
    "whisper_d256_l8_b2_n200": (dict(n_audio_state=256, n_audio_head=4, n_audio_layer=8), 21, 2, 200, 31),
    "whisper_d512_l4_b1_n301": (dict(n_audio_state=512, n_audio_head=8, n_audio_layer=4), 22, 1, 301, 32),
}
_SMALL_TEXT = dict(n_vocab=64, n_text_ctx=8, n_text_state=64, n_text_head=1, n_text_layer=1)


def whisper_dims(over):
    return dict(synth.WHISPER_LARGE_V2_DIMS, **_SMALL_TEXT, **over)


def whisper_mel(seed, B, n):
    """SURVEY.md §8d config 3 input recipe: N(0,1) clipped to the log-mel range [-1, 1.5]."""
    return torch.randn(B, 80, n, generator=torch.Generator().manual_seed(seed)).clamp(-1, 1.5)


def ref_whisper(ck):
    """whisper/inference.py:11-20 verbatim in effect (the checkpoint is passed in, not read from disk)."""
    wm = ref_import.import_whisper_model()
    model = wm.Whisper(wm.ModelDimensions(**ck["dims"]))
    del model.decoder
    cut = len(model.encoder.blocks) // 4
    cut = -1 * cut
    del model.encoder.blocks[cut:]
    model.load_state_dict(ck["model_state_dict"], strict=False)
    model.eval()
    return model


def whisper_case(name):
    from oracle import whisper_oracle as WO
    over, ck_seed, B, n, in_seed = WHISPER_CASES[name]
    ck = synth.whisper_checkpoint(whisper_dims(over), seed=ck_seed)
    mel = whisper_mel(in_seed, B, n)
    with torch.no_grad():
        ppg = ref_whisper(ck).encoder(mel)
    ppg_o = WO.audio_encoder(ck, mel)
    err = (ppg - ppg_o).abs().max().item()
    assert err < 1e-5, f"whisper oracle != reference ({err})"
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), mel=mel.numpy(), ppg=ppg.numpy())
    print(name, "ppg rms %.3f" % ppg.pow(2).mean().sqrt().item(), "oracle-vs-reference max abs", err)


HUBERT_CASES = {  # name: (checkpoint seed, B, n_samples, input seed)
    "hubert_soft_b2_n8000": (31, 2, 8000, 32),
    "hubert_soft_b1_n16123": (33, 1, 16123, 34),
}


def hubert_wav(seed, B, n):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n) / 16000.0
    tone = 0.3 * torch.sin(2 * math.pi * 220.0 * t)[None, :] * (1.0 + 0.5 * torch.sin(2 * math.pi * 3.0 * t))[None, :]
    return (tone + 0.1 * torch.randn(B, n, generator=g)).float().unsqueeze(1)


def ref_hubert(sd):
    """hubert/hubert_model.py:212-222 in effect (the state dict is passed in, not read from disk)."""
    hm = ref_import.import_hubert_model()
    model = hm.HubertSoft()
    model.load_state_dict(sd)
    return model.eval()


def hubert_case(name):
    from oracle import hubert_oracle as HO
    ck_seed, B, n, in_seed = HUBERT_CASES[name]
    sd = synth.hubert_checkpoint(ck_seed)
    wav = hubert_wav(in_seed, B, n)
    units = ref_hubert(sd).units(wav)
    units_o = HO.units(sd, wav)
    err = (units - units_o).abs().max().item()
    assert err < 2e-5, f"hubert oracle != reference ({err})"
    assert units.shape[1] == HO.frames(n)
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), wav=wav.numpy(), units=units.numpy())
    print(name, tuple(units.shape), "units rms %.3f" % units.pow(2).mean().sqrt().item(), "oracle-vs-reference max abs", err)


LIVE_WHISPER = [(dict(n_audio_state=256, n_audio_head=4, n_audio_layer=8), 2, 120),
                (dict(n_audio_state=384, n_audio_head=6, n_audio_layer=4), 1, 77)]
LIVE_THREADS = 8   # CPU matmuls split their sums by thread count: the tests run the oracle with this many too


def live_case(name, hp):
    """What the *_reference_live tests of tests/test_oracle_cpu.py compare the oracle with: the reference's outputs
    on their inputs (each as tests.util.seeded_sample plus `<key>_shape`), the number of Whisper encoder blocks the
    loader keeps, the layout (names, shapes as "d0,d1,...") and alias-filter taps of a fresh SynthesizerInfer, and
    the intra-op thread count the outputs were computed with."""
    from tests.util import seeded_sample
    torch.set_num_threads(LIVE_THREADS)
    out, arrays = {}, {"threads": np.int64(LIVE_THREADS)}
    sd = synth.svc_state_dict(hp, 1234)
    d = make_inputs(77, 2, 33, hp, ragged=True)
    with torch.no_grad(), FeedRNG([d["rand_ini"]], [d["noise"], d["eps"]]):
        m = ref_model(hp, sd)
        out["infer_source"] = m.pitch2source(d["pit"])
        out["infer_wave"] = m.inference(d["ppg"], d["vec"], d["pit"], d["spk"], d["ppg_l"], out["infer_source"])
    for over, B, n in LIVE_WHISPER:
        key = f"whisper_d{over['n_audio_state']}_b{B}_n{n}"
        model = ref_whisper(synth.whisper_checkpoint(whisper_dims(over), seed=5))
        with torch.no_grad():
            out[key] = model.encoder(whisper_mel(6, B, n))
        arrays[key + "_blocks"] = np.int64(len(model.encoder.blocks))
    out["hubert_b1_n5003"] = ref_hubert(synth.hubert_checkpoint(7)).units(hubert_wav(8, 1, 5003))
    for k, v in out.items():
        arrays[k] = seeded_sample(v).numpy()
        arrays[k + "_shape"] = np.array(v.shape, dtype=np.int64)
    fresh = ref_import.import_synthesizer()(hp.data.filter_length // 2 + 1, hp.data.segment_size // hp.data.hop_length,
                                             ref_import.to_attr(hp)).state_dict()
    arrays["sd_keys"] = np.array(list(fresh))
    arrays["sd_shapes"] = np.array([",".join(map(str, v.shape)) for v in fresh.values()])
    arrays["sd_filter"] = fresh["dec.activation_post.upsample.filter"].numpy()
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **arrays)
    print(name, {k: tuple(v.shape) for k, v in out.items()})


if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    hp = hparams.load_hparams(os.path.join(ROOT, "configs", "base.yaml"))
    full_case("infer_b2_t48", hp, seed=11, B=2, T=48, ragged=False)
    full_case("infer_b3_t70_ragged", hp, seed=12, B=3, T=70, ragged=True)
    hp24 = hparams.override(hp, gen__upsample_input=80, data__sampling_rate=24000)
    gen_case("gen80_b2_t36", hp24, seed=13, B=2, T=36)
    gen_case("gen192_b1_t64", hp, seed=14, B=1, T=64)
    for name in WHISPER_CASES:
        whisper_case(name)
    for name in HUBERT_CASES:
        hubert_case(name)
    live_case("reference_live", hp)
