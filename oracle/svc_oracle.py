"""CPU oracle for the SVC inference hot path (TEST INFRASTRUCTURE, not product code).

A functional, torch-CPU fp32 restatement of the reference's algorithm for
`SynthesizerInfer.inference` / `pitch2source` / `source2wav`.  It consumes the
reference's *own* checkpoint format (the 903-entry `model_g` state-dict with
`weight_g`/`weight_v` pairs) and takes every random draw of the reference as an
explicit input, so the CUDA path and the oracle can be compared on identical
numbers.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline /
`--impl reference` leg may import this module.  The product path
(`whisper-vits-svc_b200`) never does.

Parity status: the reference ships no tests or golden vectors (SURVEY.md §4),
so the pin is the reference code itself: `oracle/make_golden.py` imports
`/root/reference` in the build container, checks this restatement against it
(tests/test_oracle_cpu.py::test_oracle_matches_reference_live does the same when the
reference is present) and writes `tests/golden/*.npz`, which travel to the GPU box.

Reference citations are relative to /root/reference.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

SD = Dict[str, torch.Tensor]


# --------------------------------------------------------------------------- helpers
def fold_weight_norm(sd: SD, prefix: str) -> torch.Tensor:
    """w = g * v / ||v|| with the norm over every dim but 0
    (torch.nn.utils.weight_norm default dim=0; generator.py:73, bigv.py:23-38,
    modules.py:153,165,175).  Plain `weight` is returned when the pair is absent
    (checkpoint written after remove_weight_norm)."""
    if prefix + ".weight" in sd:
        return sd[prefix + ".weight"]
    v = sd[prefix + ".weight_v"]
    g = sd[prefix + ".weight_g"]
    return torch._weight_norm(v, g, 0)


def sequence_mask(lengths: torch.Tensor, max_len: int) -> torch.Tensor:
    """vits/commons.py:147-151"""
    pos = torch.arange(max_len, dtype=lengths.dtype, device=lengths.device)
    return pos[None, :] < lengths[:, None]


_F0_MEL_MIN = 1127 * np.log(1 + 50.0 / 700)
_F0_MEL_MAX = 1127 * np.log(1 + 1100.0 / 700)


def f0_to_coarse(f0: torch.Tensor) -> torch.Tensor:
    """vits/utils.py:20-33 (torch branch): mel-scale, affine to 1..255, +0.5, truncate."""
    mel = 1127 * (1 + f0 / 700).log()
    pos = mel > 0
    mel = torch.where(pos, (mel - _F0_MEL_MIN) * 254 / (_F0_MEL_MAX - _F0_MEL_MIN) + 1, mel)
    mel = torch.where(mel <= 1, torch.ones_like(mel), mel)
    mel = torch.where(mel > 255, torch.full_like(mel, 255.0), mel)
    return (mel + 0.5).long()


def channel_layer_norm(x: torch.Tensor, gamma, beta, eps=1e-5) -> torch.Tensor:
    """vits/modules.py:19-22 — LayerNorm over the channel dim of [B,C,T]."""
    return F.layer_norm(x.transpose(1, -1), (x.shape[1],), gamma, beta, eps).transpose(1, -1)


# --------------------------------------------------------------------------- prior encoder
def _rel_embeddings(emb: torch.Tensor, length: int, window: int = 4) -> torch.Tensor:
    """vits/attentions.py:294-312: zero-pad the (2w+1)-row table to 2T-1 rows."""
    pad = max(length - (window + 1), 0)
    start = max((window + 1) - length, 0)
    if pad > 0:
        emb = F.pad(emb, (0, 0, pad, pad))
    return emb[:, start:start + 2 * length - 1]


def _rel_to_abs(x: torch.Tensor) -> torch.Tensor:
    """vits/attentions.py:314-331: [b,h,l,2l-1] -> [b,h,l,l] by the pad/reshape skew."""
    b, h, l, _ = x.shape
    x = F.pad(x, (0, 1))
    flat = F.pad(x.reshape(b, h, l * 2 * l), (0, l - 1))
    return flat.reshape(b, h, l + 1, 2 * l - 1)[:, :, :l, l - 1:]


def _abs_to_rel(x: torch.Tensor) -> torch.Tensor:
    """vits/attentions.py:333-346: [b,h,l,l] -> [b,h,l,2l-1]."""
    b, h, l, _ = x.shape
    x = F.pad(x, (0, l - 1))
    flat = F.pad(x.reshape(b, h, l * l + l * (l - 1)), (l, 0))
    return flat.reshape(b, h, l, 2 * l)[:, :, :, 1:]


def rel_attention(sd: SD, p: str, x: torch.Tensor, attn_mask: torch.Tensor, n_heads=2, window=4):
    """vits/attentions.py:215-274 (self-attention, heads share the 9-row tables)."""
    q = F.conv1d(x, sd[p + ".conv_q.weight"], sd[p + ".conv_q.bias"])
    k = F.conv1d(x, sd[p + ".conv_k.weight"], sd[p + ".conv_k.bias"])
    v = F.conv1d(x, sd[p + ".conv_v.weight"], sd[p + ".conv_v.bias"])
    b, d, t = q.shape
    dk = d // n_heads
    q = q.view(b, n_heads, dk, t).transpose(2, 3)
    k = k.view(b, n_heads, dk, t).transpose(2, 3)
    v = v.view(b, n_heads, dk, t).transpose(2, 3)
    qs = q / math.sqrt(dk)
    scores = torch.matmul(qs, k.transpose(-2, -1))
    rel_k = _rel_embeddings(sd[p + ".emb_rel_k"], t, window)
    scores = scores + _rel_to_abs(torch.matmul(qs, rel_k.unsqueeze(0).transpose(-2, -1)))
    scores = scores.masked_fill(attn_mask == 0, -1e4)
    pa = F.softmax(scores, dim=-1)
    out = torch.matmul(pa, v)
    rel_v = _rel_embeddings(sd[p + ".emb_rel_v"], t, window)
    out = out + torch.matmul(_abs_to_rel(pa), rel_v.unsqueeze(0))
    out = out.transpose(2, 3).contiguous().view(b, d, t)
    return F.conv1d(out, sd[p + ".conv_o.weight"], sd[p + ".conv_o.bias"])


def ffn(sd: SD, p: str, x: torch.Tensor, mask: torch.Tensor, k: int = 3):
    """vits/attentions.py:390-398 with `_same_padding` (:409-416), ReLU branch."""
    pl, pr = (k - 1) // 2, k // 2
    h = F.conv1d(F.pad(x * mask, (pl, pr)), sd[p + ".conv_1.weight"], sd[p + ".conv_1.bias"])
    h = torch.relu(h)
    h = F.conv1d(F.pad(h * mask, (pl, pr)), sd[p + ".conv_2.weight"], sd[p + ".conv_2.bias"])
    return h * mask


def enc_front(sd: SD, ppg, vec, pit, mask):
    """pre + hub + pitch embedding, vits/models.py:40-47, before Encoder.forward's `x * x_mask`.
    The pitch bin is computed from the float32 pitch whatever the dtype of the rest: the reference reads
    pitch as a FloatTensor and bins it in float32, and float64 arithmetic puts some pitches in the
    neighbouring bin."""
    f0c = f0_to_coarse(pit.float())
    x = F.conv1d(ppg.transpose(1, -1), sd["enc_p.pre.weight"], sd["enc_p.pre.bias"], padding=2) * mask
    v = F.conv1d(vec.transpose(1, -1), sd["enc_p.hub.weight"], sd["enc_p.hub.bias"], padding=2) * mask
    return x + v + F.embedding(f0c, sd["enc_p.pit.weight"]).transpose(1, 2)


def enc_layer(sd: SD, i: int, x, mask):
    """Encoder layer i (attention + FFN, each with its residual LayerNorm), attentions.py:63-71.
    Layer 0 expects x already multiplied by the mask (attentions.py:62)."""
    e = "enc_p.enc."
    attn_mask = mask.unsqueeze(2) * mask.unsqueeze(-1)
    y = rel_attention(sd, f"{e}attn_layers.{i}", x, attn_mask)
    x = channel_layer_norm(x + y, sd[f"{e}norm_layers_1.{i}.gamma"], sd[f"{e}norm_layers_1.{i}.beta"])
    y = ffn(sd, f"{e}ffn_layers.{i}", x, mask)
    return channel_layer_norm(x + y, sd[f"{e}norm_layers_2.{i}.gamma"], sd[f"{e}norm_layers_2.{i}.beta"])


def enc_proj(sd: SD, x, mask, eps):
    """Encoder's final mask, proj and the reparameterisation, attentions.py:72 + vits/models.py:49-51 -> z_p."""
    x = x * mask
    stats = F.conv1d(x, sd["enc_p.proj.weight"], sd["enc_p.proj.bias"]) * mask
    m, logs = torch.split(stats, stats.shape[1] // 2, dim=1)
    return (m + eps * torch.exp(logs)) * mask


def prior_encoder(sd: SD, ppg, ppg_l, vec, pit, eps, n_layers=6, stages: Optional[dict] = None):
    """TextEncoder.forward, vits/models.py:39-52; Encoder.forward attentions.py:60-72.
    `eps` replaces torch.randn_like(m) at models.py:51."""
    mask = sequence_mask(ppg_l, ppg.shape[1]).unsqueeze(1).to(ppg.dtype)
    x = enc_front(sd, ppg, vec, pit, mask)
    if stages is not None:
        stages["enc_front"] = x
    x = x * mask
    for i in range(n_layers):
        x = enc_layer(sd, i, x, mask)
        if stages is not None:
            stages[f"enc_layer{i}"] = x
    return enc_proj(sd, x, mask, eps), mask


# --------------------------------------------------------------------------- flow
def wavenet(sd: SD, p: str, x, mask, n_layers=4, hidden=192, k=5):
    """WN.forward, vits/modules.py:178-203, g=None branch; gate = commons.py:126-133."""
    out = torch.zeros_like(x)
    for i in range(n_layers):
        w = fold_weight_norm(sd, f"{p}.in_layers.{i}")
        a = F.conv1d(x, w, sd[f"{p}.in_layers.{i}.bias"], padding=(k - 1) // 2)
        acts = torch.tanh(a[:, :hidden]) * torch.sigmoid(a[:, hidden:])
        w = fold_weight_norm(sd, f"{p}.res_skip_layers.{i}")
        rs = F.conv1d(acts, w, sd[f"{p}.res_skip_layers.{i}.bias"])
        if i < n_layers - 1:
            x = (x + rs[:, :hidden]) * mask
            out = out + rs[:, hidden:]
        else:
            out = out + rs
    return out * mask


def coupling_reverse(sd: SD, p: str, x, mask, spk):
    """ResidualCouplingLayer.forward(reverse=True), vits/modules.py:288-302,313-318 (mean_only)."""
    half = x.shape[1] // 2
    s = F.conv1d(spk.unsqueeze(-1), sd[p + ".snac.weight"], sd[p + ".snac.bias"])
    s_m, s_v = s.chunk(2, dim=1)
    x0, x1 = x[:, :half], x[:, half:]
    x0n = (x0 - s_m) * torch.exp(-s_v) * mask
    h = F.conv1d(x0n, sd[p + ".pre.weight"], sd[p + ".pre.bias"]) * mask
    h = wavenet(sd, p + ".enc", h, mask)
    m = F.conv1d(h, sd[p + ".post.weight"], sd[p + ".post.bias"]) * mask
    x1 = (x1 - m) * mask  # logs == 0 -> exp(-logs) == 1
    x1 = (s_m + x1 * torch.exp(s_v)) * mask
    return torch.cat([x0, x1], 1)


def flow_step(sd: SD, i: int, x, mask, spk):
    """Flip (modules.py:225-229) then coupling layer i in reverse (`flow.flows.{2i}`)."""
    return coupling_reverse(sd, f"flow.flows.{2 * i}", torch.flip(x, [1]), mask, spk)


def flow_reverse(sd: SD, z_p, mask, spk, n_flows=4, stages: Optional[dict] = None):
    """ResidualCouplingBlock.forward(reverse=True), vits/models.py:89-94: reversed([RCL,Flip]*4)."""
    x = z_p
    for i in reversed(range(n_flows)):
        x = flow_step(sd, i, x, mask, spk)
        if stages is not None:
            stages[f"flow{i}"] = x
    return x


# --------------------------------------------------------------------------- generator
def snake_alias(sd: SD, p: str, x: torch.Tensor) -> torch.Tensor:
    """SnakeAlias.forward alias/act.py:124-128 = UpSample1d (resample.py:25-33) ->
    SnakeBeta log-scale (act.py:79-92) -> DownSample1d (filter.py:86-94)."""
    c = x.shape[1]
    fu = sd[p + ".upsample.filter"]
    fd = sd[p + ".downsample.lowpass.filter"]
    ku = fu.shape[-1]
    ratio = 2
    pad = ku // ratio - 1
    pl = pad * ratio + (ku - ratio) // 2
    pr = pad * ratio + (ku - ratio + 1) // 2
    u = F.pad(x, (pad, pad), mode="replicate")
    u = ratio * F.conv_transpose1d(u, fu.expand(c, -1, -1), stride=ratio, groups=c)
    u = u[..., pl:-pr]
    alpha = torch.exp(sd[p + ".act.alpha"])[None, :, None]
    beta = torch.exp(sd[p + ".act.beta"])[None, :, None]
    u = u + (1.0 / (beta + 1e-9)) * torch.sin(u * alpha) ** 2
    kd = fd.shape[-1]
    u = F.pad(u, (kd // 2 - (1 - kd % 2), kd // 2), mode="replicate")
    return F.conv1d(u, fd.expand(c, -1, -1), stride=ratio, groups=c)


def amp_block(sd: SD, p: str, x: torch.Tensor, k: int, dilations=(1, 3, 5)) -> torch.Tensor:
    """AMPBlock.forward, vits_decoder/bigv.py:50-58."""
    for j, d in enumerate(dilations):
        t = snake_alias(sd, f"{p}.activations.{2 * j}", x)
        t = F.conv1d(t, fold_weight_norm(sd, f"{p}.convs1.{j}"), sd[f"{p}.convs1.{j}.bias"],
                     dilation=d, padding=d * (k - 1) // 2)
        t = snake_alias(sd, f"{p}.activations.{2 * j + 1}", t)
        t = F.conv1d(t, fold_weight_norm(sd, f"{p}.convs2.{j}"), sd[f"{p}.convs2.{j}.bias"],
                     padding=(k - 1) // 2)
        x = t + x
    return x


def gen_pre(sd: SD, spk, x):
    """SpeakerAdapter (vits_decoder/generator.py:36-47) + conv_pre + Mish (generator.py:178-181)."""
    # SpeakerAdapter: biased variance, eps inside the sqrt
    xt = x.transpose(1, -1)
    mean = xt.mean(dim=-1, keepdim=True)
    var = ((xt - mean) ** 2).mean(dim=-1, keepdim=True)
    y = (xt - mean) / (var + 1e-5).sqrt()
    scale = F.linear(spk, sd["dec.adapter.W_scale.weight"], sd["dec.adapter.W_scale.bias"])
    bias = F.linear(spk, sd["dec.adapter.W_bias.weight"], sd["dec.adapter.W_bias.bias"])
    y = y * scale.unsqueeze(1) + bias.unsqueeze(1)
    x = y.transpose(1, -1)
    x = F.conv1d(x, sd["dec.conv_pre.weight"], sd["dec.conv_pre.bias"], padding=3)
    return x * torch.tanh(F.softplus(x))


def gen_up(sd: SD, hp, i: int, x, source):
    """Up-sampling stage i: ups[i] (ConvTranspose1d) + noise_convs[i](source), generator.py:183-186."""
    rates = list(hp.gen.upsample_rates)
    u, k = rates[i], list(hp.gen.upsample_kernel_sizes)[i]
    w = fold_weight_norm(sd, f"dec.ups.{i}")
    x = F.conv_transpose1d(x, w, sd[f"dec.ups.{i}.bias"], stride=u, padding=(k - u) // 2)
    nw = sd[f"dec.noise_convs.{i}.weight"]
    if i + 1 < len(rates):
        s = int(np.prod(rates[i + 1:]))
        return x + F.conv1d(source, nw, sd[f"dec.noise_convs.{i}.bias"], stride=s, padding=s // 2)
    return x + F.conv1d(source, nw, sd[f"dec.noise_convs.{i}.bias"])


def gen_amp_stage(sd: SD, hp, i: int, x):
    """The mean of stage i's n_res AMP blocks, generator.py:188-194."""
    rk = list(hp.gen.resblock_kernel_sizes)
    rd = [tuple(d) for d in hp.gen.resblock_dilation_sizes]
    acc = None
    for j, kk in enumerate(rk):
        r = amp_block(sd, f"dec.resblocks.{i * len(rk) + j}", x, kk, rd[j])
        acc = r if acc is None else acc + r
    return acc / len(rk)


def gen_post(sd: SD, x):
    """activation_post + conv_post + tanh, generator.py:196-199."""
    x = snake_alias(sd, "dec.activation_post", x)
    x = F.conv1d(x, sd["dec.conv_post.weight"], None, padding=3)
    return torch.tanh(x)


def generator(sd: SD, hp, spk, x, source, stages: Optional[dict] = None):
    """Generator.inference, vits_decoder/generator.py:175-200 (+ SpeakerAdapter :36-47).
    Runs in the dtype of its arguments: a float64 state dict and inputs give a float64 generator."""
    x = gen_pre(sd, spk, x)
    if stages is not None:
        stages["gen_pre"] = x
    for i in range(len(hp.gen.upsample_rates)):
        x = gen_up(sd, hp, i, x, source)
        if stages is not None:
            stages[f"gen_up{i}"] = x
        x = gen_amp_stage(sd, hp, i, x)
        if stages is not None:
            stages[f"gen_stage{i}"] = x
    return gen_post(sd, x)


# --------------------------------------------------------------------------- NSF source
def pitch2source(sd: SD, hp, f0: torch.Tensor, rand_ini: torch.Tensor, noise: torch.Tensor):
    """Generator.pitch2source generator.py:160-165 -> SourceModuleHnNSF.forward nsf.py:383-394 ->
    SineGen.forward/_f02sine nsf.py:217-316.
    f0 [B,T] Hz; rand_ini [B,11] replaces torch.rand (nsf.py:232-235, column 0 is forced to 0 here
    as the reference does); noise [B,T*hop,11] replaces torch.randn_like (nsf.py:311)."""
    hop = int(np.prod(list(hp.gen.upsample_rates)))
    sr = float(hp.data.sampling_rate)
    f0u = f0[:, :, None].repeat_interleave(hop, dim=1)  # nn.Upsample nearest, [B,L,1]
    harm = torch.arange(1, 12, dtype=f0.dtype)
    fbuf = f0u * harm[None, None, :]
    rad = (fbuf / sr) % 1
    ri = rand_ini.clone()
    ri[:, 0] = 0
    rad[:, 0, :] = rad[:, 0, :] + ri
    wrapped = torch.cumsum(rad, 1) % 1
    over = (wrapped[:, 1:, :] - wrapped[:, :-1, :]) < 0
    shift = torch.zeros_like(rad)
    shift[:, 1:, :] = over * -1.0
    sines = torch.sin(torch.cumsum(rad + shift, dim=1) * 2 * np.pi) * 0.1
    uv = (f0u > 0).to(f0.dtype)
    namp = uv * 0.003 + (1 - uv) * 0.1 / 3
    sines = sines * uv + namp * noise
    merged = F.linear(sines, sd["dec.m_source.merge_w"]) + sd["dec.m_source.merge_b"]
    return torch.tanh(merged).transpose(1, 2)  # [B,1,L]


def source2wav(source: torch.Tensor) -> np.ndarray:
    """generator.py:167-173"""
    a = (32768.0 * source.squeeze()).clamp(min=-32768.0, max=32767.0)
    return a.short().cpu().numpy()


# --------------------------------------------------------------------------- whole path
def synthesizer_infer(sd: SD, hp, ppg, vec, pit, spk, ppg_l, source, eps, stages: Optional[dict] = None):
    """SynthesizerInfer.inference, vits/models.py:251-256."""
    with torch.no_grad():
        z_p, mask = prior_encoder(sd, ppg, ppg_l, vec, pit, eps, stages=stages)
        if stages is not None:
            stages["z_p"] = z_p
        z = flow_reverse(sd, z_p, mask, spk, stages=stages)
        if stages is not None:
            stages["z"] = z
        return generator(sd, hp, spk, z * mask, source, stages=stages)
