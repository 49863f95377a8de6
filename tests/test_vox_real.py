"""Real speech, ragged: five utterances of the reference's own sample data (4.4 .. 14.2 s, `tests/golden/vox_real_large2l.npz`, made
by tools/make_vox_golden.py from the UNMODIFIED reference) as one zero-padded batch with a padding mask, WavLM-Large widths, 2
layers; the fixture keeps every 12th frame of 16 seeded hidden channels.  CPU: the oracle against the reference's numbers.  GPU:
the kernels against the reference's numbers on the valid frames."""
import os

import numpy as np
import pytest
import torch

from oracle import wavlm_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden", "vox_real_large2l.npz")


def _batch(g):
    pcm, lengths = g["pcm"], [int(v) for v in g["lengths"]]
    B, L = pcm.shape
    wav = torch.zeros(B, L)
    pmask = torch.zeros(B, L, dtype=torch.bool)
    for b, n in enumerate(lengths):
        w = torch.from_numpy(pcm[b, :n].astype(np.float32)) / 32768.0
        wav[b, :n] = torch.nn.functional.layer_norm(w, (n,))
        pmask[b, n:] = True
    return wav, pmask


def test_oracle_on_real_speech_matches_reference():
    g = np.load(GOLD)
    cfg = O.large_config(encoder_layers=2)
    sd = O.deterministic_state_dict(cfg)
    wav, pmask = _batch(g)
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    with torch.no_grad():
        r = O.extract_features(sd, wav, cfg, padding_mask=pmask)
    rows, cols = torch.from_numpy(g["rows"]), torch.from_numpy(g["cols"])
    fpm = torch.from_numpy(g["frame_padding_mask"])
    assert torch.equal(r["padding_mask"], fpm)
    want = torch.from_numpy(g["x_final"].astype(np.float32))
    keep = ~fpm[:, rows]
    d = (r["x"][:, rows][..., cols] - want)[keep].abs()
    assert d.max().item() < 2e-2 and d.mean().item() < 2e-3, (d.max().item(), d.mean().item())   # fp16 storage of values up to ~20


@pytest.mark.gpu
def test_kernels_on_real_speech_match_reference(cuda_device):
    from unispeech_b200.wavlm import WavLM, WavLMConfig
    g = np.load(GOLD)
    cfg = O.large_config(encoder_layers=2)
    m = WavLM(WavLMConfig(vars(cfg)))
    m.load_state_dict(O.deterministic_state_dict(cfg))
    m = m.to(cuda_device).eval()
    wav, pmask = _batch(g)
    with torch.no_grad():
        (x, lr), fpm = m.extract_features(wav.to(cuda_device), padding_mask=pmask, ret_layer_results=True,
                                          output_layer=cfg.encoder_layers)
        xf, _ = m.extract_features(wav.to(cuda_device), padding_mask=pmask)
    torch.cuda.synchronize()
    rows, cols = torch.from_numpy(g["rows"]), torch.from_numpy(g["cols"])
    pad = torch.from_numpy(g["frame_padding_mask"])
    assert torch.equal(fpm.cpu(), pad)
    keep = ~pad[:, rows]
    for name, got, want in (("x_final", xf[:, rows.to(xf.device)].float().cpu()[..., cols], torch.from_numpy(g["x_final"].astype(np.float32))),
                            ("layer1", lr[1][0][rows.to(xf.device)].float().cpu()[..., cols].transpose(0, 1),
                             torch.from_numpy(g["layer1"].astype(np.float32)).transpose(0, 1))):
        d = (got - want)[keep].abs()
        scale, mscale = want[keep].abs().max().item(), want[keep].abs().mean().item()
        # same bounds as the full-depth tests (tests/test_fullscale_gpu.py): bf16 operands against the fp32 reference
        assert d.max().item() <= 0.03 * scale and d.mean().item() <= 0.015 * mscale, (name, d.max().item(), scale, d.mean().item(), mscale)
