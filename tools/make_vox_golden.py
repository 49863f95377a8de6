"""Real-speech ragged fixture: five utterances of the reference's own sample data
(/root/reference/downstreams/speaker_verification/vox1_data/*/*.wav, 16 kHz int16, 4.4 .. 14.2 s) through the UNMODIFIED reference
model (oracle/_ref) as ONE zero-padded batch with a sample-level padding mask -- WavLM-Large widths, 2 layers, deterministic weights.
The waveforms travel with the fixture; of the outputs (final hidden state and the first layer's output) every 12th frame of 16 seeded
channels is stored, in fp16, which keeps the file under 1 MB.

    python -m oracle.build_ref && python tools/make_vox_golden.py        (authoring container only)
"""
import glob
import os
import sys

import numpy as np
import torch
from scipy.io import wavfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import build_ref  # noqa: E402
from oracle import wavlm_oracle as O  # noqa: E402

STEP = 12
CHANNELS = 16
PICK = ["Lea_Thompson/mHTAr5dlAgc_0000004.wav", "David_Faustino/hn8GyCJIfLM_0000012.wav", "Zulay_Henao/WbB8m9-wlIQ_0000001.wav",
        "Zulay_Henao/gFfcgOVmiO0_0000002.wav", "Josh_Gad/RFyw7V3SOnQ_0000001.wav"]


def main():
    base = "/root/reference/downstreams/speaker_verification/vox1_data"
    wavs = []
    for rel in PICK:
        sr, w = wavfile.read(os.path.join(base, rel))
        assert sr == 16000 and w.dtype == np.int16 and w.ndim == 1
        wavs.append(w)
    lengths = [len(w) for w in wavs]
    L = max(lengths)
    pcm = np.zeros((len(wavs), L), dtype=np.int16)
    for i, w in enumerate(wavs):
        pcm[i, :len(w)] = w
    cfg = O.large_config(encoder_layers=2)
    sd = O.deterministic_state_dict(cfg)
    m = build_ref.build_model(cfg, sd)
    wav, pmask = vox_batch(pcm, lengths)
    with torch.no_grad():
        (x, lr), fpm = m.extract_features(wav.clone(), padding_mask=pmask, mask=False, ret_layer_results=True,
                                          output_layer=cfg.encoder_layers)
        xf, _ = m.extract_features(wav.clone(), padding_mask=pmask, mask=False)
    T = xf.shape[1]
    rows = np.arange(0, T, STEP)
    cols = np.sort(np.random.default_rng(0).choice(xf.shape[2], CHANNELS, replace=False))
    out = os.path.join(ROOT, "tests", "golden", "vox_real_large2l.npz")
    np.savez_compressed(out, pcm=pcm, lengths=np.asarray(lengths), rows=rows, cols=cols, frame_padding_mask=fpm.numpy(),
                        x_final=xf[:, rows][..., cols].numpy().astype(np.float16),
                        layer1=lr[1][0][rows][..., cols].numpy().astype(np.float16))
    print("T", T, "rows", len(rows), "valid frames", (~fpm).sum(1).tolist(), "bytes", os.path.getsize(out))


def vox_batch(pcm, lengths):
    """int16 PCM [B, L] + lengths -> (float waveform, padding mask): per-utterance normalisation as the reference's data path does for
    `normalize=True` models (utterance_mixing_dataset.py:571-573), zeros in the padding."""
    B, L = pcm.shape
    wav = torch.zeros(B, L)
    pmask = torch.zeros(B, L, dtype=torch.bool)
    for b, n in enumerate(lengths):
        w = torch.from_numpy(pcm[b, :n].astype(np.float32)) / 32768.0
        wav[b, :n] = torch.nn.functional.layer_norm(w, (n,))
        pmask[b, n:] = True
    return wav, pmask


if __name__ == "__main__":
    main()
