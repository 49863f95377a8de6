"""Long-utterance measurements: WavLM-Large end to end on minutes of audio, the long attention kernels alone, and the old
and new attention kernels alternately at the lengths where both run (the evidence for the T-based selection in
engine.attn_kernels).

    python tools/bench_long.py [--out FILE]

Times are CUDA-event times on the device; the device name and power limit are printed first and belong to every number."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import wavlm_oracle as O  # noqa: E402

SR = 16000
PEAK_BF16 = 2250e12   # dense BF16 FLOP/s of one B200 (data sheet, 1000 W)
LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return f"device: {torch.cuda.get_device_name()} | nvidia-smi: {q[torch.cuda.current_device()] if q else 'n/a'}"


def timed(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def model_section():
    from unispeech_b200.wavlm import WavLM, WavLMConfig
    torch.manual_seed(0)
    cfg = O.large_config()
    m = WavLM(WavLMConfig(vars(cfg))).cuda()
    say("== WavLM-Large (24 x 1024, 16 heads, random init, bf16 kernels), B = 1")
    m.eval()
    for sec in (60, 120, 300):
        wav = torch.randn(1, sec * SR, device="cuda")
        T = O.num_frames(sec * SR, cfg)

        def run():
            with torch.no_grad():
                m.extract_features(wav)
        run()
        torch.cuda.reset_peak_memory_stats()
        ms = timed(run, reps=5)
        say(f"eval extract_features {sec:4d} s (T={T:5d}): {ms:9.2f} ms  {sec / (ms / 1e3):8.1f} audio-s/s  "
            f"peak {torch.cuda.max_memory_allocated() / 1e9:6.2f} GB")
    m.train()
    sec = 120
    wav = torch.randn(1, sec * SR, device="cuda")
    T = O.num_frames(sec * SR, cfg)

    def step():
        x, _ = m.extract_features(wav)
        x.float().square().mean().backward()
    step()
    torch.cuda.reset_peak_memory_stats()
    ms = timed(step, reps=3)
    say(f"train fwd+bwd          {sec:4d} s (T={T:5d}): {ms:9.2f} ms  {sec / (ms / 1e3):8.1f} audio-s/s  "
        f"peak {torch.cuda.max_memory_allocated() / 1e9:6.2f} GB")
    del m
    torch.cuda.empty_cache()


class AttnCase:
    """Operands of one attention layer: B x T, H heads, the released bucketing (320 / 800) with a random embedding."""

    def __init__(self, B, T, H, bias=True, seed=0):
        from unispeech_b200.engine import bias_radius, relative_positions_bucket_lut
        g = torch.Generator(device="cuda").manual_seed(seed)
        D = H * 64
        self.B, self.T, self.H = B, T, H
        self.qkv = torch.randn(B, T, 3 * D, device="cuda", generator=g).bfloat16()
        self.gate = torch.rand(B, H, T, device="cuda", generator=g) * 2 if bias else None
        lut = relative_positions_bucket_lut(T, 320, 800)
        self.R = bias_radius(lut, 320)
        self.tab = torch.randn(320, H, device="cuda", generator=g)[lut.cuda().long()].t().contiguous() if bias else None
        self.out = torch.empty(B, T, D, device="cuda", dtype=torch.bfloat16)
        self.lse = torch.empty(B, H, T, device="cuda")
        self.dout = torch.randn(B, T, D, device="cuda", generator=g).bfloat16()
        self.delta = torch.empty(B, H, T, device="cuda")
        self.dqkv = torch.empty(B, T, 3 * D, device="cuda", dtype=torch.bfloat16)
        self.dgate = torch.empty(B, H, T, device="cuda") if bias else None
        self.dtab = torch.zeros(H, 2 * T - 1, device="cuda") if bias else None

    def fwd(self):
        from unispeech_b200 import ops
        ops.attn_fwd(self.qkv, self.gate, self.tab, None, self.out, self.lse, self.B, self.T, self.H, 0.125)

    def fwd_long(self):
        from unispeech_b200 import ops
        ops.attn_fwd_long(self.qkv, self.gate, self.tab, self.R, None, self.out, self.lse, self.B, self.T, self.H, 0.125)

    def bwd(self):
        from unispeech_b200 import ops
        ops.attn_bwd(self.qkv, self.out, self.dout, self.gate, self.tab, None, self.lse, self.delta, self.dqkv, self.dgate,
                     self.dtab, self.B, self.T, self.H, 0.125)

    def bwd_long(self):
        from unispeech_b200 import ops
        ops.attn_bwd_long(self.qkv, self.out, self.dout, self.gate, self.tab, self.R, None, self.lse, self.delta, self.dqkv,
                          self.dgate, self.dtab, self.B, self.T, self.H, 0.125)

    def flops(self, which):  # algorithmic: 2 GEMMs forward, 5 backward, 2*T*T*64 each per (b, h)
        return (4.0 if which == "fwd" else 10.0) * self.B * self.H * self.T * self.T * 64


def kernel_section():
    say("== long attention kernels alone, H = 16, B = 1, table 320 / 800 (R derived from the LUT), mean over launches")
    for T in (6000, 16384):
        c = AttnCase(1, T, 16)
        c.fwd_long()
        for name, fn, which in (("attn_fwd_long", c.fwd_long, "fwd"), ("attn_bwd_long", c.bwd_long, "bwd")):
            reps = 40 if T < 10000 else 10
            ms = timed(fn, reps=reps)
            rate = c.flops(which) / (ms / 1e3)
            say(f"{name:14s} T={T:5d} R={c.R}: {ms:8.3f} ms  {rate / 1e12:7.1f} TFLOP/s  = {100 * rate / PEAK_BF16:5.1f} % of "
                f"2,250 dense BF16")
    say("  (attention is bound by the exponentials and their issue slots, 128 x 128 exp2 per S tile against a 128x128x64"
        " MMA, not by the tensor core)")


def overlap_section():
    say("== overlap: old and new kernel alternately on the same operands (H = 16, B = 1, bias on), 5 rounds x 20 launches")
    for T, old, new, which in ((3000, "fwd", "fwd_long", "fwd"), (4000, "bwd", "bwd_long", "bwd")):
        c = AttnCase(1, T, 16)
        c.fwd_long()   # (lse for the backward; attn_fwd takes the bias only up to 3072 frames)
        fo, fn = getattr(c, old), getattr(c, new)
        to, tn = [], []
        for _ in range(5):
            to.append(timed(fo, reps=20))
            tn.append(timed(fn, reps=20))
        mo, mn = min(to), min(tn)
        say(f"T={T} attn_{old:8s} {mo:7.3f} ms (runs {', '.join(f'{t:.3f}' for t in to)})")
        say(f"T={T} attn_{new:8s} {mn:7.3f} ms (runs {', '.join(f'{t:.3f}' for t in tn)})  new / old = {mn / mo:.3f}")


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--skip-model", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long.py measures on the GPU; no CUDA device found")
    from unispeech_b200 import build
    build.build()
    say(device_line())
    if not args.skip_model:
        model_section()
    kernel_section()
    overlap_section()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
