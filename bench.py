"""Headline benchmark: WavLM forward+backward throughput in audio-seconds/second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model base|large] [--impl ours|reference] [--dump-outputs DIR]

Workload = the model BASELINE.json's metric names: WavLM-Large, batch 8 x 20 s synthetic 16 kHz waveform per GPU (configs[2]'s
per-GPU batch; it fits one B200), masking on, fwd + bwd of the whole encoder through the public API (`WavLM.extract_features` +
probe loss + `backward()`), bf16 kernels, dropout 0 as in BASELINE.md section 3.  At N=1 the line also carries, under `also`,
WavLM-Base 16 x 15 s (configs[1]) and the same Large workload with the reference's default dropouts (0.1 / 0.1).
N>1 (launched with torch.distributed.run): same per-GPU batch (weak scaling), plus the gradient average of the flat fp32
gradient buffer: NCCL all-reduce (AVG) in a few contiguous buckets issued WHILE the backward pass runs (parallel.OverlappedGradSync).
Timing: CUDA events around exactly K steps, barrier + synchronize on both sides, max over ranks.
Inputs are far larger than L2 (the first conv activation alone is 786 MB), so no explicit L2 flush is needed.

`--impl reference` times the reference's own CPU implementation: the UNMODIFIED `WavLM/{WavLM,modules}.py` vendored into
`oracle/_ref` by `oracle/build_ref.py` (kind "reference"; the oracle port only if that copy is absent), fwd+bwd on a bounded
sample of the same workload, on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SR = 16000


def model_config(name: str):
    from types import SimpleNamespace
    from unispeech_b200 import workloads
    cfg, B, secs = workloads.model_config(name)
    return SimpleNamespace(**cfg), B, secs


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _cpu_arm(cfg):
    """(kind, make_step): the reference's own CPU path when oracle/_ref holds the unmodified reference modules, else the oracle
    port.  make_step(B, secs) -> callable running one fwd+bwd (probe loss) and returning nothing."""
    from oracle import build_ref
    from oracle import wavlm_oracle as O
    sd = O.deterministic_state_dict(cfg)
    if build_ref.available():
        m = build_ref.build_model(cfg, sd, train=True)

        def make_step(B, secs):
            wav, _ = O.deterministic_waveform(B, secs * SR, seed=3)
            pm = torch.zeros(B, secs * SR, dtype=torch.bool)

            def step():
                m.zero_grad(set_to_none=True)
                x, fpm = m.extract_features(wav, padding_mask=pm, mask=True)  # the reference's own host-RNG span sampler
                O.probe_loss(x, fpm, seed=2).backward()
            return step
        return "reference", make_step
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}

    def make_step(B, secs):
        wav, _ = O.deterministic_waveform(B, secs * SR, seed=3)
        pm = torch.zeros(B, secs * SR, dtype=torch.bool)
        mi = O.hash_uniform("benchmask", (B, O.num_frames(secs * SR, cfg))) > 0.3

        def step():
            res = O.extract_features(sdr, wav, cfg, padding_mask=pm, mask_indices=mi)
            O.probe_loss(res["x"], res["padding_mask"], seed=2).backward()
            for v in sdr.values():
                v.grad = None
        return step
    return "port", make_step


def cpu_measure(cfg, B, secs, steps, warmup=1):
    """Bounded CPU sample: fwd+bwd on B x secs of audio.  Thread policy (fixed): the fastest of {16, 32, all} intra-op threads on a
    2 x 5 s probe (a 128-thread host oversubscribed with 128 threads is ~80x slower than with 16), then `warmup` untimed and
    `steps` timed steps; the MEDIAN step is reported.  Returns dict(value, seconds, threads, kind)."""
    kind, make_step = _cpu_arm(cfg)
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (16, 32) if c <= ncpu} | ({ncpu} if ncpu <= 64 else set())) or [ncpu]
    probe = make_step(2, 5)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            probe()
            ts.append(time.perf_counter() - t0)
        if min(ts) < best_t:
            best, best_t = c, min(ts)
    torch.set_num_threads(best)
    step = make_step(B, secs)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return {"value": B * secs / med, "seconds": med, "threads": best, "kind": kind, "steps": steps}


def run_reference(args):
    cfg, B, secs = model_config(args.model)
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, csecs = {"tiny": B, "base": 4, "large": 2}[args.model], secs
    steps = max(3, min(args.steps, 5))
    r = cpu_measure(cfg, cb, csecs, steps, warmup=1)
    what = ("the UNMODIFIED reference modules WavLM/{WavLM,modules}.py (oracle/_ref; out-of-place encoder patch for autograd)"
            if r["kind"] == "reference" else "oracle port (CPU restatement of the reference PyTorch path)")
    line = {
        "impl": "reference", "metric": "audio-sec/sec fwd+bwd", "value": r["value"], "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"WavLM-{args.model} fwd+bwd on the host CPU, {what}, bounded sample {cb} x {csecs} s per step"},
        "cpu_baseline": {"value": r["value"], "unit": "audio-s/s", "cores": r["threads"], "kind": r["kind"],
                         "sample": f"{cb} x {csecs} s per step, 1 warm-up + {steps} timed steps, median; fastest of 16 / 32 / all "
                                   f"intra-op threads on a 2 x 5 s probe (host has {os.cpu_count()} logical CPUs)"},
        "e2e": {"value": r["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


class Workload:
    """One model + one synthetic batch per rank, stepped through the public API (extract_features + probe loss + backward
    [+ the gradient allreduce for N > 1])."""

    def __init__(self, model_name, dev, rank, world, dropout=0.0, ragged=False, pretrain=False, sat=False):
        from unispeech_b200 import workloads
        from unispeech_b200.wavlm import WavLM, WavLMConfig
        self.name, self.dev, self.world, self.dropout, self.pretrain = model_name, dev, world, dropout, pretrain
        self.opt, self.sync, self.sat = None, None, sat
        pretrain = self.pretrain = pretrain or sat
        cfg, B, secs = model_config(model_name)
        if sat:
            # BASELINE.json configs[3]: UniSpeech-SAT Large as shipped (SURVEY.md section 8c): WavLM-Large encoder geometry WITHOUT the
            # relative-position bias / gate, masked-prediction head (504 labels, final_dim 768, mask_prob 0.8) + utterance-contrastive
            # loss on layer 12 with 100 cross-sample instances and Gumbel-quantised targets (320 x 2 codes), utterance mixing on the
            # host in front of every batch
            cfg.relative_position_embedding, cfg.gru_rel_pos, cfg.mask_prob = False, False, 0.8
        if dropout > 0:  # the reference's WavLMConfig defaults: dropout = attention_dropout = 0.1 (WavLM/WavLM.py:180-181)
            cfg.dropout, cfg.attention_dropout = dropout, dropout
        self.cfg, self.B, self.secs, self.ragged = cfg, B, secs, ragged
        # BASELINE.json configs[4]: utterances of 4 .. 30 s (seeded per rank), zero-padded to the longest of the batch, with the
        # sample-level padding mask the reference collater builds; the fixed-length workloads use `secs` for every utterance
        def lengths_of(r):
            if not ragged:
                return [secs * SR] * B
            g = torch.Generator().manual_seed(4242 + r)
            return [int(v) for v in torch.randint(4 * SR, 30 * SR + 1, (B,), generator=g)]
        self.lengths = lengths_of(rank)
        self.all_lengths = [lengths_of(r) for r in range(world)]
        self.L = max(self.lengths)
        self.T = workloads.num_frames(self.L, vars(cfg))
        if pretrain:
            # full optimisation step of the masked-prediction pre-training (SURVEY.md section 8f rows 1-2): 504-class k-means labels
            # at 50 Hz, final_dim 768 (the released Large recipe), WavLMCriterion with features_pen x 10, Adam(0.9, 0.98), clip 1.0
            from unispeech_b200.pretrain import WavLMForPretraining, WavLMPretrainConfig
            torch.manual_seed(20 + 0)  # random init of the architecture (the reference's initialisers), same on every rank
            fd = 768 if model_name == "large" else 256
            if sat:
                from unispeech_b200.unispeech_sat import UniSpeechSATConfig, UniSpeechSATForPretraining
                model = UniSpeechSATForPretraining(UniSpeechSATConfig(dict(
                    vars(cfg), final_dim=fd, utterance_contrastive_layer=cfg.encoder_layers // 2, num_instances=0,
                    cross_sample_instances=100, quantize_targets=True, latent_vars=320, latent_groups=2, latent_dim=fd,
                    layer_norm_for_extract=True)), [504])
            else:
                model = WavLMForPretraining(WavLMPretrainConfig(dict(vars(cfg), final_dim=fd)), [504])
            self.labels = [torch.randint(0, 504, (B, self.T), generator=torch.Generator().manual_seed(99 + rank))]
            self.final_dim = model.final_dim
        else:
            torch.manual_seed(20 + 0)  # random init of the architecture (the reference's initialisers), same on every rank
            model = WavLM(WavLMConfig(vars(cfg)))
        self.model = model.to(dev).train()
        gen = torch.Generator().manual_seed(1337 + rank)
        wav = torch.randn(B, self.L, generator=gen)
        self.pad_host = torch.zeros(B, self.L, dtype=torch.bool)  # the reference always passes a mask in training (all-False when nothing is padded, S14)
        for b, n in enumerate(self.lengths):
            if cfg.normalize:  # per-utterance normalisation of the data path (utterance_mixing_dataset.py:571-573), before padding
                wav[b, :n] = torch.nn.functional.layer_norm(wav[b, :n], (n,))
            wav[b, n:] = 0.0
            self.pad_host[b, n:] = True
        self.wav_host = wav.pin_memory()
        self.wav_mixed = torch.empty_like(wav).pin_memory() if sat else None
        self.wav_dev = self.wav_host.to(dev)
        self.R = torch.randn(B, self.T, cfg.encoder_embed_dim, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
        if ragged:  # the probe loss reads VALID frames only, like every criterion of the reference (padded frames carry no loss)
            tl = torch.tensor([workloads.num_frames(n, vars(cfg)) for n in self.lengths], device=dev)
            self.R.mul_((torch.arange(self.T, device=dev)[None, :] < tl[:, None]).unsqueeze(-1))
        self.loss_host = torch.zeros(1).pin_memory()
        self.fwd_flops = workloads.forward_flops(self.L, vars(cfg))          # padded shape (what the kernels execute)
        self.valid_fwd_flops = sum(workloads.forward_flops(n, vars(cfg)) for n in self.lengths) / B   # per utterance at its own length

    def _mark(self, name):
        """(--phases) a CUDA event at a phase boundary of the step, on the current stream."""
        if getattr(self, "phases", None) is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.phases.append((name, ev))

    def _sync_for(self, collective: bool):
        """Bucketed gradient averaging overlapped with the backward pass (N > 1); created once the engine owns the layout."""
        if self.world == 1:
            return None
        if self.sync is None:
            from unispeech_b200.parallel import OverlappedGradSync
            self.sync = OverlappedGradSync(self.model, layers_per_bucket=6)
        self.sync.active = bool(collective)
        self.sync.begin()
        return self.sync

    def step(self, e2e: bool, collective: bool = True):
        """One step; the NVTX range names are the reference trainer's (src/fairseq/trainer.py:781-827, fairseq_cli/train.py:288-290)."""
        nvtx = torch.cuda.nvtx
        model = self.model
        if model._engine is not None and model._engine.flat is not None:
            if not self.pretrain:  # (the optimizer step of the pre-training workload zeroes the gradients itself)
                model.zero_grad_buffer()
            model._engine.prepared_version = None  # parameters change every optimisation step: re-derive the bf16 operands
        if self.sat and e2e:
            # the data path of the reference mixes utterances on the host for every batch (utterance_mixing_dataset.py:373-438);
            # in the end-to-end measurement it is inside the timed region, like the host-to-device copy
            from unispeech_b200.mixing import mix_utterances
            self.wav_mixed.copy_(self.wav_host)
            mix_utterances(self.wav_mixed, mixing_prob=0.5, mixing_num=1, mixing_max_len=-1, normalize=self.cfg.normalize)
            wav = self.wav_mixed.to(self.dev, non_blocking=True)
        else:
            wav = self.wav_host.to(self.dev, non_blocking=True) if e2e else self.wav_dev
        if self.pretrain:
            return self.pretrain_step(wav, e2e, collective)
        self._mark("start")
        nvtx.range_push("forward")
        x, fpm = model.extract_features(wav, padding_mask=self.pad_host, mask=True)
        loss = (x.float() * self.R).sum()
        self.outputs = {"hidden": x, "padding_mask": fpm, "loss": loss}
        nvtx.range_pop()
        self._mark("forward")
        sync = self._sync_for(collective)
        nvtx.range_push("backward")
        loss.backward()
        nvtx.range_pop()
        self._mark("backward")
        if sync is not None:
            nvtx.range_push("reduce-grads")
            sync.finish()  # buckets were issued during backward; this sends the last one and joins the NCCL stream
            nvtx.range_pop()
        self._mark("reduce-grads")
        if e2e:
            self.loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        return loss

    def pretrain_step(self, wav, e2e: bool, collective: bool):
        """forward -> masked-prediction criterion -> backward (+ overlapped gradient average) -> scale / clip / Adam."""
        from unispeech_b200.optim import FusedAdam
        nvtx = torch.cuda.nvtx
        model = self.model
        self._mark("start")
        nvtx.range_push("forward")
        out = model(wav, target_list=self.labels, padding_mask=self.pad_host, mask=True)
        lw = [10.0, 10.0, 0.0, 0.1] if self.sat else [10.0]   # features_pen, loss_spk_m, loss_spk_u, diversity (prob_perplexity)
        loss, sample_size, _ = model.criterion(out, pred_masked_weight=1.0, pred_nomask_weight=0.0, loss_weights=lw)
        self.outputs = {"hidden": out["x"], "padding_mask": out["padding_mask"], "loss": loss}
        nvtx.range_pop()
        self._mark("forward")
        sync = self._sync_for(collective)
        nvtx.range_push("backward")
        loss.backward()
        nvtx.range_pop()
        self._mark("backward")
        if sync is not None:
            nvtx.range_push("reduce-grads")
            sync.finish()
            nvtx.range_pop()
        self._mark("reduce-grads")
        if self.opt is None:
            self.opt = FusedAdam(model, lr=1e-5, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.01)
        self.opt.multiply_grads(self.world / max(sample_size, 1))   # trainer.py:796-801 (sample_size is per rank here: equal shards)
        nvtx.range_push("clip-grads")
        self.opt.clip_grad_norm(1.0)
        nvtx.range_pop()
        self._mark("clip-grads")
        nvtx.range_push("optimizer")
        self.opt.step(zero_grad=True)
        nvtx.range_pop()
        self._mark("optimizer")
        if e2e:
            self.loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        return loss

    def timed(self, n_steps: int, e2e: bool) -> float:
        """Milliseconds for exactly n_steps: barrier + synchronize on both sides, CUDA events, max over ranks."""
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(n_steps):
            self.step(e2e)
        ev1.record()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        ms = ev0.elapsed_time(ev1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def audio_seconds(self, n_steps: int) -> float:
        """VALID (unpadded) audio seconds over all ranks: padding is overhead, not credit (SURVEY.md section 8d)."""
        return sum(sum(l) for l in self.all_lengths) / SR * n_steps

    def padded_audio_seconds(self, n_steps: int) -> float:
        return sum(len(l) * max(l) for l in self.all_lengths) / SR * n_steps

    def describe(self) -> str:
        drop = f"dropout {self.dropout} / attention_dropout {self.dropout}" if self.dropout > 0 else "dropout 0"
        if self.sat:
            return (f"UniSpeech-SAT {self.name} full pre-training step (BASELINE configs[3]): fwd (no rel-pos bias, as shipped) + masked-"
                    f"prediction head (504 classes, final_dim {self.final_dim}) + utterance-contrastive loss on layer "
                    f"{self.cfg.encoder_layers // 2} (100 cross-sample instances, Gumbel-quantised targets 320 x 2, training mode) + "
                    f"WavLMCriterion (features_pen x 10, loss_spk_m x 10, diversity x 0.1) + bwd + gradient scale / clip 1.0 / Adam, "
                    f"batch {self.B} x {self.secs} s per GPU, mask_prob {self.cfg.mask_prob}, {drop}; utterance mixing (p 0.5) on "
                    f"the host inside the end-to-end timed region")
        if self.pretrain:
            return (f"WavLM-{self.name} full optimisation step: fwd + masked-prediction head (504 classes, final_dim "
                    f"{self.final_dim}) + WavLMCriterion (features_pen x 10) + bwd + gradient scale / clip 1.0 / Adam, batch "
                    f"{self.B} x {self.secs} s per GPU, mask_prob {self.cfg.mask_prob}, {drop}")
        if self.ragged:
            secs = ", ".join(f"{n / SR:.1f}" for n in self.lengths)
            return (f"WavLM-{self.name} fwd+bwd, ragged batch of {self.B} utterances per GPU drawn from 4..30 s (rank 0: {secs} s), "
                    f"zero-padded to {self.L / SR:.1f} s with a sample-level padding mask, 16 kHz synthetic, mask_prob "
                    f"{self.cfg.mask_prob}, {drop}; value counts VALID audio only")
        return (f"WavLM-{self.name} fwd+bwd, batch {self.B} x {self.secs} s per GPU, 16 kHz synthetic, mask_prob "
                f"{self.cfg.mask_prob}, {drop}, all-False padding mask")

    def free(self):
        self.model = self.R = self.wav_dev = self.opt = self.sync = self.outputs = None
        torch.cuda.empty_cache()


def parity_line(dev, model_name: str):
    """The other half of BASELINE.json's metric ("...; max-abs hidden diff").  Two numbers, both measured in this run:
    (1) FULL DEPTH at the benchmark's sequence length: all layers of the model, one utterance of the workload's duration, same
        hash-generated weights and waveform on both sides, against the reference's own CPU forward (the unmodified modules in
        oracle/_ref when present, else the oracle port) -- final hidden states and the worst layer;
    (2) the committed fixture of the unmodified reference (tests/golden, 2 layers, 0.5 s) as a box-independent anchor.
    The per-layer tables and the gradient parity at real widths are the GPU test suite (tests/test_fullscale_gpu.py)."""
    import numpy as np
    from oracle import build_ref
    from oracle import wavlm_oracle as O
    from unispeech_b200.wavlm import WavLM, WavLMConfig
    name = {"large": "large2l_halfsec", "base": "base2l_halfsec"}.get(model_name)
    if name is None:
        return None
    mk = O.large_config if model_name == "large" else O.base_config
    out = {}
    # ---- (1) full depth
    cfg = mk()
    secs = 20 if model_name == "large" else 15
    sd = O.deterministic_state_dict(cfg)
    wav, _ = O.deterministic_waveform(1, secs * SR, seed=3)
    n = cfg.encoder_layers
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    with torch.no_grad():
        if build_ref.available():
            mref = build_ref.build_model(cfg, sd)
            (_, lr), _ = mref.extract_features(wav, ret_layer_results=True, output_layer=n)
            want_layers = [t[0] for t in lr]
            want_x = mref.extract_features(wav)[0]
            against = "unmodified reference modules (oracle/_ref), fp32 CPU"
            del mref
        else:
            r = O.extract_features(sd, wav, cfg, output_layer=n)
            want_layers = r["layer_results"]
            want_x = O.extract_features(sd, wav, cfg)["x"]
            against = "oracle port, fp32 CPU"
    m = WavLM(WavLMConfig(vars(cfg)))
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    with torch.no_grad():
        (_, got_lr), _ = m.extract_features(wav.to(dev), ret_layer_results=True, output_layer=n)
        got_x = m.extract_features(wav.to(dev))[0]
    worst = max(range(n + 1), key=lambda i: ((got_lr[i][0].float().cpu() - want_layers[i]).abs().max() / want_layers[i].abs().max()).item())
    dw = (got_lr[worst][0].float().cpu() - want_layers[worst]).abs()
    d = (got_x.float().cpu() - want_x).abs()
    out["full_depth"] = {
        "model": f"WavLM-{model_name}, {n} layers, 1 x {secs} s (T = {want_x.shape[1]})", "against": against,
        "max_abs_hidden_diff": d.max().item(), "mean_abs_hidden_diff": d.mean().item(),
        "hidden_abs_max": want_x.abs().max().item(), "hidden_abs_mean": want_x.abs().mean().item(),
        "worst_layer": worst, "worst_layer_max_abs_diff": dw.max().item(), "worst_layer_abs_max": want_layers[worst].abs().max().item(),
        "tolerance": "max-abs <= 3 % of the layer's max|h|, mean-abs <= 1.5 % of its mean|h| (tests/test_fullscale_gpu.py)"}
    del m, sd
    torch.cuda.empty_cache()
    # ---- (2) committed fixture
    g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    cfg = mk(encoder_layers=2)
    m = WavLM(WavLMConfig(vars(cfg)))
    m.load_state_dict(O.deterministic_state_dict(cfg))
    m = m.to(dev).eval()
    wav, _ = O.deterministic_waveform(1, 8000, seed=1)
    with torch.no_grad():
        x, _ = m.extract_features(wav.to(dev))
    want = torch.from_numpy(g["x_final"]).float()
    d = (x.float().cpu() - want).abs()
    out.update({"max_abs_hidden_diff": d.max().item(), "mean_abs_hidden_diff": d.mean().item(), "hidden_abs_max": want.abs().max().item(),
                "tolerance_max_abs": 0.12, "against": f"tests/golden/{name}.npz (unmodified reference WavLM forward, fp32 CPU; WavLM-{model_name} "
                                                      "widths, 2 layers, 1 x 0.5 s, same weights and waveform)"})
    return out


def quick_line(w: Workload, steps: int, warmup: int, e2e: bool = True):
    """Secondary measurement (reported under `also`): same timing rules, fewer outputs."""
    for _ in range(warmup):
        w.step(False)
    ms = w.timed(steps, False)
    out = {"workload": w.describe(), "value": w.audio_seconds(steps) / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms / steps,
           "model_tflops": 3 * w.valid_fwd_flops * w.world * w.B * steps / (ms * 1e-3) / 1e12}
    if w.ragged:
        out["padded_equivalent_value"] = w.padded_audio_seconds(steps) / (ms * 1e-3)
        out["padded_model_tflops"] = 3 * w.fwd_flops * w.world * w.B * steps / (ms * 1e-3) / 1e12
    if e2e:
        for _ in range(2):
            w.step(True)
        ms_e = w.timed(steps, True)
        out["e2e"] = {"value": w.audio_seconds(steps) / (ms_e * 1e-3), "unit": "audio-s/s", "ms_per_step": ms_e / steps}
    return out


DUMP_BYTES = 60 * 10**6   # --dump-outputs: float32 payload in all (the .npy headers keep it well inside 64 MB)


def dump_outputs(w: Workload, out_dir: str):
    """--dump-outputs: what the last step handed its caller, as float32 `<name>.npy` files, so that two builds can be compared
    output for output: the encoder output (`hidden`), the frame padding mask, the loss, and the gradients of all parameters
    (`grads`; for the optimisation-step workloads, which consume their gradients, the updated parameters, `params`) concatenated
    in `parameters()` order, which does not depend on how the engine lays out its buffers.  Smallest first, each array gets an
    equal share of what is left of DUMP_BYTES; an array larger than its share is replaced by a fixed sample of its flattened
    elements (positions drawn from a generator seeded with 0, sorted)."""
    import numpy as np
    arrays = {k: v for k, v in w.outputs.items() if v is not None}
    params = [p if w.pretrain else p.grad for p in w.model.parameters()]
    arrays["params" if w.pretrain else "grads"] = torch.cat([t.detach().reshape(-1).float() for t in params if t is not None])
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES // 4
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        n = min(t.numel(), left // (len(items) - i))
        if n < t.numel():
            pos = torch.randint(t.numel(), (n,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[pos.to(t.device)]
        left -= n
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def graph_probe(args):
    """The fixed-length fwd+bwd workload captured as ONE CUDA graph (unispeech_b200.graphed.GraphedForwardBackward): device time per
    replayed step, the same with the batch coming from pinned host memory, and what the HOST spends per step (span-mask sampling +
    two small copies + one graph launch).  Runs in its own process: a failed capture must not take the bench line with it."""
    from unispeech_b200 import _lib
    from unispeech_b200.graphed import GraphedForwardBackward
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.check_device()
    w = Workload(args.model, dev, 0, 1, dropout=0.0)
    g = GraphedForwardBackward(w.model, lambda x: (x.float() * w.R).sum(), w.B, w.L, dev)
    g.wav.copy_(w.wav_dev)
    g.capture(warmup=3)
    loss_host = torch.zeros(1).pin_memory()

    def run(n, e2e):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            loss = g.step(w.wav_host if e2e else None)
            if e2e:
                loss_host.copy_(loss.reshape(1), non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    run(3, False)
    ms = run(args.steps, False)
    run(2, True)
    ms_e = run(args.steps, True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(4):
        g.step(None)
    host_ms = (time.perf_counter() - t0) * 1e3 / 4
    torch.cuda.synchronize()
    audio = w.audio_seconds(args.steps)
    print(json.dumps({"workload": w.describe() + "; forward + loss + backward replayed as one CUDA graph, span mask re-sampled on the "
                      "host every step", "value": audio / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms / args.steps,
                      "e2e": {"value": audio / (ms_e * 1e-3), "unit": "audio-s/s", "ms_per_step": ms_e / args.steps},
                      "host_ms_per_step": host_ms, "capture_host_ms": g.capture_host_ms,   # one-off: host time of the stream capture of one step (incl. graph-node creation)
                      "loss_finite": bool(torch.isfinite(g.loss).item())}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--model", default="large", choices=["base", "large", "tiny"],
                    help="large = the model BASELINE.json's metric names (configs[2] per-GPU batch 8 x 20 s); base = configs[1]")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dropout", type=float, default=0.0, help="dropout = attention_dropout of the headline run (BASELINE.md "
                    "section 3 times both arms with dropout 0; the reference's config default 0.1 is reported under `also`)")
    ap.add_argument("--ragged", action="store_true", help="BASELINE.json configs[4]: variable-length batch 4..30 s with padding mask")
    ap.add_argument("--pretrain", action="store_true", help="time the full optimisation step (loss head + criterion + optimizer)")
    ap.add_argument("--sat", action="store_true", help="BASELINE.json configs[3]: UniSpeech-SAT Large pre-training step (masked "
                    "prediction + utterance-contrastive loss + Gumbel quantizer + host utterance mixing)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary measurements (WavLM-Base, reference dropouts)")
    ap.add_argument("--ncu-step", action="store_true", help="profile exactly one step (cudaProfilerStart/Stop) and exit")
    ap.add_argument("--phases", action="store_true", help="add `phases_ms` (device time between the NVTX phase boundaries of a step, "
                    "rank 0, mean of 3 extra steps) to the line")
    ap.add_argument("--graph-probe", action="store_true", help="(internal) measure the whole step as one CUDA graph "
                    "(unispeech_b200/graphed.py) and print a small JSON object; the default run calls this in a child process")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (encoder "
                    "output, padding mask, loss, a fixed sample of the gradients) as DIR/<name>.npy, float32, under 64 MB")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.graph_probe:
        return graph_probe(args)

    import torch.distributed as dist
    from unispeech_b200 import _lib, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nccl_ctas = None
    if world > 1:
        from unispeech_b200.parallel import configure_overlap
        _lib.check_device()
        nccl_ctas = configure_overlap(int(os.environ.get("B200S_NCCL_CTAS", "0")))   # optional: NCCL_MAX_CTAS + SMs the persistent GEMMs leave free
        # the host side of a step (span-mask sampling, instance draws) is torch / numpy CPU work: torchrun pins every rank to ONE
        # OpenMP thread unless told otherwise
        if os.environ.get("OMP_NUM_THREADS", "1") == "1":
            torch.set_num_threads(max(1, min(8, (os.cpu_count() or 8) // max(1, world))))
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    # the span masks are drawn from numpy's global generator (the reference's sampler): seeded, the same arguments give the
    # same inputs on every run
    import numpy as np
    np.random.seed(rank)
    w = Workload(args.model, dev, rank, world, dropout=args.dropout, ragged=args.ragged, pretrain=args.pretrain, sat=args.sat)
    cfg, B, secs, T = w.cfg, w.B, w.secs, w.T

    for _ in range(args.warmup):
        w.step(False)
    torch.cuda.synchronize()
    if args.ncu_step:
        # exactly one warmed-up step between cudaProfilerStart/Stop: run under `ncu --profile-from-start off ...`
        torch.cuda.profiler.start()
        w.step(False)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lc0 = _lib.load().b200s_launch_count
    lc0.restype = __import__("ctypes").c_longlong
    n0 = lc0()
    ms = w.timed(args.steps, False)
    launches = lc0() - n0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(w, args.dump_outputs)
    for _ in range(2):
        w.step(True)
    ms_e2e = w.timed(args.steps, True)

    # host cost of enqueueing one step (launch queue empty at the start, two steps timed without synchronising): if this
    # approaches ms_per_step the run is launch-bound, not GPU-bound
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
        w.step(False)
    host_ms = (time.perf_counter() - t0) * 1e3 / 2
    torch.cuda.synchronize()

    phases_ms = None
    if args.phases:
        w.phases = []
        for _ in range(3):
            w.step(False)
        torch.cuda.synchronize()
        acc = {}
        for (n0_, e0_), (n1_, e1_) in zip(w.phases[:-1], w.phases[1:]):
            if n1_ != "start":
                acc.setdefault(n1_, []).append(e0_.elapsed_time(e1_))
        phases_ms = {k: round(sum(v) / len(v), 3) for k, v in acc.items()}
        w.phases = None

    audio_s = w.audio_seconds(args.steps)
    value = audio_s / (ms * 1e-3)
    e2e_value = audio_s / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel family (tcgen05 GEMM): per-op CUDA-event timing in one extra profiled step
    roofline, breakdown = None, None
    if rank == 0 and not args.no_profile:
        prof = ops.Profiler()
        ops.set_profiler(prof)
        w.step(False, collective=False)  # rank 0 only: no collective in this extra, per-op-timed step
        torch.cuda.synchronize()
        ops.set_profiler(None)
        breakdown = prof.summary()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        is_gemm = lambda k: k.startswith("gemm") or k.startswith("posconv_gemm") or k.startswith("posconv_wgrad")
        gemm_ms = sum(v["ms"] for k, v in breakdown.items() if is_gemm(k))
        gemm_flops = sum(v["flops"] for k, v in breakdown.items() if is_gemm(k))
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        n_gemm = sum(v["calls"] for k, v in breakdown.items() if is_gemm(k))
        traffic, traffic_src = None, None
        try:  # DRAM bytes of the same launches from the committed ncu capture of one step (profiles/, same workload)
            tj = json.load(open(os.path.join(ROOT, "profiles", f"gemm_traffic_{args.model}.json")))
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
        except Exception:
            pass
        roofline = {"bound": "tensor", "kernel": "gemm_bf16_pair_kernel / gemm_bf16_kernel (all tcgen05 GEMM launches of one step, "
                                                 "per-launch averages)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1400",
                    "flop_per_launch": gemm_flops / max(n_gemm, 1), "launches_per_step": n_gemm,
                    "us_per_launch": gemm_ms * 1e3 / max(n_gemm, 1), "traffic": traffic, "traffic_source": traffic_src,
                    "gemm_ms_per_step": gemm_ms, "gemm_share_of_step": gemm_ms / (ms / args.steps)}
        # the other kernel families of the same profiled step, each against its own bound (algorithmic work / CUDA-event time)
        fam = {}
        att = {k: v for k, v in breakdown.items() if k.startswith("attn_")}
        for k, v in att.items():
            if v["ms"] > 0 and v["flops"] > 0:
                tf = v["flops"] / (v["ms"] * 1e-3) / 1e12
                fam[k] = {"bound": "tensor (+ SFU: one exp2 per score)", "achieved": tf, "unit": "TFLOP/s (algorithmic)",
                          "frac": tf / peak, "ms_per_step": v["ms"], "launches": v["calls"]}
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        for k in ("layer_norm_fwd", "layer_norm_gate_fwd", "layer_norm_bwd", "colsum"):
            v = breakdown.get(k)
            if v and v["ms"] > 0 and v["bytes"] > 0:
                gbs = v["bytes"] / (v["ms"] * 1e-3) / 1e9
                fam[k] = {"bound": "hbm", "achieved": gbs, "unit": "GB/s (algorithmic)", "frac": gbs / hbm_peak,
                          "ms_per_step": v["ms"], "launches": v["calls"]}
        roofline["other_families"] = fam

    parity = None
    if rank == 0 and not args.no_profile:
        try:
            parity = parity_line(dev, args.model)
        except Exception as exc:  # never at the expense of the measured line
            parity = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- secondary measurements (N = 1 only): the reference's default dropouts on the same workload, and WavLM-Base (configs[1])
    also = None
    if world == 1 and not args.no_also and args.model != "tiny":
        also = {}
        w.free()
        try:
            if args.dropout == 0.0:
                wd = Workload(args.model, dev, rank, world, dropout=0.1)
                also["reference_default_dropouts"] = quick_line(wd, args.steps, 3, e2e=False)
                wd.free()
            if not args.ragged and args.model == "large":
                wr = Workload("large", dev, rank, world, dropout=0.0, ragged=True)
                also["wavlm_large_ragged_4_30s"] = quick_line(wr, args.steps, 3, e2e=False)
                wr.free()
            if not args.ragged:
                wp = Workload(args.model, dev, rank, world, dropout=0.0, pretrain=True)
                also[f"wavlm_{args.model}_pretrain_step"] = quick_line(wp, args.steps, 3, e2e=True)
                wp.free()
            if not args.ragged and not args.sat and args.model == "large":
                ws = Workload("large", dev, rank, world, dropout=0.0, sat=True)
                also["unispeech_sat_large_pretrain_step"] = quick_line(ws, args.steps, 3, e2e=True)
                ws.free()
            other = "base" if args.model == "large" else "large"
            wo = Workload(other, dev, rank, world, dropout=0.0)
            also[f"wavlm_{other}"] = quick_line(wo, args.steps, 3, e2e=True)
            wo.free()
        except Exception as exc:  # a secondary line must never cost the headline
            also["error"] = f"{type(exc).__name__}: {exc}"

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        cb = {"tiny": B, "base": 4, "large": 2}[args.model]
        r = cpu_measure(cfg, cb, secs, steps=1, warmup=0)
        what = "unmodified reference modules (oracle/_ref)" if r["kind"] == "reference" else "oracle port"
        cpu_baseline = {"value": r["value"], "unit": "audio-s/s", "cores": r["threads"], "kind": r["kind"],
                        "sample": f"{what} fwd+bwd fp32, {cb} x {secs} s, 1 step ({r['seconds']:.1f} s); fastest of 16 / 32 / all "
                                  f"intra-op threads on a 2 x 5 s probe (host has {os.cpu_count()} logical CPUs); "
                                  "`--impl reference` times 3+ steps"}

    # ---- the same step replayed as one CUDA graph (N = 1, fixed-length fwd+bwd workload): host cost per step with the launches
    # taken off the host; measured in a child process
    graph = None
    if world == 1 and not (args.no_also or args.ragged or args.pretrain or args.sat) and args.dropout == 0.0 and args.model != "tiny":
        import subprocess
        try:
            if w is not None:
                w.free()
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--graph-probe", "--model", args.model, "--steps",
                                str(args.steps)], capture_output=True, text=True, timeout=420)
            last = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
            graph = json.loads(last[-1]) if (r.returncode == 0 and last) else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as exc:  # never at the expense of the measured line
            graph = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        fwd_flops = w.valid_fwd_flops
        line = {
            "metric": "audio-sec/sec fwd+bwd", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": w.describe() + (f"; gradient exchange: bucketed NCCL all-reduce (AVG, fp32) overlapped with backward, "
                                                   + (f"NCCL_MAX_CTAS={nccl_ctas}, the persistent GEMMs leave that many SMs free" if nccl_ctas else "NCCL defaults")
                                                   if world > 1 else ""),
                       "global_batch": world * B,
                       "frames": T, "parallelism": f"dp{world}", "l2": "inputs larger than L2 (no flush needed)", 
                       "algorithmic_gflop_per_audio_s": 3 * fwd_flops * B / (sum(w.lengths) / SR) / 1e9},
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": w.wav_host.numel() * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_ms,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "model_tflops": 3 * fwd_flops * world * B * args.steps / (ms * 1e-3) / 1e12,
        }
        if parity is not None:
            line["parity"] = parity
        if phases_ms is not None:
            line["phases_ms"] = phases_ms
        if args.ragged:
            line["padded_equivalent_value"] = w.padded_audio_seconds(args.steps) / (ms * 1e-3)
        if also is not None:
            line["also"] = also
        if graph is not None:
            line["cuda_graph_step"] = graph
        if breakdown is not None:
            line["breakdown_ms"] = {k: round(v["ms"], 3) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"])}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()  # the other ranks wait here while rank 0 finishes its profiled step and the CPU baseline
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
