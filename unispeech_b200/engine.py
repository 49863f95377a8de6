"""Host-side orchestration of the WavLM hot path over the C-ABI kernels (forward and backward).

Everything numerical runs in the hand-written sm_100a kernels (`ops.*`); this file only owns buffers, parameter
preparation, the order of launches and the autograd glue.  PyTorch is used for device memory and streams.

Layouts
  * activations: bf16, channels-last / batch-major `[B, T, C]` (the reference's `T x B x C` tensors are views of these);
  * conv stack gradients: `[B, Tg, C]` with `lead` zero rows in front (so the input-gradient GEMM can read row u-1);
  * pos_conv input / its output gradient: `[B, T+128, D]` with 64 zero rows on each side (taps become a TMA dimension);
  * parameters: fp32 masters in the reference state_dict layout; bf16 GEMM operands are re-derived by `prepare()`;
  * gradients: one flat fp32 buffer, `param.grad` are views into it (q/k/v projections adjacent so the fused [3D,D]
    weight gradient is a single GEMM); the data-parallel allreduce runs on the flat buffer.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

from . import _lib as L
from . import dropout as DR
from . import ops

BF = torch.bfloat16


def _even(n: int) -> int:
    return n + (n & 1)


def _grad_rows(B: int, Tg: int, C: int, lead: int, valid: int, device) -> torch.Tensor:
    """Gradient buffer [B, Tg, C] (bf16) in `lead` layout: rows [lead, lead + valid) are fully written by the producing
    kernel, so only the zero rows the input-gradient GEMM reads around them are cleared (not the whole buffer)."""
    g = torch.empty(B, Tg, C, dtype=BF, device=device)
    if lead > 0:
        g[:, :lead].zero_()
    if lead + valid < Tg:
        g[:, lead + valid:].zero_()
    return g


def relative_positions_bucket_lut(T: int, num_buckets: int, max_distance: int) -> torch.Tensor:
    """bucket(delta) for delta in [-(T-1), T-1] (index delta+T-1).  Host integer/fp32 glue computed with the same torch
    CPU ops as the reference `_relative_positions_bucket` (WavLM/modules.py:417-443), which also runs on the host."""
    rp = torch.arange(-(T - 1), T, dtype=torch.long)
    nb = num_buckets // 2
    buckets = (rp > 0).to(torch.long) * nb
    rp = torch.abs(rp)
    max_exact = nb // 2
    is_small = rp < max_exact
    large = max_exact + (torch.log(rp.float() / max_exact) / math.log(max_distance / max_exact) * (nb - max_exact)).to(torch.long)
    large = torch.min(large, torch.full_like(large, nb - 1))
    return (buckets + torch.where(is_small, rp, large)).to(torch.int32)


def bias_radius(lut: torch.Tensor, num_buckets: int) -> int:
    """Smallest r such that every |delta| >= r falls in the last bucket of its side (num_buckets - 1 for delta > 0,
    num_buckets // 2 - 1 for delta < 0): the log branch of the bucketing clamps there, so tab[h, delta] = tab[h, +-r] beyond.
    T - 1 when a side never saturates within the utterance.  `lut`: bucket(delta) for delta in [-(T-1), T-1]."""
    T = (lut.numel() + 1) // 2
    lut = lut.cpu()
    nb = num_buckets // 2
    r = 0
    for side, last in ((lut[T - 1:], 2 * nb - 1), (lut[:T].flip(0), nb - 1)):   # index = |delta|
        off = (side != last).nonzero()
        if off.numel():
            r = max(r, int(off[-1]) + 1)
    return min(r, T - 1)


ATTN_MAX_FRAMES = 16384   # longest input of the long-utterance attention kernels (csrc/attn_long.cu)
_T_BWD_FUSED = 2048       # longest input of the fused attention backward (its shared-memory tables grow with T)
_T_BWD_SPLIT = 4096       # longest input of the two-kernel attention backward (same reason)


def attn_kernels(T: int, has_bias: bool):
    """(forward, backward) attention kernels for T frames.  Shapes the per-CTA-table kernels accept stay on them: forward
    `attn_fwd` up to its shared-memory limit (3072 frames with the bias, 16384 without), backward the fused kernel up to 2048
    and `attn_bwd` up to 4096.  Longer inputs, up to ATTN_MAX_FRAMES, run the long-utterance kernels, whose shared memory
    does not depend on T."""
    if not 1 <= T <= ATTN_MAX_FRAMES:
        raise ValueError(f"attention supports 1..{ATTN_MAX_FRAMES} frames (got T={T}, {T / 50:.1f} s of audio)")
    fwd = "attn_fwd" if T <= ops.attn_fwd_max_frames(has_bias) else "attn_fwd_long"
    bwd = "attn_bwd_fused" if T <= _T_BWD_FUSED else ("attn_bwd" if T <= _T_BWD_SPLIT else "attn_bwd_long")
    return fwd, bwd


class FlatGrads:
    """One flat fp32 gradient buffer; every parameter's `.grad` is a view into it."""

    def __init__(self, groups: List[List[torch.nn.Parameter]], device):
        self.params: List[torch.nn.Parameter] = [p for g in groups for p in g]
        total, self.offsets = 0, {}
        for p in self.params:
            self.offsets[id(p)] = total
            total += (p.numel() + 3) // 4 * 4  # keep every view 16-byte aligned
        self.flat = torch.zeros(total, dtype=torch.float32, device=device)
        self.views = {id(p): self.flat[self.offsets[id(p)]: self.offsets[id(p)] + p.numel()].view_as(p) for p in self.params}

    def view(self, p) -> torch.Tensor:
        return self.views[id(p)]

    def attach(self):
        """Make every trainable p.grad the flat view.  A parameter whose grad was reset to None (optimizer.zero_grad) gets a
        zeroed view: autograd semantics are 'accumulate into .grad', and the kernels accumulate with atomics."""
        need_zero = any(p.requires_grad and p.grad is None for p in self.params)
        if need_zero:
            self.flat.zero_()
        for p in self.params:
            if not p.requires_grad:
                continue
            v = self.views[id(p)]
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                if p.grad is not None:
                    v.copy_(p.grad)
                p.grad = v


def grad_layout(m):
    """[(stage, [groups of parameters])] in the order the backward pass COMPLETES the gradients: loss heads and the final
    encoder LayerNorm first, then the layers from the last to the first (q/k/v adjacent so the fused [3D, D] weight gradient is
    one GEMM), then the stem (pos_conv, projection, mask embedding), then the conv stack from its last layer to its first.
    The flat buffer is laid out in this order, so a contiguous slice is final as soon as its last stage has run backward and
    can be all-reduced while the rest of the backward pass is still running (parallel.OverlappedGradSync)."""
    layers = list(m.encoder.layers)
    taken = set()

    def take(ps):
        out = [p for p in ps if id(p) not in taken]
        taken.update(id(p) for p in out)
        return out

    per_layer = []
    for lyr in layers:
        a = lyr.self_attn
        w = take([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight])
        b = take([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias])
        rest = take(list(lyr.parameters()))
        per_layer.append([w, b, rest])
    conv = []
    for blk in reversed(list(m.feature_extractor.conv_layers)):
        conv += take(list(blk.parameters()))
    stem = take(list(m.encoder.pos_conv.parameters()))
    if m.post_extract_proj is not None:
        stem += take(list(m.post_extract_proj.parameters()))
    stem += take(list(m.layer_norm.parameters())) + take([m.mask_emb])
    head = take(list(m.parameters()))  # everything else: encoder.layer_norm[_for_extract], final_proj, label embeddings, ...
    stages = [("head", [head])]
    for i in reversed(range(len(layers))):
        stages.append((("layer", i), per_layer[i]))
    stages.append(("stem", [stem]))
    stages.append(("conv", [conv]))
    return stages


def build_flat_grads(m, device):
    """(FlatGrads, {stage: [first, last) element}, [stages in backward order]) for a model (host logic, any device)."""
    stages = grad_layout(m)
    flat = FlatGrads([g for _, groups in stages for g in groups], device)
    ranges = {}
    for stage, groups in stages:
        ps = [p for g in groups for p in g]
        if ps:
            ranges[stage] = (flat.offsets[id(ps[0])], flat.offsets[id(ps[-1])] + (ps[-1].numel() + 3) // 4 * 4)
    return flat, ranges, [st for st, _ in stages if st in ranges]


class ConvGeom:
    """Frame counts and buffer geometry of the strided conv stack (WavLM/WavLM.py:378-449)."""

    def __init__(self, conv_layers, L_: int):
        self.layers = conv_layers
        self.T = []
        t = L_
        for (_, k, s) in conv_layers:
            t = (t - k) // s + 1
            self.T.append(t)
        assert self.T[-1] >= 1, "waveform too short for the conv stack"
        self.Tp = [_even(t) for t in self.T]                       # activation rows per batch (even)
        self.lead, self.Tg = [], []                                # gradient buffers
        for i, (_, k, s) in enumerate(conv_layers):
            lead = (k + s - 1) // s - 1
            self.lead.append(lead)
            t_in = L_ if i == 0 else self.T[i - 1]
            self.Tg.append(_even((t_in + s - 1) // s + lead + 1))


def conv_valid_rows(last: torch.Tensor, conv_layers, T_list) -> torch.Tensor:
    """Rows of every conv layer's output that the first `last[b]` output frames of the LAST layer depend on: int32 [n_layers, B]
    (row l contiguous).  V_L = last;  V_l = s_{l+1} * (V_{l+1} - 1) + k_{l+1}  (0 stays 0), clamped to the layer's frame count.
    Works on host or device tensors; anything beyond V_l[b] is padding that no valid frame ever reads (the reference's own
    length formula, WavLM.py:311-321, makes the receptive field of a valid frame end inside the valid samples)."""
    v = last.to(torch.int32)
    out = [None] * len(conv_layers)
    out[-1] = v.clamp(max=int(T_list[-1]))
    for l in range(len(conv_layers) - 2, -1, -1):
        _, k, s = conv_layers[l + 1]
        nxt = out[l + 1]
        out[l] = torch.where(nxt > 0, s * (nxt - 1) + k, torch.zeros_like(nxt)).clamp(max=int(T_list[l]))
    return torch.stack(out).to(torch.int32).contiguous()


class Engine:
    def __init__(self, model):
        self.m = model
        self.cfg = model.cfg
        self.dev = None
        self.prepared_version = None
        self.lut_cache: Dict[int, torch.Tensor] = {}
        self.radius_cache: Dict[int, int] = {}
        self.flat: Optional[FlatGrads] = None
        self._params = None
        self.drop: Optional[DR.DropState] = None  # set per forward pass by WavLM._begin (training-mode dropout)
        self.conv_valid_last = None  # ragged batch: int32 [B] valid frames of the extractor output (set per call by WavLM._extractor)
        self.grad_sync = None  # parallel.OverlappedGradSync: told when a stage of the backward pass has produced its gradients
        self.ragged_valid = None  # int32 [B] valid frames per utterance of the current forward (ragged batch), else None

    def backward_stage_done(self, stage):
        if self.grad_sync is not None:
            self.grad_sync.stage_done(stage)

    # ------------------------------------------------------------------------------------------------ setup
    def _ensure_device(self, device):
        if self.dev == device:
            return
        L.check_device()
        self.dev = device
        m, cfg = self.m, self.cfg
        D, Fd, H = cfg.encoder_embed_dim, cfg.encoder_ffn_embed_dim, cfg.encoder_attention_heads
        convs = m.conv_cfg
        C = convs[-1][0]
        assert all(c[0] == C for c in convs), "conv stack must have a constant channel count"
        assert D == H * 64, "head_dim must be 64"
        assert m.post_extract_proj is not None, "encoder_embed_dim must differ from the conv dim (projection layer)"
        e = lambda *s: torch.empty(*s, dtype=BF, device=device)
        self.wf, self.wd = {}, {}
        for i, (_, k, s) in enumerate(convs):
            if i == 0:
                continue
            self.wf[i] = e(C, k * C)
            self.wd[i] = [e(C, ((k - rho + s - 1) // s) * C) for rho in range(min(s, k))]
        self.wp, self.wpT = e(D, C), e(C, D)
        G, taps = cfg.conv_pos_groups, cfg.conv_pos
        self.pc_fwd, self.pc_dg = e(G, 64, taps, 64), e(G, 64, taps, 64)
        self.pc_norm2 = torch.zeros(2 * taps, dtype=torch.float32, device=device)   # holds fp64[taps] (deterministic tap norms)
        self.lw = []
        for lyr in m.encoder.layers:
            # q/k/v masters become views of ONE fused [3D, D] / [3D] fp32 tensor (same values, same state_dict keys): the fused
            # projection operand is then a single prep call and the fused bias needs no copy at all
            a = lyr.self_attn
            fw = torch.cat([a.q_proj.weight.data, a.k_proj.weight.data, a.v_proj.weight.data], 0).contiguous()
            fb = torch.cat([a.q_proj.bias.data, a.k_proj.bias.data, a.v_proj.bias.data], 0).contiguous()
            for j, proj in enumerate((a.q_proj, a.k_proj, a.v_proj)):
                proj.weight.data = fw[j * D:(j + 1) * D]
                proj.bias.data = fb[j * D:(j + 1) * D]
            self.lw.append(dict(qkv=e(3 * D, D), qkvT=e(D, 3 * D), bqkv=fb, wqkv_master=fw,
                                o=e(D, D), oT=e(D, D), w1=e(Fd, D), w1T=e(D, Fd), w2=e(D, Fd), w2T=e(Fd, D)))
        # descriptor table for the one-launch nn.Linear operand preparation (b200s_prep_linear_batched)
        import struct
        recs, tiles = [], 0

        def add(src, N, K, dst, ld, dstT, ldT):
            nonlocal tiles
            tk = (K + 63) // 64  # 64 x 64 tiles (b200s_prep_linear_batched)
            recs.append(struct.pack("<QQQqqiiii", src.data_ptr(), dst.data_ptr(), dstT.data_ptr(), ld, ldT, N, K, tiles, tk))
            tiles += ((N + 63) // 64) * tk

        add(m.post_extract_proj.weight.data, D, C, self.wp, C, self.wpT, D)
        for lyr, w in zip(m.encoder.layers, self.lw):
            add(w["wqkv_master"], 3 * D, D, w["qkv"], D, w["qkvT"], 3 * D)
            add(lyr.self_attn.out_proj.weight.data, D, D, w["o"], D, w["oT"], D)
            add(lyr.fc1.weight.data, Fd, D, w["w1"], D, w["w1T"], Fd)
            add(lyr.fc2.weight.data, D, Fd, w["w2"], Fd, w["w2T"], D)
        self.prep_descs = torch.frombuffer(bytearray(b"".join(recs)), dtype=torch.uint8).to(device)
        self.prep_n, self.prep_tiles = len(recs), tiles
        self.prep_ptrs = [(lyr.self_attn.k_proj.weight, w["wqkv_master"]) for lyr, w in zip(m.encoder.layers, self.lw)]
        # flat gradient buffer in backward-completion order, q/k/v adjacent per layer
        self.flat, self.stage_ranges, self.stage_order = build_flat_grads(m, device)

    def _param_version(self):
        if self._params is None:  # Module.parameters() walks the whole module tree: cache the list (the set never changes)
            self._params = list(self.m.parameters())
        return tuple(p._version for p in self._params)

    def prepare(self, force=False):
        """fp32 masters -> bf16 GEMM operands (transposes, tap-major conv layouts, weight-normed pos_conv, fused qkv)."""
        ver = self._param_version()
        if not force and ver == self.prepared_version:
            return
        m, cfg = self.m, self.cfg
        D, Fd = cfg.encoder_embed_dim, cfg.encoder_ffn_embed_dim
        convs = m.conv_cfg
        C = convs[-1][0]
        for i, (_, k, s) in enumerate(convs):
            if i == 0:
                continue
            w = m.feature_extractor.conv_layers[i][0].weight
            ops.prep_conv_fwd(w, C, C, k, self.wf[i])
            for rho in range(min(s, k)):
                ops.prep_conv_dgrad(w, C, C, k, s, rho, self.wd[i][rho])
        pc = m.encoder.pos_conv[0]
        ops.posconv_prep(pc.weight_v, pc.weight_g, D, cfg.conv_pos_groups, cfg.conv_pos, self.pc_norm2, self.pc_fwd, self.pc_dg)
        for kw, fw in self.prep_ptrs:  # the descriptor table holds raw master pointers: they must not have moved
            if kw.data_ptr() != fw.data_ptr() + 4 * D * D:
                raise RuntimeError("model parameters were re-allocated after the first GPU forward (e.g. .to()/.cuda()); "
                                   "move the model to its device before the first call")
        ops.prep_linear_batched(self.prep_descs, self.prep_n, self.prep_tiles)  # every nn.Linear operand, one launch
        self.prepared_version = ver

    def lut(self, T: int) -> torch.Tensor:
        if T not in self.lut_cache:
            self.lut_cache[T] = relative_positions_bucket_lut(T, self.cfg.num_buckets, self.cfg.max_distance).to(self.dev)
        return self.lut_cache[T]

    def tab_radius(self, T: int) -> int:
        """Saturation radius of the bias table for T frames (bias_radius of the cached LUT), for the long attention kernels."""
        if T not in self.radius_cache:
            self.radius_cache[T] = bias_radius(self.lut(T), self.cfg.num_buckets)
        return self.radius_cache[T]

    def active_drop(self) -> Optional[DR.DropState]:
        """Dropout state of the current forward pass (None in eval mode or when every probability is 0)."""
        return self.drop if self.m.training else None

    def g(self, p):  # gradient view of a parameter
        return self.flat.view(p)

    # ---- row-wise GEMMs of the layer stack: flat over all B*T rows, or -- for a ragged batch -- per utterance with the padded
    # tail of every utterance skipped (`rag`: int32 [B] valid frames on the device, see WavLM.extract_features)
    @staticmethod
    def _mm(a, K, w, N, out, rag, T, B, **epi):
        if rag is None:
            ops.gemm_rows(a, 0, K, B * T, 1, K, w, N, out, 0, N, L.make_epilogue(**epi) if epi else None)
            return
        kw = dict(epi)
        for name, ldk, bsk in (("res1", "res1_ld", "res1_bs"), ("res2", "res2_ld", "res2_bs"), ("gelu_aux", "aux_ld", "aux_bs"),
                               ("out_pre", "pre_ld", "pre_bs")):
            if kw.get(name) is not None:
                kw[bsk] = T * kw[ldk]
        ops.gemm_rows(a, T * K, K, T, B, K, w, N, out, T * N, N, L.make_epilogue(**kw) if kw else None, valid=rag)

    @staticmethod
    def _wg(y, N, x, K, dw, rag, T, B):
        if rag is None:
            ops.gemm_wgrad(y, 0, N, x, 0, K, B * T, 1, N, K, dw, K)
        else:
            ops.gemm_wgrad(y, T * N, N, x, T * K, K, T, B, N, K, dw, K, valid=rag)

    # ---- LayerNorm whose output feeds a gated attention: the gate (WavLM/modules.py:523-533) is computed in the same pass
    def _uses_gate(self) -> bool:
        return bool(getattr(self.cfg, "relative_position_embedding", False) and getattr(self.cfg, "gru_rel_pos", False))

    def _ln_with_gate(self, x, ln, y, mean, rstd, T, B, D, consumer_idx, rag=None):
        """y = ln(x) and the gate of encoder.layers[consumer_idx].self_attn; remembered until that layer consumes y."""
        a = self.m.encoder.layers[consumer_idx].self_attn
        H = self.cfg.encoder_attention_heads
        if D not in (256, 512, 768, 1024):  # the fused kernel needs 8 columns per lane; narrow models take two passes
            ops.layer_norm_fwd(x, T * D, D, ln.weight, ln.bias, y, T * D, D, mean, rstd, T, B, D, valid=rag)
            self._pending_gate = None
            return None
        gate = torch.empty(B, H, T, dtype=torch.float32, device=x.device)
        ops.layer_norm_gate_fwd(x, T * D, D, ln.weight, ln.bias, y, T * D, D, mean, rstd, T, B, D, a.grep_linear.weight,
                                a.grep_linear.bias, a.grep_a, H, gate, valid=rag)
        self._pending_gate = (y.data_ptr(), consumer_idx, gate)
        return gate

    def _take_gate(self, x, idx):
        pg = getattr(self, "_pending_gate", None)
        self._pending_gate = None
        if pg is not None and pg[0] == x.data_ptr() and pg[1] == idx:
            return pg[2]
        return None

    # ------------------------------------------------------------------------------------------------ conv stack
    def conv_forward(self, wav: torch.Tensor, save: bool):
        """ConvFeatureExtractionModel.forward (WavLM/WavLM.py:485-504) -> channels-last features [B, Tp, C] (valid rows T)."""
        m, cfg = self.m, self.cfg
        convs = m.conv_cfg
        B, L_ = wav.shape
        geo = ConvGeom(convs, L_)
        C = convs[0][0]
        ln_mode = cfg.extractor_mode == "layer_norm"
        dev = wav.device
        st = dict(geo=geo, wav=wav, a=[], y=[], mean=[], rstd=[])
        # ragged batch: per layer, the rows any valid output frame depends on; the conv GEMMs zero-fill whole tiles beyond them
        # (layer 0 and the LayerNorms still walk every row: finite values, never read by a valid frame)
        cv = None
        if self.conv_valid_last is not None:
            cv = conv_valid_rows(self.conv_valid_last, convs, geo.T).to(dev, non_blocking=True)
        st["cv"] = cv
        vrow = (lambda i: cv[i]) if cv is not None else (lambda i: None)
        blk0 = m.feature_extractor.conv_layers[0]
        _, k0, s0 = convs[0]
        a0 = torch.empty(B, geo.Tp[0], C, dtype=BF, device=dev)
        norm0 = blk0[2][1] if ln_mode else blk0[2]
        if ln_mode:
            fmean = torch.empty(B, geo.T[0], dtype=torch.float32, device=dev)
            frstd = torch.empty(B, geo.T[0], dtype=torch.float32, device=dev)
            ops.conv0_fwd(wav, L_, B, geo.T[0], C, k0, s0, blk0[0].weight, norm0.weight, norm0.bias, 1, None, fmean, frstd,
                          a0, geo.Tp[0] * C)
            st["stats0"] = (fmean, frstd)
        else:
            stats = torch.empty(B * C * 2 + B * 128, dtype=torch.float64, device=dev)  # per-(b,c) sums + autocorrelation
            ops.conv0_fwd(wav, L_, B, geo.T[0], C, k0, s0, blk0[0].weight, norm0.weight, norm0.bias, 0, stats, None, None,
                          a0, geo.Tp[0] * C)
            st["stats0"] = stats
        st["a"].append(a0)
        st["y"].append(None)
        st["mean"].append(None)
        st["rstd"].append(None)
        for i in range(1, len(convs)):
            _, k, s = convs[i]
            Ti, Tpi = geo.T[i], geo.Tp[i]
            a_prev = st["a"][i - 1]
            out = torch.empty(B, Tpi, C, dtype=BF, device=dev)
            if ln_mode:
                y = torch.empty(B, Tpi, C, dtype=BF, device=dev)
                ops.gemm_rows(a_prev, geo.Tp[i - 1] * C, s * C, Ti, B, k * C, self.wf[i], C, y, Tpi * C, C, None, valid=vrow(i))
                ln = m.feature_extractor.conv_layers[i][2][1]
                mean = torch.empty(B * Ti, dtype=torch.float32, device=dev)
                rstd = torch.empty(B * Ti, dtype=torch.float32, device=dev)
                ops.layer_norm_fwd(y, Tpi * C, C, ln.weight, ln.bias, out, Tpi * C, C, mean, rstd, Ti, B, C, gelu=True, valid=vrow(i))
                st["y"].append(y); st["mean"].append(mean); st["rstd"].append(rstd)
            else:
                y = torch.empty(B, Tpi, C, dtype=BF, device=dev) if save else None
                epi = L.make_epilogue(gelu=2, out_pre=y, pre_bs=Tpi * C, pre_ld=C)  # y = gelu'(conv output), used by backward
                ops.gemm_rows(a_prev, geo.Tp[i - 1] * C, s * C, Ti, B, k * C, self.wf[i], C, out, Tpi * C, C, epi, valid=vrow(i))
                st["y"].append(y); st["mean"].append(None); st["rstd"].append(None)
            st["a"].append(out)
            if not save:
                st["a"][i - 1] = None if i - 1 > 0 else st["a"][0]
        return st

    def conv_backward(self, st, dfeat: torch.Tensor):
        """dfeat: gradient w.r.t. the extractor output a[-1] (bf16 [B, Tp, C] layout).  Accumulates all conv-stack
        parameter gradients; the waveform gets none."""
        m, cfg = self.m, self.cfg
        convs = m.conv_cfg
        geo: ConvGeom = st["geo"]
        wav = st["wav"]
        B, L_ = wav.shape
        C = convs[0][0]
        dev = wav.device
        ln_mode = cfg.extractor_mode == "layer_norm"
        n = len(convs)
        dA = dfeat  # gradient w.r.t. a[i], no-lead layout [B, Tp_i, C]
        gpad = None
        cv = st.get("cv")
        for i in range(n - 1, 0, -1):
            _, k, s = convs[i]
            Ti, Tpi, lead, Tg = geo.T[i], geo.Tp[i], geo.lead[i], geo.Tg[i]
            # ---- dY_i (gradient w.r.t. the conv output of layer i) in lead layout
            if gpad is None:
                gpad = _grad_rows(B, Tg, C, lead, Ti, dev)
                gv = gpad[:, lead:]
                if ln_mode:
                    ln = m.feature_extractor.conv_layers[i][2][1]
                    ops.layer_norm_bwd(dA, Tpi * C, C, st["y"][i], Tpi * C, C, st["mean"][i], st["rstd"][i], ln.weight,
                                       ln.bias, None, 0, 0, gv, Tg * C, C, self.g(ln.weight), self.g(ln.bias), None, Ti, B, C,
                                       gelu=True, valid=cv[i] if cv is not None else None)
                else:
                    ops.dgelu_mul(dA, Tpi * C, C, st["y"][i], Tpi * C, C, gv, Tg * C, C, Ti, B, C, None, pre_is_grad=True)
            gv = gpad[:, lead:]
            # ---- weight gradient: dW[co, (j,ci)] = sum dY[b,t,co] * a_{i-1}[b, s*t + j, ci]
            a_prev = st["a"][i - 1]
            dwk = torch.zeros(C, k * C, dtype=torch.float32, device=dev)
            ops.gemm_wgrad(gv, Tg * C, C, a_prev, geo.Tp[i - 1] * C, s * C, Ti, B, C, k * C, dwk, k * C,
                           valid=cv[i] if cv is not None else None)
            w = m.feature_extractor.conv_layers[i][0].weight
            ops.unprep_conv_wgrad(dwk, C, C, k, self.g(w))
            # ---- input gradient, one GEMM per phase rho of the stride
            T_in, Tp_in = geo.T[i - 1], geo.Tp[i - 1]
            fuse_dgelu = (not ln_mode) and (i - 1 >= 1)
            if fuse_dgelu or (ln_mode and i - 1 >= 1):
                lead_p, Tg_p = geo.lead[i - 1], geo.Tg[i - 1]
                gnext = _grad_rows(B, Tg_p, C, lead_p, T_in, dev)
            if fuse_dgelu:
                dst, dst_bs, dst_off = gnext, Tg_p * C, lead_p * C
            else:
                dAp = torch.empty(B, Tp_in, C, dtype=BF, device=dev)  # rows < T_in are written by the phase GEMMs; the pad row is never read
                dst, dst_bs, dst_off = dAp, Tp_in * C, 0
            for rho in range(min(s, k)):
                nm = (k - rho + s - 1) // s
                n_u = (T_in - rho + s - 1) // s
                if n_u <= 0:
                    continue
                a_view = gpad.view(-1)[(lead - (nm - 1)) * C:]
                epi = None
                if fuse_dgelu:
                    y_prev = st["y"][i - 1]
                    epi = L.make_epilogue(dgelu=2, gelu_aux=y_prev.view(-1)[rho * C:], aux_bs=Tp_in * C, aux_ld=s * C)
                # rows u' of phase rho are input frames s*u' + rho: beyond the utterance's valid input frames the gradient is zero
                pv = ((cv[i - 1] - rho + (s - 1)).clamp(min=0) // s).to(torch.int32) if cv is not None else None
                ops.gemm_rows(a_view, Tg * C, C, n_u, B, nm * C, self.wd[i][rho], C, dst.view(-1)[dst_off + rho * C:], dst_bs,
                              s * C, epi, valid=pv)
            if fuse_dgelu:
                gpad = gnext
                dA = None
            elif ln_mode and i - 1 >= 1:
                ln = m.feature_extractor.conv_layers[i - 1][2][1]
                ops.layer_norm_bwd(dAp, Tp_in * C, C, st["y"][i - 1], Tp_in * C, C, st["mean"][i - 1], st["rstd"][i - 1],
                                   ln.weight, ln.bias, None, 0, 0, gnext[:, lead_p:], Tg_p * C, C, self.g(ln.weight),
                                   self.g(ln.bias), None, T_in, B, C, gelu=True, valid=cv[i - 1] if cv is not None else None)
                gpad = gnext
                dA = None
            else:
                dA = dAp  # gradient w.r.t. a[0]
        # ---- layer 0
        blk0 = m.feature_extractor.conv_layers[0]
        _, k0, s0 = convs[0]
        norm0 = blk0[2][1] if ln_mode else blk0[2]
        if n == 1:
            dA = dfeat
        if ln_mode:
            fmean, frstd = st["stats0"]
            # (the incoming gradient buffer doubles as the dconv workspace: it is engine-owned scratch, consumed here)
            ws = dA if (n > 1 and dA.dtype == BF and dA.is_contiguous() and k0 <= 10) else None
            ops.conv0_bwd(wav, L_, B, geo.T[0], C, k0, s0, blk0[0].weight, norm0.weight, norm0.bias, 1, None, None, fmean,
                          frstd, dA, geo.Tp[0] * C, self.g(blk0[0].weight), self.g(norm0.weight), self.g(norm0.bias),
                          dconv_ws=ws, ws_bs=geo.Tp[0] * C)
        else:
            bstats = torch.empty(B, C, 12, dtype=torch.float32, device=dev)
            ops.conv0_bwd(wav, L_, B, geo.T[0], C, k0, s0, blk0[0].weight, norm0.weight, norm0.bias, 0, st["stats0"], bstats,
                          None, None, dA, geo.Tp[0] * C, self.g(blk0[0].weight), self.g(norm0.weight), self.g(norm0.bias))

    # ------------------------------------------------------------------------------------------------ LN + proj + mask
    def project_forward(self, feats, T, mask_u8, pad_u8, save, want_features):
        """transpose -> LayerNorm(C) -> post_extract_proj -> mask_emb / zero padded frames (WavLM/WavLM.py:341-357,574-575).
        Writes into the zero-padded pos_conv input buffer."""
        m, cfg = self.m, self.cfg
        B, Tp, C = feats.shape
        D = cfg.encoder_embed_dim
        dev = feats.device
        half = cfg.conv_pos // 2
        fn = torch.empty(B, T, C, dtype=BF, device=dev)
        mean = torch.empty(B * T, dtype=torch.float32, device=dev)
        rstd = torch.empty(B * T, dtype=torch.float32, device=dev)
        ops.layer_norm_fwd(feats, Tp * C, C, m.layer_norm.weight, m.layer_norm.bias, fn, T * C, C, mean, rstd, T, B, C)
        Tpad = T + cfg.conv_pos
        xpad = torch.zeros(B, Tpad, D, dtype=BF, device=dev)
        xv = xpad[:, half:]
        epi = L.make_epilogue(bias=m.post_extract_proj.bias)
        ops.gemm_rows(fn, T * C, C, T, B, C, self.wp, D, xv, Tpad * D, D, epi)
        d = self.active_drop()
        if d is not None and d.p_input > 0:  # features = dropout_input(features), WavLM/WavLM.py:350
            ops.dropout_rows(xv, Tpad * D, D, None, 0, 0, xv, Tpad * D, D, T, B, D, d.p_input, d.key(DR.SITE_INPUT))
        features = xv[:, :T].clone() if want_features else None
        ops.frame_mask_fwd(xv, Tpad * D, D, T, B, D, mask_u8, pad_u8, m.mask_emb)
        return dict(fn=fn, mean=mean, rstd=rstd, xpad=xpad, feats=feats if save else None, features=features, drop=d)

    def project_backward(self, st, dxm, T, mask_u8, pad_u8, dfn_extra=None):
        """dxm: gradient w.r.t. the masked projection output, bf16 [B,T,D] (modified in place). Returns d(features) [B,Tp,C].
        `dfn_extra` (bf16 [B,T,C]): gradient arriving at the LayerNorm output from a second consumer (wav2vec 2.0 quantizer)."""
        m, cfg = self.m, self.cfg
        B = dxm.shape[0]
        D = cfg.encoder_embed_dim
        feats = st["feats"]
        Tp, C = feats.shape[1], feats.shape[2]
        dev = dxm.device
        ops.frame_mask_bwd(dxm, T * D, D, T, B, D, mask_u8, pad_u8, self.g(m.mask_emb))
        d = st["drop"]
        if d is not None and d.p_input > 0:
            ops.dropout_rows(dxm, T * D, D, None, 0, 0, dxm, T * D, D, T, B, D, d.p_input, d.key(DR.SITE_INPUT))
        ops.colsum(dxm, T * D, D, T, B, D, self.g(m.post_extract_proj.bias))
        ops.gemm_wgrad(dxm, T * D, D, st["fn"], T * C, C, T, B, D, C, self.g(m.post_extract_proj.weight), C)
        dfn = torch.empty(B, T, C, dtype=BF, device=dev)
        ops.gemm_rows(dxm, T * D, D, T, B, D, self.wpT, C, dfn, T * C, C,
                      L.make_epilogue(res1=dfn_extra, res1_bs=T * C, res1_ld=C) if dfn_extra is not None else None)
        dfeat = torch.empty(B, Tp, C, dtype=BF, device=dev)  # rows < T written below; the pad row is never read
        ops.layer_norm_bwd(dfn, T * C, C, feats, Tp * C, C, st["mean"], st["rstd"], m.layer_norm.weight, m.layer_norm.bias,
                           None, 0, 0, dfeat, Tp * C, C, self.g(m.layer_norm.weight), self.g(m.layer_norm.bias), None, T, B, C)
        return dfeat

    # ------------------------------------------------------------------------------------------------ pos_conv stage
    def posconv_forward(self, xpad, T, save):
        """x + gelu(pos_conv(x)) [-> encoder.layer_norm for post-LN models]  (WavLM/WavLM.py:577-582)."""
        m, cfg = self.m, self.cfg
        B, Tpad, D = xpad.shape
        dev = xpad.device
        G, taps, half = cfg.conv_pos_groups, cfg.conv_pos, cfg.conv_pos // 2
        xs = torch.empty(B, T, D, dtype=BF, device=dev)
        pre = torch.empty(B, T, D, dtype=BF, device=dev) if save else None
        pc = m.encoder.pos_conv[0]
        epi = L.make_epilogue(bias=pc.bias, gelu=2, out_pre=pre, pre_bs=T * D, pre_ld=D, res1=xpad[:, half:],
                              res1_bs=Tpad * D, res1_ld=D)
        ops.posconv_gemm(xpad, Tpad * D, T, B, D, G, taps, self.pc_fwd, xs, T * D, D, epi)
        d = self.active_drop()
        d = d if (d is not None and d.p > 0) else None
        st = dict(xpad=xpad, pre=pre, xs=xs, drop=d)
        if not cfg.layer_norm_first:
            x0 = torch.empty(B, T, D, dtype=BF, device=dev)
            mean = torch.empty(B * T, dtype=torch.float32, device=dev)
            rstd = torch.empty(B * T, dtype=torch.float32, device=dev)
            ln = m.encoder.layer_norm
            if d is None and self._uses_gate() and len(m.encoder.layers) > 0:
                self._ln_with_gate(xs, ln, x0, mean, rstd, T, B, D, 0)
            else:  # (with dropout the first layer's gate must see the DROPPED x: it is computed by that layer instead)
                ops.layer_norm_fwd(xs, T * D, D, ln.weight, ln.bias, x0, T * D, D, mean, rstd, T, B, D)
                self._pending_gate = None
            st.update(mean=mean, rstd=rstd)
            out = x0
        else:
            out = xs
        if d is not None:  # x = F.dropout(x, p=self.dropout), WavLM/WavLM.py:584 (in place: nothing below needs the undropped value)
            ops.dropout_rows(out, T * D, D, None, 0, 0, out, T * D, D, T, B, D, d.p, d.key(DR.SITE_ENCODER))
        return out, st

    def posconv_backward(self, st, dx0, T):
        m, cfg = self.m, self.cfg
        xpad = st["xpad"]
        B, Tpad, D = xpad.shape
        dev = xpad.device
        G, taps, half = cfg.conv_pos_groups, cfg.conv_pos, cfg.conv_pos // 2
        Cg = D // G
        d = st["drop"]
        if d is not None:
            dx0d = torch.empty(B, T, D, dtype=BF, device=dev)
            ops.dropout_rows(dx0, T * D, D, None, 0, 0, dx0d, T * D, D, T, B, D, d.p, d.key(DR.SITE_ENCODER))
            dx0 = dx0d
        if not cfg.layer_norm_first:
            ln = m.encoder.layer_norm
            dxs = torch.empty(B, T, D, dtype=BF, device=dev)
            ops.layer_norm_bwd(dx0, T * D, D, st["xs"], T * D, D, st["mean"], st["rstd"], ln.weight, ln.bias, None, 0, 0, dxs,
                               T * D, D, self.g(ln.weight), self.g(ln.bias), None, T, B, D)
        else:
            dxs = dx0
        pc = m.encoder.pos_conv[0]
        dpre = torch.zeros(B, Tpad, D, dtype=BF, device=dev)
        ops.dgelu_mul(dxs, T * D, D, st["pre"], T * D, D, dpre[:, half:], Tpad * D, D, T, B, D, self.g(pc.bias),
                      pre_is_grad=True)
        dwp = torch.zeros(G, Cg, taps, 64, dtype=torch.float32, device=dev)
        ops.posconv_wgrad(dpre[:, half:], Tpad * D, D, xpad, Tpad * D, T, B, D, G, taps, dwp)
        work = torch.empty(4 * taps, dtype=torch.float32, device=dev)   # fp64[2 * taps]
        ops.posconv_unprep(pc.weight_v, pc.weight_g, dwp, D, G, taps, work, self.g(pc.weight_v), self.g(pc.weight_g))
        # input gradient: correlation with the flipped, transposed taps; frame t reads dpre rows t-63 .. t+64
        dxm = torch.empty(B, T, D, dtype=BF, device=dev)
        epi = L.make_epilogue(res1=dxs, res1_bs=T * D, res1_ld=D)
        ops.posconv_gemm(dpre.view(-1)[D:], Tpad * D, T, B, D, G, taps, self.pc_dg, dxm, T * D, D, epi)
        return dxm

    # ------------------------------------------------------------------------------------------------ transformer layer
    def layer_forward(self, idx: int, x: torch.Tensor, pad_u8, tab, save: bool):
        """TransformerSentenceEncoderLayer.forward (WavLM/WavLM.py:677-742) + MultiheadAttention fast path
        (WavLM/modules.py:457-564) on x: bf16 [B,T,D]."""
        m, cfg = self.m, self.cfg
        lyr = m.encoder.layers[idx]
        a = lyr.self_attn
        w = self.lw[idx]
        B, T, D = x.shape
        M = B * T
        Fd, H = cfg.encoder_ffn_embed_dim, cfg.encoder_attention_heads
        dev = x.device
        e = lambda *s: torch.empty(*s, dtype=BF, device=dev)
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        pre_ln = cfg.layer_norm_first
        d = self.active_drop()
        p_h = d.p if d is not None else 0.0
        p_a = d.p_attn if d is not None else 0.0
        p_act = d.p_act if d is not None else 0.0
        if p_a > 0 and T > _T_BWD_FUSED:
            raise NotImplementedError(f"attention_dropout > 0 is implemented in the fused attention kernels for T <= {_T_BWD_FUSED} "
                                      f"frames (got T={T}); set attention_dropout=0 for longer inputs")
        attn_fwd_kernel = attn_kernels(T, tab is not None)[0]
        st = dict(x=x, drop=d)
        rag = self.ragged_valid if pad_u8 is not None else None   # int32 [B] valid frames (ragged batch) or None
        want_gate = tab is not None and cfg.gru_rel_pos
        gate = self._take_gate(x, idx) if (want_gate and not pre_ln) else None
        if pre_ln:
            xn, st["mean1"], st["rstd1"] = e(B, T, D), f(M), f(M)
            ln = lyr.self_attn_layer_norm
            if want_gate:
                gate = self._ln_with_gate(x, ln, xn, st["mean1"], st["rstd1"], T, B, D, idx, rag=rag)
                self._pending_gate = None
            else:
                ops.layer_norm_fwd(x, T * D, D, ln.weight, ln.bias, xn, T * D, D, st["mean1"], st["rstd1"], T, B, D, valid=rag)
            st["xn"] = xn
        else:
            xn = x
        qkv = e(B, T, 3 * D)
        self._mm(xn, D, w["qkv"], 3 * D, qkv, rag, T, B, bias=w["bqkv"])
        if want_gate and gate is None:  # the producer of x did not leave a gate behind (first use, layerdrop, foreign input)
            gate = f(B, H, T)
            ops.gate_fwd(xn, T * D, D, T, B, H, a.grep_linear.weight, a.grep_linear.bias, a.grep_a, gate)
        ao, lse = e(B, T, D), f(B, H, T)
        dmask = None
        if p_a > 0:  # dropout on the probabilities (WavLM/modules.py:551); the kernel leaves the keep bits for the backward
            dmask = torch.empty(ops.attn_dropout_mask_words(B, T, H), dtype=torch.int32, device=dev)
            ops.attn_fwd_dropout(qkv, gate, tab, pad_u8, ao, lse, B, T, H, 64 ** -0.5, p_a,
                                 d.key(DR.layer_site(idx, DR.L_ATTENTION)), dmask)
        elif attn_fwd_kernel == "attn_fwd":
            ops.attn_fwd(qkv, gate, tab, pad_u8, ao, lse, B, T, H, 64 ** -0.5)
        else:
            ops.attn_fwd_long(qkv, gate, tab, self.tab_radius(T), pad_u8, ao, lse, B, T, H, 64 ** -0.5)
        y1 = e(B, T, D)
        if p_h > 0:  # x + dropout1(out_proj(attn)), WavLM/WavLM.py:702-703,726-727
            self._mm(ao, D, w["o"], D, y1, rag, T, B, bias=a.out_proj.bias)
            ops.dropout_rows(y1, T * D, D, x, T * D, D, y1, T * D, D, T, B, D, p_h, d.key(DR.layer_site(idx, DR.L_DROPOUT1)))
        else:
            self._mm(ao, D, w["o"], D, y1, rag, T, B, bias=a.out_proj.bias, res1=x, res1_ld=D)
        if pre_ln:
            x1 = y1
            x1n, st["mean2"], st["rstd2"] = e(B, T, D), f(M), f(M)
            ln = lyr.final_layer_norm
            ops.layer_norm_fwd(x1, T * D, D, ln.weight, ln.bias, x1n, T * D, D, st["mean2"], st["rstd2"], T, B, D, valid=rag)
            ffn_in = x1n
        else:
            x1, st["mean1"], st["rstd1"] = e(B, T, D), f(M), f(M)
            ln = lyr.self_attn_layer_norm
            ops.layer_norm_fwd(y1, T * D, D, ln.weight, ln.bias, x1, T * D, D, st["mean1"], st["rstd1"], T, B, D, valid=rag)
            ffn_in = x1
        hg = e(B, T, Fd)
        hp = e(B, T, Fd) if save else None
        self._mm(ffn_in, D, w["w1"], Fd, hg, rag, T, B, bias=lyr.fc1.bias, gelu=2, out_pre=hp, pre_ld=Fd)  # hp = gelu'(fc1 output)
        if p_act > 0:  # dropout2 after the activation (WavLM/WavLM.py:711,736); the same mask folded into the stored
            # derivative makes the backward epilogue (dy * hp) the gradient through activation AND dropout
            k_act = d.key(DR.layer_site(idx, DR.L_ACTIVATION))
            ops.dropout_rows(hg, T * Fd, Fd, None, 0, 0, hg, T * Fd, Fd, T, B, Fd, p_act, k_act)
            if hp is not None:
                ops.dropout_rows(hp, T * Fd, Fd, None, 0, 0, hp, T * Fd, Fd, T, B, Fd, p_act, k_act)
        y2 = e(B, T, D)
        if p_h > 0:  # residual + dropout3(fc2(.)), WavLM/WavLM.py:713-714,738-739
            self._mm(hg, Fd, w["w2"], D, y2, rag, T, B, bias=lyr.fc2.bias)
            ops.dropout_rows(y2, T * D, D, x1, T * D, D, y2, T * D, D, T, B, D, p_h, d.key(DR.layer_site(idx, DR.L_DROPOUT3)))
        else:
            self._mm(hg, Fd, w["w2"], D, y2, rag, T, B, bias=lyr.fc2.bias, res1=x1, res1_ld=D)
        if pre_ln:
            out = y2
        else:
            out, st["mean2"], st["rstd2"] = e(B, T, D), f(M), f(M)
            ln = lyr.final_layer_norm
            if want_gate and idx + 1 < len(m.encoder.layers):  # `out` is the next layer's input: leave its gate behind
                self._ln_with_gate(y2, ln, out, st["mean2"], st["rstd2"], T, B, D, idx + 1, rag=rag)
            else:
                ops.layer_norm_fwd(y2, T * D, D, ln.weight, ln.bias, out, T * D, D, st["mean2"], st["rstd2"], T, B, D, valid=rag)
        if save:
            st.update(qkv=qkv, gate=gate, ao=ao, lse=lse, y1=y1, x1=x1, ffn_in=ffn_in, hp=hp, hg=hg, y2=y2, tab=tab, pad=pad_u8,
                      dmask=dmask, rag=rag)
        return out, (st if save else None)

    def layer_backward(self, idx: int, st, dout: torch.Tensor, dtab):
        m, cfg = self.m, self.cfg
        lyr = m.encoder.layers[idx]
        a = lyr.self_attn
        w = self.lw[idx]
        x = st["x"]
        B, T, D = x.shape
        M = B * T
        Fd, H = cfg.encoder_ffn_embed_dim, cfg.encoder_attention_heads
        dev = x.device
        e = lambda *s: torch.empty(*s, dtype=BF, device=dev)
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        g = self.g
        pre_ln = cfg.layer_norm_first
        tab, pad = st["tab"], st["pad"]
        rag = st["rag"]
        d = st["drop"]
        p_h = d.p if d is not None else 0.0
        p_a = d.p_attn if d is not None else 0.0

        def through_dropout(dy, which):  # gradient entering a dropped branch: same mask, same scale (dy itself feeds the residual)
            dz = e(B, T, D)
            ops.dropout_rows(dy, T * D, D, None, 0, 0, dz, T * D, D, T, B, D, p_h, d.key(DR.layer_site(idx, which)))
            return dz

        # ---------------- FFN block
        if pre_ln:
            dy2 = dout                                           # x2 = x1 + fc2(...)
            dz2 = through_dropout(dy2, DR.L_DROPOUT3) if p_h > 0 else dy2
            ops.colsum(dz2, T * D, D, T, B, D, g(lyr.fc2.bias), valid=rag)
        else:
            dy2 = e(B, T, D)
            ln = lyr.final_layer_norm
            ops.layer_norm_bwd(dout, T * D, D, st["y2"], T * D, D, st["mean2"], st["rstd2"], ln.weight, ln.bias, None, 0, 0,
                               dy2, T * D, D, g(ln.weight), g(ln.bias), None if p_h > 0 else g(lyr.fc2.bias), T, B, D, valid=rag)
            dz2 = dy2
            if p_h > 0:
                dz2 = through_dropout(dy2, DR.L_DROPOUT3)
                ops.colsum(dz2, T * D, D, T, B, D, g(lyr.fc2.bias), valid=rag)
        self._wg(dz2, D, st["hg"], Fd, g(lyr.fc2.weight), rag, T, B)
        dhp = e(B, T, Fd)
        self._mm(dz2, D, w["w2T"], Fd, dhp, rag, T, B, dgelu=2, gelu_aux=st["hp"], aux_ld=Fd, colsum=g(lyr.fc1.bias))
        self._wg(dhp, Fd, st["ffn_in"], D, g(lyr.fc1.weight), rag, T, B)
        dx1 = e(B, T, D)
        if pre_ln:
            dffn_in = e(B, T, D)
            self._mm(dhp, Fd, w["w1T"], D, dffn_in, rag, T, B)
            ln = lyr.final_layer_norm
            # (without dropout1 the out_proj bias gradient is the column sum of dx1: taken inside the LayerNorm backward)
            ops.layer_norm_bwd(dffn_in, T * D, D, st["x1"], T * D, D, st["mean2"], st["rstd2"], ln.weight, ln.bias, dy2, T * D, D,
                               dx1, T * D, D, g(ln.weight), g(ln.bias), None if p_h > 0 else g(a.out_proj.bias), T, B, D, valid=rag)
            dy1 = dx1                                            # x1 = x + out_proj(attn)
            dz1 = dy1
            if p_h > 0:
                dz1 = through_dropout(dy1, DR.L_DROPOUT1)
                ops.colsum(dz1, T * D, D, T, B, D, g(a.out_proj.bias), valid=rag)
        else:
            self._mm(dhp, Fd, w["w1T"], D, dx1, rag, T, B, res1=dy2, res1_ld=D)
            dy1 = e(B, T, D)
            ln = lyr.self_attn_layer_norm
            ops.layer_norm_bwd(dx1, T * D, D, st["y1"], T * D, D, st["mean1"], st["rstd1"], ln.weight, ln.bias, None, 0, 0,
                               dy1, T * D, D, g(ln.weight), g(ln.bias), None if p_h > 0 else g(a.out_proj.bias), T, B, D, valid=rag)
            dz1 = dy1
            if p_h > 0:
                dz1 = through_dropout(dy1, DR.L_DROPOUT1)
                ops.colsum(dz1, T * D, D, T, B, D, g(a.out_proj.bias), valid=rag)
        # ---------------- attention block
        self._wg(dz1, D, st["ao"], D, g(a.out_proj.weight), rag, T, B)
        dao = e(B, T, D)
        self._mm(dz1, D, w["oT"], D, dao, rag, T, B)
        dqkv = e(B, T, 3 * D)
        delta = f(B, H, T)
        gate = st["gate"]
        dgate = f(B, H, T) if tab is not None else None
        attn_bwd_kernel = attn_kernels(T, tab is not None)[1]
        if attn_bwd_kernel == "attn_bwd_fused":
            key = (B, T, D)
            if getattr(self, "_dq_acc_key", None) != key:  # fp32 dQ accumulator: zero on entry, re-zeroed by the kernel
                self._dq_acc = torch.zeros(B, T, D, dtype=torch.float32, device=dev)
                self._dq_acc_key = key
            if p_a > 0:
                ops.attn_bwd_fused_dropout(st["qkv"], st["ao"], dao, gate, tab, pad, st["lse"], delta, self._dq_acc, dqkv, dgate,
                                           dtab if tab is not None else None, B, T, H, 64 ** -0.5, p_a, st["dmask"])
            else:
                ops.attn_bwd_fused(st["qkv"], st["ao"], dao, gate, tab, pad, st["lse"], delta, self._dq_acc, dqkv, dgate,
                                   dtab if tab is not None else None, B, T, H, 64 ** -0.5)
        elif attn_bwd_kernel == "attn_bwd":
            ops.attn_bwd(st["qkv"], st["ao"], dao, gate, tab, pad, st["lse"], delta, dqkv, dgate,
                         dtab if tab is not None else None, B, T, H, 64 ** -0.5)
        else:  # (with R < T-1 the saturated diagonals' gradient lands at delta = +-R: same bucket, same embedding gradient)
            ops.attn_bwd_long(st["qkv"], st["ao"], dao, gate, tab, self.tab_radius(T) if tab is not None else 0, pad, st["lse"],
                              delta, dqkv, dgate, dtab if tab is not None else None, B, T, H, 64 ** -0.5)
        ops.colsum(dqkv, T * 3 * D, 3 * D, T, B, 3 * D, g(a.q_proj.bias).view(-1), valid=rag)  # q,k,v bias grads are adjacent in the flat buffer
        attn_in = st["xn"] if pre_ln else x
        dxg = None
        if gate is not None:
            dxg = e(B, T, D)
            ops.gate_bwd(attn_in, T * D, D, T, B, H, a.grep_linear.weight, a.grep_linear.bias, a.grep_a, dgate, dxg, T * D, D,
                         g(a.grep_linear.weight), g(a.grep_linear.bias), g(a.grep_a), valid=rag)
        self._wg(dqkv, 3 * D, attn_in, D, g(a.q_proj.weight), rag, T, B)
        dx = e(B, T, D)
        if pre_ln:
            dxn = e(B, T, D)
            if dxg is not None:
                self._mm(dqkv, 3 * D, w["qkvT"], D, dxn, rag, T, B, res1=dxg, res1_ld=D)
            else:
                self._mm(dqkv, 3 * D, w["qkvT"], D, dxn, rag, T, B)
            ln = lyr.self_attn_layer_norm
            ops.layer_norm_bwd(dxn, T * D, D, x, T * D, D, st["mean1"], st["rstd1"], ln.weight, ln.bias, dy1, T * D, D, dx,
                               T * D, D, g(ln.weight), g(ln.bias), None, T, B, D, valid=rag)
        else:
            if dxg is not None:
                self._mm(dqkv, 3 * D, w["qkvT"], D, dx, rag, T, B, res1=dy1, res1_ld=D, res2=dxg, res2_ld=D)
            else:
                self._mm(dqkv, 3 * D, w["qkvT"], D, dx, rag, T, B, res1=dy1, res1_ld=D)
        return dx
