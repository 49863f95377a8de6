"""Long-utterance attention kernels (csrc/attn_long.cu) on the GPU: kernel parity against a row-chunked fp32 reference,
determinism, whole-model parity against the CPU oracle beyond the per-CTA-table kernels' limits, and full-width padding
invariance at 16383 frames."""
import pytest
import torch
from torch.utils.checkpoint import checkpoint

from oracle import wavlm_oracle as O

pytestmark = pytest.mark.gpu
SR = 16000


def bf(x):
    return x.to(torch.bfloat16)


def _attn_chunk(q, k, v, g, tab, pad, i0, T, scale):
    """Rows [i0, i0 + q.shape[2]) of the attention output; holds at most [B, H, chunk, T]."""
    s = torch.matmul(q, k.transpose(-1, -2)) * scale
    if tab is not None:
        i = torch.arange(i0, i0 + q.shape[2], device=q.device)[:, None]
        j = torch.arange(T, device=q.device)[None, :]
        s = s + g.unsqueeze(-1) * tab[:, (j - i) + T - 1].unsqueeze(0)
    if pad is not None:
        s = s.masked_fill(pad.bool()[:, None, None, :], float("-inf"))
    return torch.matmul(torch.softmax(s, dim=-1), v)


def attn_ref(qkv, gate, tab, pad, B, T, H, scale, chunk=1024):
    """fp32 dense attention, computed (and, under autograd, recomputed) chunk by chunk of query rows."""
    D = H * 64
    q, k, v = qkv.float().split(D, dim=-1)
    q, k, v = (t.reshape(B, T, H, 64).transpose(1, 2) for t in (q, k, v))
    g = gate if gate is not None else torch.ones(B, H, T, device=qkv.device)
    outs = []
    for i0 in range(0, T, chunk):
        i1 = min(T, i0 + chunk)
        outs.append(checkpoint(_attn_chunk, q[:, :, i0:i1], k, v, g[:, :, i0:i1], tab, pad, i0, T, scale, use_reentrant=False))
    return torch.cat(outs, dim=2).transpose(1, 2).reshape(B, T, D)


def make_case(B, T, H, table, padded, dev, seed):
    """table: 'random' (R = T-1), 'saturated' (released bucketing + random embedding, derived R) or None (no bias)."""
    from unispeech_b200.engine import bias_radius, relative_positions_bucket_lut
    torch.manual_seed(seed)
    D = H * 64
    qkv = bf(torch.randn(B, T, 3 * D, device=dev))
    gate = torch.rand(B, H, T, device=dev) * 2 + 0.2 if table else None
    tab, lut, R = None, None, 0
    if table == "random":
        tab, R = torch.randn(H, 2 * T - 1, device=dev), T - 1
    elif table == "saturated":
        lut = relative_positions_bucket_lut(T, 320, 800)
        R = bias_radius(lut, 320)
        lut = lut.to(dev)
        tab = torch.randn(320, H, device=dev)[lut.long()].t().contiguous()
    pad = None
    if padded:
        pad = torch.zeros(B, T, device=dev, dtype=torch.uint8)
        pad[0, T - T // 3:] = 1
    return qkv, gate, tab, lut, R, pad


FWD_CASES = [(1, 3073, 2, "random", False), (2, 5000, 2, "saturated", True), (1, 16384, 1, "saturated", False),
             (2, 100, 2, "random", True), (1, 1499, 2, "saturated", True)]


@pytest.mark.parametrize("B,T,H,table,padded", FWD_CASES)
def test_attn_fwd_long(cuda_device, B, T, H, table, padded):
    from unispeech_b200 import ops
    qkv, gate, tab, lut, R, pad = make_case(B, T, H, table, padded, cuda_device, seed=T)
    out = torch.empty(B, T, H * 64, device=cuda_device, dtype=torch.bfloat16)
    lse = torch.empty(B, H, T, device=cuda_device)
    ops.attn_fwd_long(qkv, gate, tab, R, pad, out, lse, B, T, H, 0.125)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = attn_ref(qkv, gate, tab, pad, B, T, H, 0.125)
    assert torch.isfinite(out.float()).all()
    d = (out.float() - ref).abs()
    if padded:
        d = d[pad == 0]
    assert d.max().item() < 0.03, d.max().item()


@pytest.mark.parametrize("B,T,H,table,padded", FWD_CASES + [(2, 4500, 2, None, True)])
def test_attn_bwd_long(cuda_device, B, T, H, table, padded):
    from unispeech_b200 import ops
    dev = cuda_device
    qkv, gate, tab, lut, R, pad = make_case(B, T, H, table, padded, dev, seed=T + 1)
    D = H * 64
    out = torch.empty(B, T, D, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, H, T, device=dev)
    if tab is None:
        ops.attn_fwd(qkv, gate, tab, pad, out, lse, B, T, H, 0.125)
    else:
        ops.attn_fwd_long(qkv, gate, tab, R, pad, out, lse, B, T, H, 0.125)
    dout = bf(torch.randn(B, T, D, device=dev))
    if padded:
        dout[pad.bool()] = 0
    delta = torch.empty(B, H, T, device=dev)
    dqkv = torch.zeros(B, T, 3 * D, device=dev, dtype=torch.bfloat16)
    dgate = torch.full((B, H, T), 7.0, device=dev) if tab is not None else None   # written, not accumulated
    dtab = torch.zeros(H, 2 * T - 1, device=dev) if tab is not None else None
    ops.attn_bwd_long(qkv, out, dout, gate, tab, R, pad, lse, delta, dqkv, dgate, dtab, B, T, H, 0.125)
    torch.cuda.synchronize()
    qr = qkv.float().requires_grad_(True)
    gr = gate.clone().requires_grad_(True) if tab is not None else None
    tr = tab.clone().requires_grad_(True) if tab is not None else None
    attn_ref(qr, gr, tr, pad, B, T, H, 0.125).backward(dout.float())
    assert torch.isfinite(dqkv.float()).all()
    scale_ref = qr.grad.abs().max().item()
    err = (dqkv.float() - qr.grad).abs().max().item()
    assert err < 0.03 * max(1.0, scale_ref), (err, scale_ref)
    if tab is None:
        return
    e1 = (dgate - gr.grad).abs().max().item()
    assert e1 < 0.03 * max(1.0, gr.grad.abs().max().item()), e1
    if lut is None:   # R = T - 1: d tab entry by entry
        want, got = tr.grad, dtab
    else:             # saturated: compare the embedding gradient after the bucket scatter
        want = torch.zeros(320, H, device=dev).index_add_(0, lut.long(), tr.grad.t().contiguous())
        got = torch.zeros(320, H, device=dev).index_add_(0, lut.long(), dtab.t().contiguous())
        beyond = torch.arange(-(T - 1), T, device=dev).abs() > R
        assert (dtab[:, beyond] == 0).all()   # the saturated diagonals are summed at +-R
    e2 = (got - want).abs().max().item()
    assert e2 < 0.03 * max(1.0, want.abs().max().item()), (e2, want.abs().max().item())


def test_attn_fwd_long_deterministic(cuda_device):
    from unispeech_b200 import ops
    B, T, H = 2, 5000, 2
    qkv, gate, tab, lut, R, pad = make_case(B, T, H, "saturated", True, cuda_device, seed=9)
    outs = []
    for _ in range(2):
        out = torch.empty(B, T, H * 64, device=cuda_device, dtype=torch.bfloat16)
        lse = torch.empty(B, H, T, device=cuda_device)
        ops.attn_fwd_long(qkv, gate, tab, R, pad, out, lse, B, T, H, 0.125)
        outs.append((out, lse))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def _hidden(h):
    return h[0] if isinstance(h, (tuple, list)) else h


# max-abs on hidden states.  tests/test_model_gpu.py uses 0.12 up to 1499 frames; at 5000 frames the no-bias pre-LN model,
# whose forward runs only the per-CTA-table kernel attn_fwd, reaches 0.121 on the B200 (mean-abs 0.015): the bf16 error of a
# softmax over 5000 keys, not of the long kernels
HID_TOL = 0.15
GRAD_NAMES = ["encoder.layers.0.self_attn.relative_attention_bias.weight", "encoder.layers.1.self_attn.grep_linear.weight",
              "encoder.layers.0.self_attn.grep_a", "encoder.layers.1.self_attn.q_proj.weight", "encoder.layers.0.fc1.weight",
              "feature_extractor.conv_layers.0.0.weight"]


@pytest.mark.parametrize("pre_ln,relpos", [(False, True), (True, True), (True, False)])
def test_long_model_vs_oracle(cuda_device, pre_ln, relpos):
    """Tiny model, ragged B = 2 batch of 100 s and 70 s (T = 4999 and 3499): hidden states of every layer and the gradients
    of a fixed projection loss against the fp32 CPU oracle.  Without the bias (T = 5000) the forward stays on attn_fwd and
    the backward runs the long kernel without a table."""
    from unispeech_b200.wavlm import WavLM, WavLMConfig
    extra = {} if relpos else dict(relative_position_embedding=False, gru_rel_pos=False)
    cfg = O.tiny_config(pre_ln=pre_ln, **extra)
    m = WavLM(WavLMConfig(vars(cfg)))
    m.load_state_dict(O.deterministic_state_dict(cfg), strict=True)
    m = m.to(cuda_device).eval()
    lengths = [100 * SR, 70 * SR] if relpos else [5000 * 320 + 80, 3000 * 320]
    L = lengths[0]
    wav, pmask = O.deterministic_waveform(2, L, seed=4, lengths=lengths)
    x, fpm = m.extract_features(wav.to(cuda_device), padding_mask=pmask.to(cuda_device))
    T = x.shape[1]
    assert T == (4999 if relpos else 5000)
    loss = O.probe_loss(x.float(), fpm, seed=3)
    loss.backward()
    with torch.no_grad():
        (_, layer_results), _ = m.extract_features(wav.to(cuda_device), padding_mask=pmask.to(cuda_device),
                                                   ret_layer_results=True, output_layer=cfg.encoder_layers)
    torch.cuda.synchronize()

    sd = {k: v.clone().requires_grad_(True) for k, v in O.deterministic_state_dict(cfg).items()}
    want = O.extract_features(sd, wav, cfg, padding_mask=pmask)
    pad = want["padding_mask"]
    assert torch.equal(fpm.cpu(), pad)
    d = (x.detach().float().cpu() - want["x"].detach())[~pad].abs()
    assert d.max().item() < HID_TOL and d.mean().item() < 0.02, (d.max().item(), d.mean().item())
    with torch.no_grad():
        want_layers = O.extract_features(sd, wav, cfg, padding_mask=pmask, output_layer=cfg.encoder_layers)["layer_results"]
    assert len(layer_results) == len(want_layers) == cfg.encoder_layers + 1
    for i, (h, w) in enumerate(zip(layer_results, want_layers)):
        dh = (_hidden(h).float().cpu() - _hidden(w).detach())[~pad.t()].abs()
        assert dh.max().item() < HID_TOL and dh.mean().item() < 0.02, (i, dh.max().item(), dh.mean().item())
    O.probe_loss(want["x"], pad, seed=3).backward()
    params = dict(m.named_parameters())
    bad = []
    for k in GRAD_NAMES:
        if k not in sd or sd[k].grad is None:
            assert not relpos, k
            continue
        got, ref = params[k].grad.detach().double().cpu(), sd[k].grad.double()
        cos = ((got * ref).sum() / (got.norm() * ref.norm() + 1e-30)).item()
        # gate parameters: d gate_i = sum_j dS_ij tab[j - i] is a residual of sums that cancel (sum_j dS_ij = 0, and most of
        # the 5000 table entries are the saturated value), so its bf16 error grows with T while its value does not.  On
        # the B200, pre-LN, grep_a of layer 0 reaches cosine 1.0000 at 1499 frames and 0.984 at 4999 (norm -7 %); the
        # kernel-level d gate check at 5000 frames holds the tolerance of tests/test_kernels_gpu.py
        c_min, n_tol = (0.98, 0.08) if ("grep" in k and pre_ln) else (0.995, 0.06)
        if cos < c_min or abs(got.norm().item() - ref.norm().item()) > n_tol * ref.norm().item() + 2e-3:
            bad.append((k, cos, got.norm().item(), ref.norm().item()))
    assert not bad, bad


def test_large_long_batch_padding_invariance(cuda_device):
    """WavLM-Large widths, 24 layers, train mode at dropout 0: a 60 s utterance batched with a 5 min 27 s one (T = 16383, the
    long kernels) gives the same valid frames and parameter gradients as the utterance alone (T = 2999, the existing
    kernels)."""
    from unispeech_b200.wavlm import WavLM, WavLMConfig
    dev = cuda_device
    cfg = O.large_config()
    torch.manual_seed(17)
    m = WavLM(WavLMConfig(vars(cfg))).to(dev).train()
    n1, Llong = 60 * SR, 16383 * 320 + 80
    assert O.num_frames(Llong, cfg) == 16383 and O.num_frames(n1, cfg) == 2999
    g = torch.Generator().manual_seed(5)
    u0 = torch.nn.functional.layer_norm(torch.randn(Llong, generator=g), (Llong,))
    u1 = torch.nn.functional.layer_norm(torch.randn(n1, generator=g), (n1,))
    A = torch.zeros(2, Llong)
    A[0], A[1, :n1] = u0, u1
    pmA = torch.zeros(2, Llong, dtype=torch.bool)
    pmA[1, n1:] = True
    n_valid = 2999   # frames of the utterance alone (in the batch the frame mask keeps ceil(n1 / 320) = 3000)
    Rp = torch.randn(n_valid, cfg.encoder_embed_dim, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    names = ["encoder.layers.0.fc1.weight", "encoder.layers.23.self_attn.out_proj.weight",
             "encoder.layers.11.self_attn.q_proj.weight", "encoder.layers.0.self_attn.relative_attention_bias.weight",
             "encoder.layers.5.self_attn.grep_linear.weight", "encoder.pos_conv.0.weight_v", "post_extract_proj.weight",
             "feature_extractor.conv_layers.0.0.weight", "encoder.layer_norm.weight"]
    params = dict(m.named_parameters())

    def run(wav, pm, row):
        if m._engine is not None and m._engine.flat is not None:
            m.grad_buffer().zero_()
        torch.cuda.reset_peak_memory_stats()
        x, fpm = m.extract_features(wav.to(dev), padding_mask=None if pm is None else pm.to(dev))
        loss = (x[row, :n_valid].float() * Rp).sum()
        loss.backward()
        torch.cuda.synchronize()
        finite = bool(torch.isfinite(x[:, :]).all()) if pm is not None else True
        return (x[row, :n_valid].detach().float(), {k: params[k].grad.detach().double().clone() for k in names},
                torch.cuda.max_memory_allocated(), finite, x.shape[1])

    xa, ga, peak, finite, Ta = run(A, pmA, 1)
    xb, gb, _, _, Tb = run(u1[None], None, 0)
    assert (Ta, Tb) == (16383, 2999)
    assert finite    # the long utterance's outputs (and the padded rows) are finite
    d = (xa - xb).abs()
    scale = xa.abs().max().item()
    assert d.max().item() < 0.06 * max(1.0, scale) and d.mean().item() < 0.01, (d.max().item(), d.mean().item(), scale)
    bad = []
    for k in names:
        cos = ((ga[k] * gb[k]).sum() / (ga[k].norm() * gb[k].norm() + 1e-30)).item()
        rel = abs(ga[k].norm().item() - gb[k].norm().item()) / (gb[k].norm().item() + 1e-30)
        if cos < 0.995 or rel > 0.05:
            bad.append((k, round(cos, 5), round(rel, 4)))
    assert not bad, bad
    # memory is O(T): the reference materialises the [B*H, T, T] fp32 bias, 16 * 16383^2 * 4 bytes = 17.2 GB per utterance,
    # and keeps one such probability tensor per layer for its backward (24 x 34.4 GB for this batch).  Training here keeps
    # ~35 KB of activations per frame and layer; inference keeps none.
    assert peak < 2 * 34.4e9, peak
    torch.cuda.reset_peak_memory_stats()
    with torch.no_grad():
        x, _ = m.extract_features(A.to(dev), padding_mask=pmA.to(dev))
    torch.cuda.synchronize()
    assert torch.isfinite(x).all()
    assert torch.cuda.max_memory_allocated() < 17.2e9, torch.cuda.max_memory_allocated()
