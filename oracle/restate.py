"""ORACLE (test infrastructure; never imported by the product path).

CPU restatement of the reference's hot path, written from the formulas (SURVEY.md Appendix
A / B), independent of the reference's module graph.  It travels to the GPU box (where
/root/reference does not exist) and is the checker the ``-m gpu`` parity tests, ``smoke()``
and ``bench.py``'s cpu_baseline use.  It is itself pinned against results of the reference's own
code (tests/test_oracle.py), recorded in the committed fixtures in tests/golden/ by
tests/golden/make_golden.py.

PARITY STATUS: the reference repo holds no golden vectors / known-answer tests for this path
(SURVEY.md section 4), so the pin is "outputs of the reference itself run here".  Two
third-party pieces are absent from the image and restated (oracle/shims/): the asteroid STFT
filterbank (entering only as weight values W_a/W_s read from the state_dict) and the espnet2
TF-GridNet block of the enrollment net.  For those two the parity is "unpinned" at the
third-party boundary; everything defined under /root/reference is pinned.

Every function cites the reference lines it follows.  All tensors [B, T, F, C] unless noted.
"""
import math

import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------- helpers


def _ln(x, w, b, eps=1e-5):
    """nn.LayerNorm over the last dim: biased variance, eps inside the sqrt
    (tfgridnet_causal.py:594-620)."""
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def _prelu(x, a):
    return torch.where(x >= 0, x, a * x)


def _lstm_cell(gx, h, c, w_hh):
    """PyTorch LSTM cell, gate order i,f,g,o; gx already holds W_ih x + b_ih + b_hh."""
    g = gx + h @ w_hh.t()
    H = h.shape[-1]
    i, f, gg, o = g[..., :H], g[..., H:2 * H], g[..., 2 * H:3 * H], g[..., 3 * H:]
    c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
    h = torch.sigmoid(o) * torch.tanh(c)
    return h, c


_FAST = False


def set_fast(on):
    """Timing mode for bench.py's CPU baseline: run the LSTMs through ATen's fused CPU kernel
    (the same op nn.LSTM -- i.e. the reference -- dispatches to) instead of the explicit cell
    loop.  Parity checks keep the explicit loop; tests/test_oracle.py pins fast == explicit."""
    global _FAST
    _FAST = bool(on)


def _lstm_seq(x, w_ih, w_hh, b_ih, b_hh, h0=None, c0=None, reverse=False):
    """x [N, L, I] -> h [N, L, H]; returns (out, h_L, c_L)."""
    N, L, _ = x.shape
    H = w_hh.shape[1]
    if _FAST:
        h = x.new_zeros(1, N, H) if h0 is None else h0[None]
        c = x.new_zeros(1, N, H) if c0 is None else c0[None]
        xin = x.flip(1) if reverse else x
        out, hn, cn = torch._VF.lstm(xin.contiguous(), (h.contiguous(), c.contiguous()),
                                     [w_ih, w_hh, b_ih, b_hh], True, 1, 0.0, False, False, True)
        return (out.flip(1) if reverse else out), hn[0], cn[0]
    gx = x @ w_ih.t() + (b_ih + b_hh)
    h = x.new_zeros(N, H) if h0 is None else h0
    c = x.new_zeros(N, H) if c0 is None else c0
    out = x.new_empty(N, L, H)
    steps = range(L - 1, -1, -1) if reverse else range(L)
    for s in steps:
        h, c = _lstm_cell(gx[:, s], h, c, w_hh)
        out[:, s] = h
    return out, h, c


def cast_sd(sd, dtype):
    return {k: (v.detach().to(dtype) if v.is_floating_point() else v.detach()) for k, v in sd.items()}


# ----------------------------------------------------------------------------- separation


def sep_hparams(sd, prefix="tfgridnet."):
    """Derive the shape contract from the weights (configs/tsh.json:5-19)."""
    filt = sd[prefix + "enc.filterbank._filters"]
    n_fft = filt.shape[2]
    nF = filt.shape[0] // 2
    C = sd[prefix + "conv.0.weight"].shape[0]
    n_in = sd[prefix + "conv.0.weight"].shape[1]
    nblk = 0
    while (prefix + f"blocks.{nblk}.intra_norm.norm.weight") in sd:
        nblk += 1
    H = sd[prefix + "blocks.0.intra_rnn.weight_hh_l0"].shape[1]
    nqk = sd[prefix + "blocks.0.attn_conv_Q.0.weight"].shape[0]
    ln_q = sd[prefix + "blocks.0.attn_conv_Q.3.norm.weight"].shape[0]
    E = ln_q // nF
    n_head = nqk // E
    Vd = C // n_head
    n_out = sd[prefix + "deconv.weight"].shape[1]
    return dict(n_fft=n_fft, nF=nF, C=C, n_in=n_in, n_blocks=nblk, H=H, E=E, n_head=n_head,
                Vd=Vd, n_out=n_out, spk=sd[prefix + "embed_to_feats_proj.0.weight"].shape[1])


def sep_init_state(sd, B, L=50, hop=128, dtype=torch.float32, prefix="tfgridnet."):
    """Zero state, same keys/shapes as TFGridNet.init_buffers
    (tfgridnet_causal.py:173-186, 408-427)."""
    hp = sep_hparams(sd, prefix)
    z = lambda *s: torch.zeros(*s, dtype=dtype)
    bufs = {}
    for i in range(hp["n_blocks"]):
        bufs[f"buf{i}"] = dict(K_buf=z(B * hp["n_head"], L - 1, hp["E"] * hp["nF"]),
                               V_buf=z(B * hp["n_head"], L - 1, hp["Vd"] * hp["nF"]),
                               c0=z(1, B * hp["nF"], hp["H"]), h0=z(1, B * hp["nF"], hp["H"]))
    return dict(conv_buf=z(B, hp["n_in"], 2, hp["nF"]), deconv_buf=z(B, hp["C"], 2, hp["nF"]),
                istft_buf=z(B, hp["n_out"] // 2, 2 * hp["nF"], 1), gridnet_bufs=bufs)


def sep_block(sd, p, X, buf, hp, L, taps=None, tag=""):
    """One GridNetBlock (tfgridnet_causal.py:489-590) on X [B,T,F,C]; mutates buf."""
    B, T, nF, C = X.shape
    g = lambda k: sd[p + k]
    # intra: LN_C -> BiLSTM along F (zero init per frame) -> Linear(2H->C) -> +res   (:504-516)
    A = _ln(X, g("intra_norm.norm.weight"), g("intra_norm.norm.bias")).reshape(B * T, nF, C)
    yf, _, _ = _lstm_seq(A, g("intra_rnn.weight_ih_l0"), g("intra_rnn.weight_hh_l0"),
                         g("intra_rnn.bias_ih_l0"), g("intra_rnn.bias_hh_l0"))
    yb, _, _ = _lstm_seq(A, g("intra_rnn.weight_ih_l0_reverse"), g("intra_rnn.weight_hh_l0_reverse"),
                         g("intra_rnn.bias_ih_l0_reverse"), g("intra_rnn.bias_hh_l0_reverse"),
                         reverse=True)
    Y = torch.cat([yf, yb], dim=-1) @ g("intra_linear.weight").t() + g("intra_linear.bias")
    X1 = X + Y.reshape(B, T, nF, C)
    if taps is not None:
        taps[tag + "_intra"] = X1.clone()
    # inter: LN_C -> LSTM along T per (b,f) row with carried (h,c) -> Linear -> +res   (:518-538)
    Bn = _ln(X1, g("inter_norm.norm.weight"), g("inter_norm.norm.bias"))
    Bn = Bn.transpose(1, 2).reshape(B * nF, T, C)
    out, h, c = _lstm_seq(Bn, g("inter_rnn.weight_ih_l0"), g("inter_rnn.weight_hh_l0"),
                          g("inter_rnn.bias_ih_l0"), g("inter_rnn.bias_hh_l0"),
                          h0=buf["h0"][0], c0=buf["c0"][0])
    buf["h0"], buf["c0"] = h[None], c[None]
    Z = out @ g("inter_linear.weight").t() + g("inter_linear.bias")
    X2 = X1 + Z.reshape(B, nF, T, C).transpose(1, 2)
    if taps is not None:
        taps[tag + "_inter"] = X2.clone()
    # attention (:540-588, modules :351-396)
    nh, E, Vd = hp["n_head"], hp["E"], hp["Vd"]

    def proj(name, d):
        y = X2 @ g(f"{name}.0.weight").t() + g(f"{name}.0.bias")            # [B,T,F,nh*d]
        y = _prelu(y, g(f"{name}.1.weight"))
        y = y.reshape(B, T, nF, nh, d).permute(0, 3, 1, 2, 4).reshape(B * nh, T, nF * d)
        return _ln(y, g(f"{name}.3.norm.weight"), g(f"{name}.3.norm.bias"))

    q, k, v = proj("attn_conv_Q", E), proj("attn_conv_K", E), proj("attn_conv_V", Vd)
    Kall = torch.cat([buf["K_buf"], k], dim=1)            # [B*nh, L-1+T, F*E]
    Vall = torch.cat([buf["V_buf"], v], dim=1)
    buf["K_buf"], buf["V_buf"] = Kall[:, -(L - 1):].clone(), Vall[:, -(L - 1):].clone()
    scale = 1.0 / math.sqrt(nF * E)
    o = X.new_empty(B * nh, T, nF * Vd)
    for t in range(T):                                       # window = rows t .. t+L-1 (unmasked)
        s = torch.einsum("nd,njd->nj", q[:, t], Kall[:, t:t + L]) * scale
        a = torch.softmax(s, dim=-1)
        o[:, t] = torch.einsum("nj,njd->nd", a, Vall[:, t:t + L])
    # merge heads: channel = h*Vd + c   (:575-581)
    Zm = o.reshape(B, nh, T, nF, Vd).permute(0, 2, 3, 1, 4).reshape(B, T, nF, nh * Vd)
    P = _prelu(Zm @ g("attn_concat_proj.0.weight").t() + g("attn_concat_proj.0.bias"),
               g("attn_concat_proj.1.weight"))
    P = _ln(P.reshape(B, T, nF * C), g("attn_concat_proj.3.norm.weight"),
            g("attn_concat_proj.3.norm.bias")).reshape(B, T, nF, C)
    return X2 + P


def sep_core(sd, x, emb, state, L=50, hop=128, prefix="tfgridnet.", taps=None):
    """TFGridNet.forward (tfgridnet_causal.py:188-283): x [B,M,Np] (already padded),
    emb [B,256] -> y [B,S,hop*T + (n_fft-hop)]; mutates and returns state."""
    hp = sep_hparams(sd, prefix)
    g = lambda k: sd[prefix + k]
    B, M, Np = x.shape
    n_fft, nF, C = hp["n_fft"], hp["nF"], hp["C"]
    T = (Np - n_fft) // hop + 1
    Wa = g("enc.filterbank._filters")[:, 0]                           # [2F, n_fft]
    frames = x.unfold(-1, n_fft, hop)                                   # [B,M,T,n_fft]
    S = frames @ Wa.t()                                                 # [B,M,T,2F]      (:229)
    U = torch.cat([S[..., :nF], S[..., nF:]], dim=1)                    # [B,2M,T,F]      (:231-232)
    Up = torch.cat([state["conv_buf"], U], dim=2)                       # [B,2M,T+2,F]    (:239)
    state["conv_buf"] = Up[:, :, -2:].clone()
    Wc, bc = g("conv.0.weight"), g("conv.0.bias")
    if _FAST:
        X = F.conv2d(Up, Wc, bc, padding=(0, 1)).permute(0, 2, 3, 1)
    else:
        Upp = F.pad(Up, (1, 1))
        X = x.new_zeros(B, T, nF, C) + bc
        for i in range(3):
            for j in range(3):
                X = X + torch.einsum("bctf,oc->btfo", Upp[:, :, i:i + T, j:j + nF], Wc[:, :, i, j])
    gate = _ln(emb @ g("embed_to_feats_proj.0.weight").t() + g("embed_to_feats_proj.0.bias"),
               g("embed_to_feats_proj.1.weight"), g("embed_to_feats_proj.1.bias"))     # (:247)
    gate = gate.reshape(B, C, nF).transpose(1, 2)[:, None]              # [B,1,F,C]
    if taps is not None:
        taps["enc"] = X.clone()
        taps["gate"] = gate.clone()
    for b in range(hp["n_blocks"]):
        if b == 1:
            X = X * gate                                                # (:250-251)
        X = sep_block(sd, prefix + f"blocks.{b}.", X, state["gridnet_bufs"][f"buf{b}"], hp, L,
                      taps=taps, tag=f"block{b}")
        if taps is not None:
            taps[f"block{b}"] = X.clone()
    Xc = X.permute(0, 3, 1, 2)                                          # [B,C,T,F]
    Xp = torch.cat([state["deconv_buf"], Xc], dim=2)                    # (:256)
    state["deconv_buf"] = Xp[:, :, -2:].clone()
    Wd, bd = g("deconv.weight"), g("deconv.bias")                       # [C, 2S, 3, 3]
    nO = Wd.shape[1]
    if _FAST:
        D = F.conv_transpose2d(Xp, Wd, bd, padding=(2, 1))
    else:
        Xpp = F.pad(Xp, (1, 1))
        D = x.new_zeros(B, nO, T, nF) + bd[None, :, None, None]
        for i in range(3):                                              # D[o,t,f] += Wd[c,o,i,j] Xp[c,t+2-i,f+1-j]
            for j in range(3):
                D = D + torch.einsum("bctf,co->botf", Xpp[:, :, 2 - i:2 - i + T, 2 - j:2 - j + nF],
                                     Wd[:, :, i, j])
    R = D.reshape(B, nO // 2, 2, T, nF).permute(0, 1, 3, 2, 4).reshape(B, nO // 2, T, 2 * nF)  # (:260-266)
    Rp = torch.cat([state["istft_buf"].transpose(2, 3), R], dim=2)      # [B,S,T+1,2F]    (:269)
    state["istft_buf"] = Rp[:, :, -1:].transpose(2, 3).clone()
    Ws = g("dec.filterbank._filters")[:, 0]                             # [2F, n_fft]
    if _FAST:
        y = F.conv_transpose1d(Rp.reshape(-1, T + 1, 2 * nF).transpose(1, 2), g("dec.filterbank._filters"),
                               stride=hop).reshape(B, nO // 2, -1)
        return y[..., hop:], state
    w = Rp @ Ws                                                          # [B,S,T+1,n_fft]
    y = x.new_zeros(B, nO // 2, hop * T + n_fft)
    for t in range(T + 1):                                              # overlap-add      (:272)
        y[..., t * hop:t * hop + n_fft] += w[:, :, t]
    return y[..., hop:], state                                          # (:273)


def sep_predict(sd, x, emb, state, pad=True, hop=128, lookahead=64, L=50, taps=None):
    """Net.predict (net.py:54-66)."""
    mod = 0
    if pad:
        if x.shape[-1] % hop:
            mod = hop - x.shape[-1] % hop
        x = F.pad(x, (0, mod + lookahead))
    y, state = sep_core(sd, x, emb, state, L=L, hop=hop, taps=taps)
    y = y[..., :-lookahead]
    if mod:
        y = y[..., :-mod]
    return y, state


def sep_forward(sd, x, embeds, state=None, pad=True, taps=None):
    """Net.forward (net.py:68-76): x [B,2,N], embeds [B,1,256] -> [B,2,N]."""
    if state is None:
        state = sep_init_state(sd, x.shape[0], dtype=x.dtype)
    y, _ = sep_predict(sd, x, embeds[:, 0], state, pad=pad, taps=taps)
    return y


# ----------------------------------------------------------------------------- enrollment


def _ln_c(x, gamma, beta, eps=1e-5):
    """espnet2 LayerNormalization4D on [B,T,F,C] layout: stats over C."""
    return _ln(x, gamma.reshape(-1), beta.reshape(-1), eps)


def embed_block(sd, p, X, n_head=4, ks=4):
    """espnet2 GridNetBlock (non-causal; SURVEY.md Appendix B) on X [B,T,F,C]."""
    B, T, nF, C = X.shape
    g = lambda k: sd[p + k]

    def rnn_path(Xin, name, along_f):
        A = _ln_c(Xin, g(f"{name}_norm.gamma"), g(f"{name}_norm.beta"))
        if not along_f:
            A = A.transpose(1, 2)                                      # [B,F,T,C]
        N1, N2, Ls = A.shape[0], A.shape[1], A.shape[2]
        A = A.reshape(N1 * N2, Ls, C)
        # F.unfold with kernel (ks,1): feature index c*ks + k, step s covers bins s..s+ks-1
        win = A.unfold(1, ks, 1)                                       # [N, Ls-ks+1, C, ks]
        U = win.reshape(win.shape[0], win.shape[1], C * ks)
        r = f"{name}_rnn."
        yf, _, _ = _lstm_seq(U, g(r + "weight_ih_l0"), g(r + "weight_hh_l0"), g(r + "bias_ih_l0"),
                             g(r + "bias_hh_l0"))
        yb, _, _ = _lstm_seq(U, g(r + "weight_ih_l0_reverse"), g(r + "weight_hh_l0_reverse"),
                             g(r + "bias_ih_l0_reverse"), g(r + "bias_hh_l0_reverse"), reverse=True)
        Hc = torch.cat([yf, yb], dim=-1)                               # [N, S, 2H]
        Wt, bt = g(f"{name}_linear.weight"), g(f"{name}_linear.bias")  # [2H, C, ks]
        out = Xin.new_zeros(Hc.shape[0], Ls, C) + bt
        for k in range(ks):                                            # ConvTranspose1d stride 1
            out[:, k:k + Hc.shape[1]] += Hc @ Wt[:, :, k]
        out = out.reshape(N1, N2, Ls, C)
        if not along_f:
            out = out.transpose(1, 2)
        return Xin + out

    X1 = rnn_path(X, "intra", True)
    X2 = rnn_path(X1, "inter", False)
    heads = []
    for h in range(n_head):
        def pr(nm):
            W = g(f"attn_conv_{nm}_{h}.0.weight")[:, :, 0, 0]
            y = _prelu(X2 @ W.t() + g(f"attn_conv_{nm}_{h}.0.bias"), g(f"attn_conv_{nm}_{h}.1.weight"))
            gm = g(f"attn_conv_{nm}_{h}.2.gamma")[0, :, 0, :].t()      # [F, ch]
            bt = g(f"attn_conv_{nm}_{h}.2.beta")[0, :, 0, :].t()
            mu = y.mean(dim=(2, 3), keepdim=True)
            var = ((y - mu) ** 2).mean(dim=(2, 3), keepdim=True)
            return (y - mu) / torch.sqrt(var + 1e-5) * gm + bt          # [B,T,F,ch]
        q, k, v = pr("Q"), pr("K"), pr("V")
        d = q.shape[2] * q.shape[3]
        s = torch.einsum("btfe,bufe->btu", q, k) / math.sqrt(d)
        a = torch.softmax(s, dim=-1)
        heads.append(torch.einsum("btu,bufc->btfc", a, v))
    Z = torch.cat(heads, dim=-1)                                        # channel = h*Vd + c
    W = g("attn_concat_proj.0.weight")[:, :, 0, 0]
    P = _prelu(Z @ W.t() + g("attn_concat_proj.0.bias"), g("attn_concat_proj.1.weight"))
    gm = g("attn_concat_proj.2.gamma")[0, :, 0, :].t()
    bt = g("attn_concat_proj.2.beta")[0, :, 0, :].t()
    mu = P.mean(dim=(2, 3), keepdim=True)
    var = ((P - mu) ** 2).mean(dim=(2, 3), keepdim=True)
    P = (P - mu) / torch.sqrt(var + 1e-5) * gm + bt
    return X2 + P


def embed_forward(sd, x, n_fft=128, hop=64, taps=None):
    """EmbedTFGridNet.forward (tfgridnet_orig/tfgridnet.py:100-127): x [B,M,N] -> [B,256]."""
    B, M, N = x.shape
    std = x.reshape(B, -1).std(dim=1, unbiased=True)                     # (:109-110)
    xn = x / std[:, None, None]
    win = torch.hann_window(n_fft, periodic=True, dtype=x.dtype)
    xp = F.pad(xn.reshape(B * M, 1, N), (n_fft // 2, n_fft // 2), mode="reflect")[:, 0]
    fr = xp.unfold(-1, n_fft, hop) * win                                # [B*M,T,n_fft]
    n = torch.arange(n_fft, dtype=x.dtype)
    kk = torch.arange(n_fft // 2 + 1, dtype=x.dtype)
    ang = 2 * math.pi * kk[:, None] * n[None, :] / n_fft
    re = fr @ torch.cos(ang).t()
    im = -(fr @ torch.sin(ang).t())
    T, nF = re.shape[1], re.shape[2]
    re, im = re.reshape(B, M, T, nF), im.reshape(B, M, T, nF)
    U = torch.cat([re, im], dim=1)                                       # [B,2M,T,F]   (:113-114)
    Wc, bc = sd["conv.0.weight"], sd["conv.0.bias"]
    X = F.conv2d(U, Wc, bc, padding=(1, 1))                              # [B,C,T,F]
    mu = X.mean(dim=(1, 2, 3), keepdim=True)                             # GroupNorm(1, C)
    var = ((X - mu) ** 2).mean(dim=(1, 2, 3), keepdim=True)
    X = (X - mu) / torch.sqrt(var + 1e-5) * sd["conv.1.weight"][None, :, None, None] \
        + sd["conv.1.bias"][None, :, None, None]
    X = X.permute(0, 2, 3, 1).contiguous()                               # [B,T,F,C]
    if taps is not None:
        taps["enc"] = X.clone()
    nb = 0
    while f"blocks.{nb}.intra_norm.gamma" in sd:
        nb += 1
    for b in range(nb):
        X = embed_block(sd, f"blocks.{b}.", X)
        if taps is not None:
            taps[f"block{b}"] = X.clone()
    feat = X.permute(0, 1, 3, 2).reshape(B, T, -1)                       # index c*F + f  (:122-123)
    y = feat @ sd["embed_proj.0.weight"].t() + sd["embed_proj.0.bias"]
    y = _ln(y, sd["embed_proj.1.weight"], sd["embed_proj.1.bias"])
    return y.mean(dim=1)                                                 # (:125)


# ----------------------------------------------------------------------------- metrics


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def si_sdr(pred, target):
    """Scale-invariant SNR as torchmetrics computes it (zero-mean; ts_hear_test.py:144-146)."""
    eps = torch.finfo(torch.float32).eps
    p = pred.double() - pred.double().mean(dim=-1, keepdim=True)
    t = target.double() - target.double().mean(dim=-1, keepdim=True)
    alpha = ((p * t).sum(-1, keepdim=True) + eps) / ((t * t).sum(-1, keepdim=True) + eps)
    ts = alpha * t
    noise = ts - p
    return 10 * torch.log10(((ts * ts).sum(-1) + eps) / ((noise * noise).sum(-1) + eps))
