"""
Weight packing for the tensor-core conv kernels (csrc/conv_kernels.cu).

Every GEMM-shaped layer consumes its weights as the tcgen05 B operand in the SWIZZLE_NONE K-major
canonical layout:  packed[k // 8][n][k % 8]  (bf16), i.e. for each group of 8 consecutive K indices
a contiguous (N x 8) slab.  The K order of each layer matches the order in which the kernel's tap
table walks the shared-memory input tile; channel counts are zero-padded to multiples of 8 (K) and
to at least 16 (N).  Shapes on the left are the reference's state_dict shapes (SURVEY.md A.4).

The C8 planar activation layout is (B, ceil(C/8), H, T, 8) bf16.
"""

import torch

__all__ = ['pack_down_pairs', 'pack_res_rs', 'pack_res_rs_pairs', 'pack_res_rs_fold', 'to_p4', 'from_p4', 'pack_down_strip', 'pack_up_strip', 'pad8', 'to_c8', 'from_c8', 'pack_res3x3', 'pack_res1x1', 'pack_down', 'pack_up', 'pack_lat', 'pack_deconv_in', 'pack_deconv_in_film',
           'pad_vec']


class _PackedCache:
    """Packed (kernel-layout) copies of a module's parameters, rebuilt when a parameter is modified or moved."""

    epoch = 0       # bumped by code that updates parameters outside torch's version counter (framework/train.py's AdamW kernel)

    def __init__(self):
        self._key = None
        self._val = None

    def __getstate__(self):
        # pickling / deep-copying a module (the reference checkpoints whole modules, experiments/train.py:511) drops the packed
        # copies: they are rebuilt lazily from the parameters of the new object
        return dict(_key=None, _val=None)

    def get(self, params, build):
        key = (_PackedCache.epoch,) + tuple((p.data_ptr(), p._version, p.device) for p in params)
        if key != self._key:
            with torch.no_grad():
                self._val = build()
            self._key = key
        return self._val


def pad8(c):
    return (c + 7) // 8 * 8


def to_c8(x):
    """(B, C, H, T) -> (B, ceil(C/8), H, T, 8) bf16, zero-padded channels (test/plumbing helper)."""
    B, C, H, T = x.shape
    Cp = pad8(C)
    if Cp != C:
        x = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, Cp - C))
    return x.reshape(B, Cp // 8, 8, H, T).permute(0, 1, 3, 4, 2).contiguous().to(torch.bfloat16)


def from_c8(y, C):
    """(B, CG, H, T, 8) -> (B, C, H, T) fp32."""
    B, CG, H, T, _ = y.shape
    return y.permute(0, 1, 4, 2, 3).reshape(B, CG * 8, H, T)[:, :C].float()


def pad_vec(b, n):
    out = torch.zeros(n, dtype=torch.float32, device=b.device)
    out[:b.numel()] = b.detach().float()
    return out


def _to_b_operand(w_nk):
    """(N, K) fp32 with K % 8 == 0 -> packed (K/8, N, 8) bf16."""
    N, K = w_nk.shape
    return w_nk.reshape(N, K // 8, 8).permute(1, 0, 2).contiguous().to(torch.bfloat16)


def pack_res3x3(w):
    """conv1.0.weight (C, C, 3, 3) -> K order (tap = ky*3+kx, ci); C = 8 gets a 10th all-zero K group (MMA K = 16)."""
    Co, Ci = w.shape[:2]
    Cp = pad8(Ci)
    N = max(16, pad8(Co))
    k = torch.zeros((N, 9, Cp), dtype=torch.float32, device=w.device)
    k[:Co, :, :Ci] = w.detach().float().permute(0, 2, 3, 1).reshape(Co, 9, Ci)
    k = k.reshape(N, 9 * Cp)
    if Cp == 8:
        k = torch.nn.functional.pad(k, (0, 8))
    return _to_b_operand(k)


def pack_res1x1(w):
    """conv2.0.weight (C, C, 1, 1) -> K = ci, padded to at least 16."""
    Co, Ci = w.shape[:2]
    K = max(16, pad8(Ci))
    N = max(16, pad8(Co))
    k = torch.zeros((N, K), dtype=torch.float32, device=w.device)
    k[:Co, :Ci] = w.detach().float().reshape(Co, Ci)
    return _to_b_operand(k)


def pack_down(w):
    """sconv.0.weight (Cout, Cin, 4, 1) -> K order (kh, ci)."""
    Co, Ci = w.shape[:2]
    Cp = pad8(Ci)
    N = max(16, pad8(Co))
    k = torch.zeros((N, 4, Cp), dtype=torch.float32, device=w.device)
    k[:Co, :, :Ci] = w.detach().float()[..., 0].permute(0, 2, 1)
    return _to_b_operand(k.reshape(N, 4 * Cp))


def pack_up(w):
    """
    tconv.0.weight (Cin, Cout, 4, 1) -> polyphase GEMM: N = (r, co) with r the output-row parity, K = (a, ci) with
    a = 0 the input row q-1 (kernel tap r+2) and a = 1 the input row q (kernel tap r).
    """
    Ci, Co = w.shape[:2]
    Cip, Cop = pad8(Ci), pad8(Co)
    N = max(16, 2 * Cop)
    k = torch.zeros((N, 2, Cip), dtype=torch.float32, device=w.device)
    wf = w.detach().float()[..., 0]                      # (Ci, Co, 4)
    for r in range(2):
        k[r * Cop: r * Cop + Co, 0, :Ci] = wf[:, :, r + 2].t()
        k[r * Cop: r * Cop + Co, 1, :Ci] = wf[:, :, r].t()
    return _to_b_operand(k.reshape(N, 2 * Cip))


def pack_up_bias(b, Co):
    Cop = pad8(Co)
    out = torch.zeros(max(16, 2 * Cop), dtype=torch.float32, device=b.device)
    out[:Co] = b.detach().float()
    out[Cop:Cop + Co] = b.detach().float()
    return out


def pack_lat(w, latent_pad):
    """convlat.weight (D, C4, H4, 1) -> K order (kh, ci), N = D padded to latent_pad."""
    D, C4, H4 = w.shape[:3]
    Cp = pad8(C4)
    k = torch.zeros((latent_pad, H4, Cp), dtype=torch.float32, device=w.device)
    k[:D, :, :C4] = w.detach().float()[..., 0].permute(0, 2, 1)
    return _to_b_operand(k.reshape(latent_pad, H4 * Cp))


def pack_deconv_in(w, b, latent_pad):
    """
    decoder.convin.0.weight (D+1, C0, H0, 1), bias (C0) -> per output row h a (C0 x D) B operand, packed
    (H0, latent_pad/8, C0, 8); plus the two per-row bias tables (H0, C0): index 0 = transcribe (indicator 0),
    1 = reconstruct (indicator 1: the last input channel's weights are added to the bias).
    """
    D1, C0, H0 = w.shape[:3]
    D = D1 - 1
    N = max(16, pad8(C0))
    wf = w.detach().float()[..., 0]                      # (D+1, C0, H0)
    k = torch.zeros((H0, N, latent_pad), dtype=torch.float32, device=w.device)
    k[:, :C0, :D] = wf[:D].permute(2, 1, 0)
    packed = k.reshape(H0, N, latent_pad // 8, 8).permute(0, 2, 1, 3).contiguous().to(torch.bfloat16)
    bias = torch.zeros((2, H0, N), dtype=torch.float32, device=w.device)
    bias[0, :, :C0] = b.detach().float()[None, :]
    bias[1, :, :C0] = b.detach().float()[None, :] + wf[D].t()
    return packed, bias


def pack_deconv_in_film(w, b, gamma, beta, latent_pad):
    """
    decoder.convin of TimbreTrapFiLM (reference modules.py:801-809: ConvTranspose2d(D, C0, (H0, 1)), no indicator channel) with the
    FiLM layer in front of it (modules.py:838-840: latents * gamma + beta per channel) FOLDED IN - the layer is linear in its input:
        convin(gamma * z + beta) = (W scaled by gamma along its input channels) z  +  (bias + sum_d beta_d W[d])
    w (D, C0, H0, 1), b (C0), gamma / beta (D) -> packed (H0, latent_pad/8, C0, 8) bf16 and the per-row bias table (H0, C0).
    """
    D, C0, H0 = w.shape[:3]
    N = max(16, pad8(C0))
    wf = w.detach().float()[..., 0]                      # (D, C0, H0)
    k = torch.zeros((H0, N, latent_pad), dtype=torch.float32, device=w.device)
    k[:, :C0, :D] = (wf * gamma.detach().float().view(-1, 1, 1)).permute(2, 1, 0)
    packed = k.reshape(H0, N, latent_pad // 8, 8).permute(0, 2, 1, 3).contiguous().to(torch.bfloat16)
    bias = torch.zeros((H0, N), dtype=torch.float32, device=w.device)
    bias[:, :C0] = b.detach().float()[None, :] + torch.einsum('d,dch->hc', beta.detach().float(), wf)
    return packed, bias


def _bias_group(b, N):
    """(N, 8) K group that, against the kernel's constant (1, 1, 0, ..., 0) operand, adds b as bf16 hi + lo (fp32-accurate)."""
    g = torch.zeros((N, 8), dtype=torch.float32, device=b.device)
    bf = b.detach().float()
    hi = bf.to(torch.bfloat16).float()
    g[:bf.numel(), 0] = hi
    g[:bf.numel(), 1] = bf - hi
    return g


def _rows_to_groups(rows_nc, bias_group, N):
    """rows_nc: list over input rows of (N, Cin_pad) weight slabs -> packed (KG, N, 8) for csrc/updown_strip.cu."""
    Cp = rows_nc[0].shape[1]
    CG = Cp // 8
    zero = torch.zeros((N, 8), dtype=torch.float32, device=rows_nc[0].device)
    groups = []
    if CG == 1:
        for k, r in enumerate(rows_nc):
            groups += [r, bias_group if k == 0 else zero]
    else:
        for r in rows_nc:
            groups += [r[:, 8 * g: 8 * g + 8] for g in range(CG)]
        groups += [bias_group, zero]
    return torch.stack(groups, dim=0).contiguous().to(torch.bfloat16)


def pack_down_strip(w, b):
    """sconv.0.weight (Cout, Cin, 4, 1), bias -> K groups (kh, channel group) [+ bias group], N = max(16, Cout padded)."""
    Co, Ci = w.shape[:2]
    Cp, N = pad8(Ci), max(16, pad8(Co))
    rows = []
    for kh in range(4):
        r = torch.zeros((N, Cp), dtype=torch.float32, device=w.device)
        r[:Co, :Ci] = w.detach().float()[:, :, kh, 0]
        rows.append(r)
    return _rows_to_groups(rows, _bias_group(b, N), N)


def pack_up_strip(w, b):
    """tconv.0.weight (Cin, Cout, 4, 1), bias -> polyphase N = (r, co); K rows: input row q-1 (taps r+2), then row q (taps r)."""
    Ci, Co = w.shape[:2]
    Cip, Cop = pad8(Ci), pad8(Co)
    N = max(16, 2 * Cop)
    wf = w.detach().float()[..., 0]                      # (Ci, Co, 4)
    rows = []
    for a in range(2):
        r = torch.zeros((N, Cip), dtype=torch.float32, device=w.device)
        for par in range(2):
            r[par * Cop: par * Cop + Co, :Ci] = wf[:, :, par + 2 - 2 * a].t()
        rows.append(r)
    bias2 = torch.zeros(N, dtype=torch.float32, device=w.device)
    bias2[:Co] = b.detach().float()
    bias2[Cop:Cop + Co] = b.detach().float()
    return _rows_to_groups(rows, _bias_group(bias2, N), N)


# ---- packed 4-channel layout (first encoder / last decoder stage): memory (B, H, T, 4) bf16 ----------------------------

def to_p4(x):
    """(B, C <= 4, H, T) -> (B, H, T, 4) bf16, zero-padded channels (test/plumbing helper)."""
    B, C, H, T = x.shape
    if C < 4:
        x = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, 4 - C))
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def from_p4(y, C):
    return y.permute(0, 3, 1, 2)[:, :C].float()


def pack_res_rs(w1, b1, w2, b2):
    """
    Weights of one ResidualConv2dBlock for csrc/res_rs.cu (row-stationary: an input row meets all three vertical taps at once).
    W1 -> (KG1, 3 NC, 8): B rows n = j * NC + co with j = 0, 1, 2 <-> output rows r-d, r, r+d, i.e. vertical taps ky = 2, 1, 0;
      C <= 8 : K groups kx = 0, 1, 2 (8 input channels each), then a zero group so that groups pair up into K = 16 MMAs;
      C >= 16: K groups (kx, channel group), kx-major.
    W2 -> (KG2, NC, 8): channel groups (C <= 8: plus a zero group).  bias -> (2, NC) fp32: the accumulators' initial values.
    NC = 16 for C <= 16, 32 for C = 32.
    """
    Co, Ci = w1.shape[:2]
    Cp = pad8(Ci)
    CG = Cp // 8
    NC = 32 if Cp >= 32 else 16
    dev = w1.device
    w = w1.detach().float()
    taps = torch.zeros((3, 3, NC, Cp), dtype=torch.float32, device=dev)           # [j][kx][co][ci]
    for j in range(3):
        taps[j, :, :Co, :Ci] = w[:, :, 2 - j, :].permute(2, 0, 1)
    groups = [taps[:, kx, :, 8 * g: 8 * g + 8].reshape(3 * NC, 8) for kx in range(3) for g in range(CG)]
    if CG == 1:
        groups.append(torch.zeros((3 * NC, 8), dtype=torch.float32, device=dev))
    w1p = torch.stack(groups, dim=0).contiguous().to(torch.bfloat16)
    k2 = torch.zeros((NC, Cp), dtype=torch.float32, device=dev)
    k2[:Co, :Ci] = w2.detach().float().reshape(Co, Ci)
    groups2 = [k2[:, 8 * g: 8 * g + 8] for g in range(CG)]
    if CG == 1:
        groups2.append(torch.zeros((NC, 8), dtype=torch.float32, device=dev))
    w2p = torch.stack(groups2, dim=0).contiguous().to(torch.bfloat16)
    bias = torch.zeros((2, NC), dtype=torch.float32, device=dev)
    bias[0, :Co] = b1.detach().float()
    bias[1, :Co] = b2.detach().float()
    return w1p, w2p, bias


def pack_res_rs_pairs(w1, b1, w2, b2, dilation):
    """
    pack_res_rs for the packed 4-channel layout (C <= 4): a GEMM row is a PAIR of frames, a K group is (frame parity e_in, 4
    channels) of the input pair at offset o in [-hp, hp], hp = ceil((d+1)/2) (the 3x3 kernel is Toeplitz-expanded over the pair); accumulator column
    = (e_out, co).  K groups: o = -hp..hp, then a zero group.
    """
    Co, Ci = w1.shape[:2]
    assert Co <= 4 and Ci <= 4
    d = int(dilation)
    hp = (d + 1) // 2
    NC = 16
    dev = w1.device
    w = w1.detach().float()
    groups = []
    for o in range(-hp, hp + 1):
        g = torch.zeros((3, NC, 8), dtype=torch.float32, device=dev)
        for j in range(3):
            for e_out in range(2):
                for e_in in range(2):
                    s_ = 2 * o + e_in - e_out
                    for kx in range(3):
                        if (kx - 1) * d == s_:
                            g[j, 4 * e_out: 4 * e_out + Co, 4 * e_in: 4 * e_in + Ci] = w[:, :, 2 - j, kx]
        groups.append(g.reshape(3 * NC, 8))
    groups.append(torch.zeros((3 * NC, 8), dtype=torch.float32, device=dev))
    w1p = torch.stack(groups, dim=0).contiguous().to(torch.bfloat16)
    g2 = torch.zeros((NC, 8), dtype=torch.float32, device=dev)
    bias = torch.zeros((2, NC), dtype=torch.float32, device=dev)
    for e in range(2):
        g2[4 * e: 4 * e + Co, 4 * e: 4 * e + Ci] = w2.detach().float().reshape(Co, Ci)
        bias[0, 4 * e: 4 * e + Co] = b1.detach().float()
        bias[1, 4 * e: 4 * e + Co] = b2.detach().float()
    w2p = torch.stack([g2, torch.zeros_like(g2)], dim=0).contiguous().to(torch.bfloat16)
    return w1p, w2p, bias


def res_rs_fold_mmas(dilation, fold):
    """The MMAs of one folded input row (csrc/res_rs.cu, RsPlan::fold_s / fold_adj): (s, adj) = first half of GEMM row i + s and second
    half of row i + s - adj."""
    d = int(dilation)
    if (fold == 4 and d <= 2) or (fold == 2 and d == 1):
        return [(0, 1), (1, 1)]
    if fold == 2 and d == 3:
        return [(-1, 1), (0, 0), (2, 1)]
    return [(-1, 0), (0, 0), (1, 0)]


def pack_res_rs_fold(w1, b1, w2, b2, dilation, fold):
    """
    pack_res_rs for FOLDED rows (csrc/res_rs.cu layouts 2 and 4): a GEMM row is `fold` consecutive frames x Cw = 16 / fold
    channels (fold = 2: C <= 8 in C8 planar; fold = 4: C <= 4 in the packed layout), i.e. always 16 values = two K groups
    (halves).  The 3x3 kernel is Toeplitz-expanded over the frames of a row: a K group holding input frame f_in (relative to the
    first frame of the output row) meets output frame e_out through the horizontal tap kx with (kx - 1) * d = f_in - e_out.  Which
    halves of which neighbouring rows form the K = 16 of one MMA is `res_rs_fold_mmas` (only the halves some tap touches are read).
    W1 -> (2 n_mma, 48, 8): K groups (mma, half); rows n = j * 16 + e_out * Cw + co with j <-> vertical tap ky = 2 - j.
    W2 -> (2, 16, 8) block-diagonal over the frames; bias -> (2, 16).
    """
    Co, Ci = w1.shape[:2]
    Cw = 16 // fold
    assert fold in (2, 4) and Co <= Cw and Ci <= Cw
    d = int(dilation)
    dev = w1.device
    w = w1.detach().float()
    per_half = fold // 2                                       # frames per 16-byte half
    assert per_half * Cw == 8
    groups, seen = [], set()
    for s_row, adj in res_rs_fold_mmas(d, fold):
        for half in range(2):
            first = fold * (s_row - adj * half) + per_half * half          # input frame of the half's first value
            g = torch.zeros((3, 16, 8), dtype=torch.float32, device=dev)   # [j][n][k within the half]
            for e_in in range(per_half):
                f_in = first + e_in
                assert f_in not in seen
                seen.add(f_in)
                for e_out in range(fold):
                    for kx in range(3):
                        if (kx - 1) * d == f_in - e_out:
                            for j in range(3):
                                g[j, e_out * Cw: e_out * Cw + Co, e_in * Cw: e_in * Cw + Ci] = w[:, :, 2 - j, kx]
            groups.append(g.reshape(48, 8))
    assert all(e_out + (kx - 1) * d in seen for e_out in range(fold) for kx in range(3))
    w1p = torch.stack(groups, dim=0).contiguous().to(torch.bfloat16)
    g2 = torch.zeros((16, 16), dtype=torch.float32, device=dev)
    bias = torch.zeros((2, 16), dtype=torch.float32, device=dev)
    for e in range(fold):
        g2[e * Cw: e * Cw + Co, e * Cw: e * Cw + Ci] = w2.detach().float().reshape(Co, Ci)
        bias[0, e * Cw: e * Cw + Co] = b1.detach().float()
        bias[1, e * Cw: e * Cw + Co] = b2.detach().float()
    w2p = torch.stack([g2[:, :8], g2[:, 8:]], dim=0).contiguous().to(torch.bfloat16)
    return w1p, w2p, bias


def pack_down_pairs(w, b):
    """
    sconv.0.weight (Cout <= 8, Cin <= 4, 4, 1) for a packed 4-channel INPUT: GEMM row = frame pair, K group of tap row kh =
    (e_in, ci), N = (e_out, co) = 16, block-diagonal in the frame parity; each tap row pairs with the ones operand (bias for kh = 0).
    """
    Co, Ci = w.shape[:2]
    assert Co <= 8 and Ci <= 4
    N = 16
    dev = w.device
    wf = w.detach().float()[..., 0]                      # (Co, Ci, 4)
    zero = torch.zeros((N, 8), dtype=torch.float32, device=dev)
    bias = torch.zeros(N, dtype=torch.float32, device=dev)
    for e in range(2):
        bias[8 * e: 8 * e + Co] = b.detach().float()
    groups = []
    for kh in range(4):
        g = torch.zeros((N, 8), dtype=torch.float32, device=dev)
        for e in range(2):
            g[8 * e: 8 * e + Co, 4 * e: 4 * e + Ci] = wf[:, :, kh]
        groups += [g, _bias_group(bias, N) if kh == 0 else zero]
    return torch.stack(groups, dim=0).contiguous().to(torch.bfloat16)
