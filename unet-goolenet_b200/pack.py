"""Weight preparation for the engine: eval-mode BatchNorm folding (fp32) and bf16 K-major GEMM packing.

BN fold (SURVEY Appendix B): scale = gamma / sqrt(var + eps); bias' = beta + (b_conv - mean) * scale.
Packed conv weight: [Npad][R*S*Cin_pad] bf16, K index = (r*S + s)*Cin_pad + c (see ug_conv_desc).
"""
import torch


def round_up(x, m):
    return (x + m - 1) // m * m


def choose_bn(n_out, convt_cout=None, r=1):
    """N-tile of the implicit-GEMM kernel (multiple of 16).  3x3 layers whose output width is a multiple of
    256 use BN=256 (persistent kernel; halves the activation-tile traffic per FLOP), otherwise 128."""
    if convt_cout is not None:
        return min(128, convt_cout)
    if r == 3 and n_out % 256 == 0:
        return 256
    if r == 1 and n_out >= 1024 and n_out % 256 == 0:
        return 256        # wide linear layers (qkv, FFN): persistent kernel with 256-wide n-tiles (measured)
    if n_out <= 128:
        return round_up(n_out, 16)
    if n_out % 128 == 0 or r != 1:
        # 3x3 layers keep 128-wide n-tiles: one fitted tile of 144 ... 240 columns (supported by the kernel, see
        # ug_conv_desc.BN) measured slower (GoogLeNet stage 2.358 -> 2.400 ms: one accumulator per issuer and a 3-4
        # slot weight ring)
        return 128
    # 1x1 layers whose width is not a multiple of 128 (GoogLeNet: 136 ... 240): pick the tile width that minimises
    # n_tiles * (MMA issue interval of an M=128 x BN MMA); the single-issuer GEMM kernels issue one MMA per ~110 cycles
    # up to N = 220, then N/2 (profiles/r01_mma_*.txt), BN <= 256.  Ties go to the least padding.
    best, best_key = 128, None
    for bn in range(16, 256 + 1, 16):
        tiles = -(-n_out // bn)
        cyc = max(110.0, 0.5 * bn)
        key = (tiles * cyc, tiles * bn - n_out)
        if best_key is None or key < best_key:
            best, best_key = bn, key
    return best


def fold_bn(conv_bias, gamma, beta, mean, var, eps):
    scale = gamma.double() / torch.sqrt(var.double() + eps)
    b = conv_bias.double() if conv_bias is not None else torch.zeros_like(mean, dtype=torch.float64)
    bias = beta.double() + (b - mean.double()) * scale
    return scale.float().contiguous(), bias.float().contiguous()


def pack_conv_weight(w, bn):
    """w: [Cout, Cin, R, S] (fp32) -> bf16 [round_up(Cout, bn)][R*S*round_up(Cin, 64)]."""
    cout, cin, r, s = w.shape
    cin_pad = round_up(cin, 64)
    npad = round_up(cout, bn)
    out = torch.zeros(npad, r, s, cin_pad, dtype=torch.float32, device=w.device)
    out[:cout, :, :, :cin] = w.permute(0, 2, 3, 1).float()
    return out.reshape(npad, r * s * cin_pad).to(torch.bfloat16).contiguous()


def pack_linear_weight(w, bn):
    """w: [out, in] -> bf16 [round_up(out, bn)][round_up(in, 64)]."""
    return pack_conv_weight(w[:, :, None, None], bn)


def pack_convt_weight(w, bias, bn):
    """ConvTranspose2d(k=2, s=2) weight [Cin, Cout, 2, 2] -> GEMM weight with N = 4*Cout ordered (kh, kw, co),
    plus the bias replicated for the four taps."""
    cin, cout, kh, kw = w.shape
    assert kh == 2 and kw == 2
    g = w.permute(2, 3, 1, 0).reshape(4 * cout, cin)  # row (kh*2+kw)*cout + co, col ci
    return pack_linear_weight(g, bn), bias.float().repeat(4).contiguous()


def pack_conv1_s2d(w):
    """torchvision GoogLeNet conv1 weight [64, 3, 7, 7] (stride 2, pad 3) -> the GEMM weight of its space-to-depth form
    (ug_s2d_desc): bf16 [64][4*64], K index = r2*64 + s2*16 + (dy*2+dx)*3 + c = w[:, c, 2*r2+dy, 2*s2+dx] (zero where the
    7x7 filter has no tap 7 and in the padding channels 12..15)."""
    assert tuple(w.shape[1:]) == (3, 7, 7)
    cout = w.shape[0]
    w8 = torch.zeros(cout, 3, 8, 8, dtype=torch.float32, device=w.device)
    w8[:, :, :7, :7] = w.float()
    g = w8.reshape(cout, 3, 4, 2, 4, 2).permute(0, 2, 4, 3, 5, 1).reshape(cout, 4, 4, 12)   # [co, r2, s2, (dy,dx,c)]
    out = torch.zeros(cout, 4, 4, 16, dtype=torch.float32, device=w.device)
    out[..., :12] = g
    return out.reshape(cout, 256).to(torch.bfloat16).contiguous()
