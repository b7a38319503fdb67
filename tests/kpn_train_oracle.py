"""Float64 restatement of the backward of the KernelConv -> FAC block (models/Ours/model_singleframe.py:145-146,
159-162, class Modification), the reference for ebfi_kpn_fused_backward / KernelConvFACFunction:

    X = cat(Ev, Fr);  P = conv3x3(X, W, b, pad 1);  Kt = LeakyReLU(P);  Epad = ReplicationPad2d(R)(Ev)
    out[c, p] = sum_t Kt[c*KK + t, p] * Epad[c, p + t]

Given G = dL/dout:
    gP[c*KK + t, p] = G[c, p] * Epad[c, p + t] * (P > 0 ? 1 : slope)       (torch's leaky_relu_backward: P == 0 -> slope)
    gEpad[c, q]     = sum_t Kt[c*KK + t, q - t] * G[c, q - t], folded through the replication pad
    grad_bias = sum_{b,p} gP;  grad_W, grad_X = the 3x3 convolution's gradients of gP
    grad_event = gEpad folded + grad_X[:, :Ce];  grad_frame = grad_X[:, Ce:]

bf16_operands=True rounds the convolution's inputs and weights to bf16 for P only (what the fused kernel's
recompute feeds the tensor cores). grad_W and grad_X always use the unrounded fp32 values, as the fp32
convolution backward that KernelConvFACFunction runs on grad_pre does.
"""
import numpy as np

from oracle.oracle import _bf16_round


def _im2col3x3(feat):
    """(B, Cin, H, W) float64 -> (B, Cin*9, H*W), zero padding 1, column order (c, ky, kx) like a conv weight."""
    B, Cin, H, W = feat.shape
    fp = np.pad(feat, ((0, 0), (0, 0), (1, 1), (1, 1)))
    cols = np.empty((B, Cin * 9, H * W))
    for c in range(Cin):
        for i in range(3):
            for j in range(3):
                cols[:, c * 9 + i * 3 + j] = fp[:, c, i:i + H, j:j + W].reshape(B, -1)
    return cols


def _col2im3x3(cols, H, W):
    """Adjoint of _im2col3x3: (B, Cin*9, H*W) -> (B, Cin, H, W)."""
    B, n, _ = cols.shape
    Cin = n // 9
    gp = np.zeros((B, Cin, H + 2, W + 2))
    for c in range(Cin):
        for i in range(3):
            for j in range(3):
                gp[:, c, i:i + H, j:j + W] += cols[:, c * 9 + i * 3 + j].reshape(B, H, W)
    return gp[:, :, 1:H + 1, 1:W + 1]


def _fold_replication_pad(gpad, R):
    """Gradient of ReplicationPad2d(R): (B, C, H+2R, W+2R) -> (B, C, H, W)."""
    if R == 0:
        return gpad.copy()
    g = gpad[:, :, R:-R].copy()
    g[:, :, 0] += gpad[:, :, :R].sum(2)
    g[:, :, -1] += gpad[:, :, -R:].sum(2)
    out = g[:, :, :, R:-R].copy()
    out[:, :, :, 0] += g[:, :, :, :R].sum(3)
    out[:, :, :, -1] += g[:, :, :, -R:].sum(3)
    return out


def pre_activation(event_feat, frame_feat, conv_weight, conv_bias, bf16_operands=False):
    """P = conv3x3(cat(Ev, Fr), W) + b in float64, (B, Ce*K*K, H, W)."""
    feat = np.concatenate([np.asarray(event_feat, np.float32), np.asarray(frame_feat, np.float32)], axis=1)
    w = np.asarray(conv_weight, np.float32)
    if bf16_operands:
        feat, w = _bf16_round(feat), _bf16_round(w)
    feat, w = feat.astype(np.float64), w.astype(np.float64)
    B, Cin, H, W = feat.shape
    N = w.shape[0]
    P = np.matmul(w.reshape(N, Cin * 9), _im2col3x3(feat))
    P += np.asarray(conv_bias, np.float64)[None, :, None]
    return P.reshape(B, N, H, W)


def backward_parts(ev, fr, w, b, K, slope, grad_out, bf16_operands=False):
    """float64 (grad_event_fac, grad_x, grad_weight, grad_bias, grad_pre, P): grad_event_fac is the FAC +
    ReplicationPad part of dL/dEv (what ebfi_kpn_fused_backward writes), grad_x the convolution's input gradient."""
    P = pre_activation(ev, fr, w, b, bf16_operands)
    evd = np.asarray(ev, np.float64)
    G = np.asarray(grad_out, np.float64)
    B, Ce, H, W = evd.shape
    KK, R = K * K, (K - 1) // 2
    feat = np.concatenate([evd, np.asarray(fr, np.float64)], axis=1)
    Cin = feat.shape[1]
    wd = np.asarray(w, np.float64).reshape(Ce * KK, Cin * 9)
    evp = np.pad(evd, ((0, 0), (0, 0), (R, R), (R, R)), mode="edge")
    P5 = P.reshape(B, Ce, KK, H, W)
    Kt = np.where(P5 > 0, P5, P5 * slope)
    d = np.where(P5 > 0, 1.0, slope)
    gP = np.empty_like(P5)
    gpad = np.zeros((B, Ce, H + 2 * R, W + 2 * R))
    for t in range(KK):
        ky, kx = t // K, t % K
        gP[:, :, t] = G * evp[:, :, ky:ky + H, kx:kx + W] * d[:, :, t]
        gpad[:, :, ky:ky + H, kx:kx + W] += Kt[:, :, t] * G
    gP = gP.reshape(B, Ce * KK, H, W)
    gP2 = gP.reshape(B, Ce * KK, H * W)
    grad_weight = np.tensordot(gP2, _im2col3x3(feat), axes=([0, 2], [0, 2])).reshape(Ce * KK, Cin, 3, 3)
    grad_x = _col2im3x3(np.matmul(wd.T, gP2), H, W)
    return _fold_replication_pad(gpad, R), grad_x, grad_weight, gP.sum((0, 2, 3)), gP, P


def kpn_fused_backward(ev, fr, w, b, K, slope, grad_out, bf16_operands=False):
    """float64 (grad_event, grad_frame, grad_weight, grad_bias, grad_pre, P) of the block."""
    gev_fac, grad_x, grad_weight, grad_bias, gP, P = backward_parts(ev, fr, w, b, K, slope, grad_out, bf16_operands)
    Ce = gev_fac.shape[1]
    return gev_fac + grad_x[:, :Ce], grad_x[:, Ce:], grad_weight, grad_bias, gP, P
