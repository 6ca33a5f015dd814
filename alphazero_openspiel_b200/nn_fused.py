"""FusedEvaluator: the reference ResNet (network.py:21-104) on the hand-written sm_100a kernels of csrc/az_resnet.cu.

Same contract as network.BatchedEvaluator -- obs bf16 [B,H,W,4] (written by az_step) -> priors fp32 [B,A], values
fp32 [B] -- but the ten 3x3 convolutions run as tcgen05 implicit GEMMs with BatchNorm / LeakyReLU / bias / residual
fused into their epilogues (11 launches instead of ~45 PyTorch kernels), on NHWC bf16 activations [B,H+1,W,64] (row H
of every board is a zero pad row)
(see az_resnet.cu).  Host code here only folds/packs weights and sequences the launches.  The FC head is the streaming
k_head kernel (FC + softmax + tanh in one launch, fp32 logits) when A + 1 <= 8 (Connect Four) and the tcgen05 GEMM head
k_head_mma (same fusion, N = A + 1 = 433 / 769 columns) for the larger action spaces of Breakthrough.

Per evaluation:   stem(obs) -> U (channels 50-53: the raw planes)
                  X = conv(U) [+ conv1x1(obs) through those channels], T = lrelu(bn1_2(X))      (block 1, conv2)
                  for k = 2..5:  U = lrelu(conv(T) + b)  ;  X = conv(U) + X, T = lrelu(bn1_{k+1}(X))
                  head: softmax / tanh (X_flat @ Wfc + b)
"""
import ctypes as C
import os

import torch
from torch.nn import functional as F

from . import _lib as L
from .network import N_FILTERS, _fold_bn

CH = 64
SKIP_CH = 50   # first of the four spare channels that carry the raw observation planes out of the stem


N_PACK = 160   # MMA N dimension of az_nn_conv3x3: 3 kx taps x 50 filters, padded to a multiple of 16


def pack_conv3x3(w):
    """[64 out][64 in][3][3] (any float dtype; only the first 50 output channels are used -- the conv computes the
    network's 50 filters, network.py:22 -- all 64 input channels are) -> bf16 [3 ky][160][8 chunks][8]: the UMMA B operand
    image of az_nn_conv3x3, SWIZZLE_128B K-major.  Row r = kx*50 + co holds the 128 B of input channels of output channel
    co under tap (ky, kx) (rows 150..159 are zero); its 16-byte chunk c is stored at chunk position c ^ (r & 7)."""
    co, ci = w.shape[0], w.shape[1]
    assert co == CH and ci == CH
    t = torch.zeros((3, N_PACK, 8, 8), dtype=w.dtype, device=w.device)
    # [ky][kx][co < 50][ci] -> rows kx*50 + co
    t[:, :3 * N_FILTERS] = w[:N_FILTERS].permute(2, 3, 0, 1).reshape(3, 3 * N_FILTERS, 8, 8)
    r = torch.arange(N_PACK).view(1, N_PACK, 1)
    c = torch.arange(8).view(1, 1, 8)
    src_chunk = (c ^ (r & 7)).expand(3, N_PACK, 8)           # position p holds chunk p ^ (r & 7)
    out = torch.gather(t, 2, src_chunk.unsqueeze(-1).expand(3, N_PACK, 8, 8).to(t.device))
    return out.contiguous().to(torch.bfloat16)


class FusedEvaluator:
    def __init__(self, net, batch, device, n_ctas=0):
        self.lib = L.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.EngineUnavailable("FusedEvaluator needs a CUDA device; there is no CPU fallback")
        self.batch = batch
        self.h, self.w, self.A = net.height, net.width, net.num_distinct_actions
        if not (3 <= self.h <= 16 and 2 <= self.w <= 8):
            raise ValueError("FusedEvaluator supports boards with 3 <= H <= 16 and 2 <= W <= 8")
        self.n_ctas = n_ctas
        dev = self.device
        self.U = torch.zeros((batch, self.h + 1, self.w, CH), dtype=torch.bfloat16, device=dev)
        self.X = torch.zeros((batch, self.h + 1, self.w, CH), dtype=torch.bfloat16, device=dev)
        self.T = torch.zeros((batch, self.h + 1, self.w, CH), dtype=torch.bfloat16, device=dev)
        self.obs = torch.zeros((batch, self.h, self.w, 4), dtype=torch.bfloat16, device=dev)
        self.priors = torch.zeros((batch, self.A), dtype=torch.float32, device=dev)
        self.values = torch.zeros((batch,), dtype=torch.float32, device=dev)
        self.par = None
        # FC head: small action spaces (Connect Four) finish with the streaming k_head kernel, larger ones (Breakthrough)
        # with the tcgen05 GEMM head k_head_mma -- both FC + softmax + tanh in ONE launch of our own kernels.
        # (AZ_NN_HEAD=0: cuBLAS + torch softmax/tanh, kept only as a numerics cross-check.)
        self.small_head = self.A + 1 <= 8 and 8 * (self.h * self.w * 8 + 4) * 16 <= 100 * 1024
        self.fused_head = os.environ.get("AZ_NN_HEAD", "1") != "0"
        # every output row is a function of that row's board alone, whatever the other rows hold or where the row sits in
        # the batch (our kernels give each row the same reduction order); the cuBLAS head does not promise that
        self.row_independent = self.fused_head
        self.head_scratch = None
        if self.fused_head and not self.small_head:
            n = int(self.lib.az_nn_head_large_scratch_bytes(batch, self.A))
            self.head_scratch = torch.zeros((n + 3) // 4, dtype=torch.int32, device=dev)
        # AZ_NN_BLOCK=1: blocks 2-5 as ONE kernel each (k_block: conv1 -> conv2 with the intermediate tensor in shared
        # memory, 4 instead of 6 HBM passes per block).  Correct (tests/test_gpu_nn.py) but measured slower than the two conv
        # launches it replaces (az_resnet.cu, k_block STATUS), so the default stays two launches per block.
        self.fused_blocks = os.environ.get("AZ_NN_BLOCK", "0") == "1"
        self.timing = None   # set to a list to collect (kernel, start_event, end_event) per launch (bench.py roofline)
        self.load(net)

    @torch.no_grad()
    def load(self, net):
        """Fold BatchNorm, pad 50->64 filters, pack the UMMA operand images.  In place after the first call, so a
        captured CUDA graph keeps working when new weights arrive."""
        dev = self.device
        blocks = [getattr(net, "resblock%d" % i) for i in range(1, 6)]
        new = {}
        for k, blk in enumerate(blocks):
            a1, b1 = _fold_bn(blk.bn1)
            a2, b2 = _fold_bn(blk.bn2)
            a1, b1, a2, b2 = a1.cpu(), b1.cpu(), a2.cpu(), b2.cpu()
            w1 = blk.conv1.weight.double().cpu() * a2.view(-1, 1, 1, 1)       # bn2 folded into conv1
            c1b = blk.conv1.bias.double().cpu() * a2 + b2
            w2 = blk.conv2.weight.double().cpu()
            c2b = blk.conv2.bias.double().cpu()
            bias1 = torch.zeros(CH, dtype=torch.float64)
            bias1[:N_FILTERS] = c1b
            bias2 = torch.zeros(CH, dtype=torch.float64)
            bias2[:N_FILTERS] = c2b
            w2p = torch.zeros((CH, CH, 3, 3), dtype=torch.float64)
            w2p[:N_FILTERS, :N_FILTERS] = w2
            new["w2_%d" % k] = pack_conv3x3(w2p)
            new["b2_%d" % k] = bias2.float()
            new["b1_%d" % k] = bias1.float()
            if k == 0:
                cin = blk.conv1.in_channels
                assert cin == 4 and blk.use_1x1conv
                # stem operand image [9 taps][2 k-chunks][64 n][8]: conv1 on k 0-3 (its input is lrelu(bn1(x)))
                sw = torch.zeros((9, 2, CH, 8), dtype=torch.float64)
                w1p = torch.zeros((CH, 4, 3, 3), dtype=torch.float64)
                w1p[:N_FILTERS] = w1
                sw[:, 0, :, 0:4] = w1p.permute(2, 3, 0, 1).reshape(9, CH, 4)
                new["stem_w"] = sw.to(torch.bfloat16)
                sb3 = torch.zeros(CH, dtype=torch.float64)
                sb3[:N_FILTERS] = blk.conv3.bias.double().cpu()
                # the 1x1 skip projection (conv3) rides in conv2: the stem leaves the raw planes in channels 50..53 of U,
                # conv2's centre tap maps them with conv3's weights, conv3's bias joins conv2's
                w2p[:N_FILTERS, SKIP_CH:SKIP_CH + 4, 1, 1] = blk.conv3.weight.double().cpu().reshape(N_FILTERS, 4)
                new["w2_0"] = pack_conv3x3(w2p)
                new["b2_0"] = (bias2 + sb3).float()
                new["stem_st"] = torch.cat([a1, b1]).float()
            else:
                w1p = torch.zeros((CH, CH, 3, 3), dtype=torch.float64)
                w1p[:N_FILTERS, :N_FILTERS] = w1
                new["w1_%d" % k] = pack_conv3x3(w1p)
                s = torch.zeros(CH, dtype=torch.float64)
                t = torch.zeros(CH, dtype=torch.float64)
                s[:N_FILTERS], t[:N_FILTERS] = a1, b1
                new["s_%d" % k], new["t_%d" % k] = s.float(), t.float()   # bn1 of block k, applied by block k-1's epilogue
        # FC head over the flatten of one board: [A+1][H+1][W][64] (zero on the pad row)
        fw = net.fc1.weight.double().cpu().view(self.A + 1, N_FILTERS, self.h, self.w)
        fwp = torch.zeros((self.A + 1, self.h + 1, self.w, CH), dtype=torch.float64)
        fwp[:, :self.h, :, :N_FILTERS] = fw.permute(0, 2, 3, 1)
        new["fw"] = fwp.reshape(self.A + 1, -1).to(torch.bfloat16)
        new["fb"] = net.fc1.bias.double().cpu().float()
        if self.fused_head and self.small_head:   # k_head operand: [8 outputs][H*W*64] bf16 (unused outputs zero), bias [8]
            hw = torch.zeros((8, self.h * self.w * CH), dtype=torch.float64)
            hw[:self.A + 1] = fwp[:, :self.h].reshape(self.A + 1, -1)
            hb = torch.zeros(8, dtype=torch.float64)
            hb[:self.A + 1] = net.fc1.bias.double().cpu()
            new["hw"], new["hb"] = hw.to(torch.bfloat16), hb.float()
        if self.par is None:
            self.par = {k: v.contiguous().to(dev) for k, v in new.items()}
        else:
            for k, v in new.items():
                self.par[k].copy_(v.to(dev))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _timed(self, name, fn):
        if self.timing is None:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn()
        e1.record()
        self.timing.append((name, e0, e1))
        return rc

    def _conv(self, inp, w, b, res, out, out2, s2, t2, lrelu, flags=0):
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        name = "conv" + ("+res" if res is not None else "") + ("+out2" if out2 is not None else "")
        rc = self._timed(name, lambda: self.lib.az_nn_conv3x3(
            p(inp), p(w), p(b), p(res), p(out), p(out2), p(s2), p(t2), self.batch, self.h, self.w,
            1 if lrelu else 0, flags, self.n_ctas, self._stream()))
        if rc:
            raise RuntimeError("az_nn_conv3x3: " + self.lib.az_nn_last_error().decode())

    @torch.no_grad()
    def __call__(self):
        """Evaluate self.obs into self.priors / self.values on the current stream (graph-capturable)."""
        P_ = self.par
        p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        rc = self._timed("stem", lambda: self.lib.az_nn_stem(
            p(self.obs), p(P_["stem_w"]), p(P_["b1_0"]), p(P_["stem_st"]), p(self.U), self.batch, self.h, self.w,
            self.n_ctas, self._stream()))
        if rc:
            raise RuntimeError("az_nn_stem: " + self.lib.az_nn_last_error().decode())
        # Layers alternate their tile direction: each reads its input starting from the part the previous layer wrote
        # last (still in L2); the stem writes front to back, so the first conv goes back to front.
        # block 1, second conv: X = conv(U) + conv1x1(obs) ; T = lrelu(bn1_2(X))   (skip projection inside the conv)
        self._conv(self.U, P_["w2_0"], P_["b2_0"], None, self.X, self.T, P_["s_1"], P_["t_1"], False, flags=L.NN_F_REVERSE)
        t_in, t_alt = self.T, self.U     # fused blocks ping-pong the activated tensor between T and U
        for k in range(1, 5):
            last = k == 4
            if self.fused_blocks:
                t_out = None if last else t_alt
                rc = self._timed("block" if last else "block+out2", lambda: self.lib.az_nn_block(
                    p(t_in), p(P_["w1_%d" % k]), p(P_["b1_%d" % k]), p(P_["w2_%d" % k]), p(P_["b2_%d" % k]), p(self.X),
                    None if last else p(t_out), None if last else p(P_["s_%d" % (k + 1)]),
                    None if last else p(P_["t_%d" % (k + 1)]), self.batch, self.h, self.w, self.n_ctas, self._stream()))
                if rc:
                    raise RuntimeError("az_nn_block: " + self.lib.az_nn_last_error().decode())
                t_in, t_alt = t_alt, t_in
                continue
            self._conv(self.T, P_["w1_%d" % k], P_["b1_%d" % k], None, self.U, None, None, None, True)
            self._conv(self.U, P_["w2_%d" % k], P_["b2_%d" % k], self.X, self.X, None if last else self.T,
                       None if last else P_["s_%d" % (k + 1)], None if last else P_["t_%d" % (k + 1)], False,
                       flags=L.NN_F_REVERSE)
        if self.fused_head and self.small_head:
            rc = self._timed("head", lambda: self.lib.az_nn_head(
                p(self.X), p(P_["hw"]), p(P_["hb"]), p(self.priors), p(self.values), self.batch, self.h, self.w, self.A,
                self.n_ctas, self._stream()))
            if rc:
                raise RuntimeError("az_nn_head: " + self.lib.az_nn_last_error().decode())
        elif self.fused_head:
            rc = self._timed("head", lambda: self.lib.az_nn_head_large(
                p(self.X), p(P_["fw"]), p(P_["fb"]), p(self.priors), p(self.values), p(self.head_scratch), self.batch,
                self.h, self.w, self.A, self._stream()))
            if rc:
                raise RuntimeError("az_nn_head_large: " + self.lib.az_nn_last_error().decode())
        else:
            out = F.linear(self.X.view(self.batch, -1), P_["fw"]).float() + P_["fb"]
            torch.softmax(out[:, :self.A], dim=1, out=self.priors)
            torch.tanh(out[:, self.A], out=self.values)
        return self.priors, self.values

    @torch.no_grad()
    def eval_batch(self, obs):
        self.obs.copy_(obs.to(torch.bfloat16))
        pr, v = self()
        return pr.clone(), v.clone()
