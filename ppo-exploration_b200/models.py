"""Networks of the learner hot path as flat device parameter banks driven by libppx kernels.

Mirrors models.py of the reference: Policy (:15-124) over MlpNetwork / MlpIntrinsic (:137-213),
RndNetwork (:216-267) and IntrinsicCuriosityModule (:270-320).  Same class names, constructor
arguments, method names and state_dict keys (so weights move both ways), but:
  * every network keeps its parameters, gradients and Adam moments in ONE flat f32 CUDA vector
    (one clip+Adam launch per optimiser step, one flat-buffer all-reduce when sharded);
  * weights are stored in-major ([K_in, N_out]); actor / critic / int_critic first layers are
    concatenated along N and their second layers run as one strided-batched launch;
  * forward AND backward are explicit kernel sequences (ppx_linear_fwd / _bwd_data / _bwd_weight) --
    there is no autograd graph.
Initialisation replays the reference's own torch calls on the CPU in the same order
(nn.Linear default init, then orthogonal_(sqrt 2) / constant_), so identical seeds give identical
weights; that is host-side setup, not the hot path.
"""
import math

import numpy as np
import torch

from . import _lib as L

import ctypes as C
import os

ACT = {"none": 0, "tanh": 1, "leaky_relu": 2, "elu": 3, "relu": 4}
F4 = 4  # bytes per float
# tcgen05 3xTF32 path (tc_gemm.cu) for the forward of WIDE dense layers -- the bonus nets' first layers (RND
# D=28224, ICM D=3136): K >= TC_MIN_K.  PPX_TC=0 forces the SIMT fp32 kernels everywhere.  The narrow policy MLPs
# (K <= 128) run the fused SIMT kernel instead (mlp_fused.cu); PPX_TC_POLICY=1 routes them through tcgen05 for
# comparison (slower at these widths, see profiles/).
TC_ENABLED = os.environ.get("PPX_TC", "1") != "0"
TC_POLICY = os.environ.get("PPX_TC_POLICY", "0") == "1"
TC_MIN_K = 256
# normalize_obs fused into the tcgen05 A-split stage (RndNetwork.int_reward(obs, rms=...)).  Measured at C3 it LOSES to
# the separate float4 normalisation pass (3.07 vs 2.2 ms per bonus pass: the f64 arithmetic lands on the 4 splitter warps
# of both first-layer kernels and they become the pipeline's slowest stage), so it is opt-in.
TC_FUSE_NORM = os.environ.get("PPX_TC_FUSE_NORM", "0") == "1"
# fused forward / backward of the D-h-h-o policy MLPs (mlp_fused.cu); PPX_FUSED_MLP=0 forces the layer-by-layer path
FUSED_ENABLED = os.environ.get("PPX_FUSED_MLP", "1") != "0"
# h = 64 policy MLPs: fused kernels with the 64x64 GEMMs on tcgen05 (mlp_tc.cu); PPX_MLP_TC=0 keeps the SIMT pair
MLP_TC_ENABLED = os.environ.get("PPX_MLP_TC", "1") != "0"


class ParamBank:
    """Flat parameter / gradient / Adam-moment vectors with named views."""

    def __init__(self, specs, device):
        self.device = device
        self.offsets, self.shapes = {}, {}
        off = 0
        for name, shape in specs:
            n = int(np.prod(shape))
            self.offsets[name], self.shapes[name] = off, tuple(shape)
            off += (n + 3) // 4 * 4                    # keep every tensor 16-byte aligned
        self.size = off
        z = lambda: torch.zeros(off, dtype=torch.float32, device=device)
        self.flat, self.grad, self.exp_avg, self.exp_avg_sq = z(), z(), z(), z()
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=device)
        self.norm_dev = torch.zeros(1, dtype=torch.float64, device=device)
        self._ws = torch.zeros(4096, dtype=torch.float64, device=device)
        self._ticket = torch.zeros(2, dtype=torch.int32, device=device)      # rendezvous counters of the fused optimiser tail
        self._fused = None
        self.tc_weights = []                       # TcWeight shadows to refresh after every step

    def refresh_tc(self):
        for t in self.tc_weights:
            t.refresh()

    _STATE = ("flat", "grad", "exp_avg", "exp_avg_sq", "step_dev")

    def state_dict(self):
        """Parameters, gradients, Adam moments and the device step counter as CPU tensors (checkpoints)."""
        return {k: getattr(self, k).cpu() for k in self._STATE}

    def load_state_dict(self, sd):
        """Restore `state_dict()` in place (addresses, and so captured graphs, stay valid) and refresh the tensor-core
        weight shadows."""
        from .checkpoint import tensor_into
        for k in self._STATE:
            tensor_into(getattr(self, k), sd[k], f"parameter bank '{k}'")
        self.refresh_tc()

    def view(self, name, grad=False):
        o, s = self.offsets[name], self.shapes[name]
        return (self.grad if grad else self.flat)[o:o + int(np.prod(s))].view(s)

    def p(self, name, extra=0):
        return self.flat.data_ptr() + (self.offsets[name] + extra) * F4

    def g(self, name, extra=0):
        return self.grad.data_ptr() + (self.offsets[name] + extra) * F4

    def fused_adam(self, lr, max_norm, extra_name=None, betas=(0.9, 0.999), eps=1e-8, px=None):
        """ppx_fused_adam record for this bank: clip_grad_norm_(max_norm) + Adam applied by the blocks of the fused MLP
        backward's reduce kernel (no separate optimiser launch).  `extra_name`: a parameter outside the MLP whose gradient
        enters the norm (action_log_std).  `px` (dist.PeerExchange): sharded -- the same kernel also all-reduces the
        gradient over peer memory."""
        key = (float(lr), float(max_norm), extra_name, betas, eps, self.grad.data_ptr(), id(px))
        if self._fused is None or self._fused[0] != key:
            ex_ptr, ex_n = (self.g(extra_name), int(np.prod(self.shapes[extra_name]))) if extra_name else (None, 0)
            peer = (0, 0, None, None, None)
            if px is not None:
                peer = (px.W, px.rank, C.cast(px.peer_xg, C.c_void_p), px.seq[3], px.status_ptr)
            rec = L.FusedAdam(self.flat.data_ptr(), self.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                              self.size, float(max_norm), float(lr), float(betas[0]), float(betas[1]), float(eps),
                              self.step_dev.data_ptr(), self.norm_dev.data_ptr(), ex_ptr, ex_n, self._ticket.data_ptr(), *peer)
            self._fused = (key, rec, px)                        # px: keeps the host pointer tables alive
        return self._fused[1]

    def adam_step_pre(self, lr, max_norm, sumsq, n_partials, extra_name=None, betas=(0.9, 0.999), eps=1e-8):
        """clip + Adam when the producer of the gradients already left sum-of-squares partials (and bumped the step)."""
        ex_ptr, ex_n = (self.g(extra_name), int(np.prod(self.shapes[extra_name]))) if extra_name else (None, 0)
        L.call("ppx_clip_adam_pre", self.flat.data_ptr(), self.grad.data_ptr(), self.exp_avg.data_ptr(),
               self.exp_avg_sq.data_ptr(), self.size, float(max_norm), float(lr), float(betas[0]), float(betas[1]), float(eps),
               self.step_dev.data_ptr(), self.norm_dev.data_ptr(), sumsq.data_ptr(), int(n_partials), ex_ptr, ex_n, L.stream())
        self.refresh_tc()

    def adam_step(self, lr, max_norm=0.0, betas=(0.9, 0.999), eps=1e-8):
        """clip_grad_norm_(max_norm) over the whole bank + Adam (device-side step counter)."""
        L.call("ppx_clip_adam", self.flat.data_ptr(), self.grad.data_ptr(), self.exp_avg.data_ptr(),
               self.exp_avg_sq.data_ptr(), self.size, float(max_norm), self.size if max_norm > 0 else 0, float(lr),
               float(betas[0]), float(betas[1]), float(eps), 0, self.step_dev.data_ptr(), self.norm_dev.data_ptr(),
               self._ws.data_ptr(), L.stream())
        self.refresh_tc()


class TcWeight:
    """hi/lo tf32 split of one in-major weight matrix W [K,N] (and of its transpose), refreshed after every
    optimiser step: forward uses W^T [N,K] as the K-major B operand, the data-gradient uses W [K,N]."""

    def __init__(self, w_ptr, K, N, device, transposed_only=False):
        self.w_ptr, self.K, self.N = w_ptr, K, N
        e = lambda *s: torch.empty(*s, dtype=torch.float32, device=device)
        self.hi, self.lo = (None, None) if transposed_only else (e(K, N), e(K, N))
        self.hiT, self.loT = e(N, K), e(N, K)
        self.refresh()

    def refresh(self):
        L.call("ppx_tc_split", self.w_ptr, self.K, self.N, L.ptr(self.hi), L.ptr(self.lo), self.hiT.data_ptr(),
               self.loT.data_ptr(), L.stream())


def tc_ok(M, R, N, lda, ldb, a_ptr, b_ptr):
    return (TC_ENABLED and M >= 128 and L.call("ppx_tc_supported", M, R, N, lda, ldb, a_ptr, b_ptr) == 1)


_splitk_ws = {}          # device -> f32 workspace of the split-K tensor-core GEMM (grows; captured graphs are retired when it moves)


def _tc_workspace(M, R, N):
    need = int(L.call("ppx_tc_linear_workspace", int(M), int(R), int(N)))
    if need == 0:
        return None, 0
    dev = torch.cuda.current_device()
    ws = _splitk_ws.get(dev)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.float32, device=torch.device("cuda", dev))
        _splitk_ws[dev] = ws
        _Scratch.generation += 1
    return ws.data_ptr(), ws.numel()


def dense_fwd(x_ptr, ldx, w_ptr, b_ptr, M, K, N, act, y_ptr, ldy, tcw=None, a_norm=None):
    """act(X @ W + b): tensor-core path when the shape allows it, SIMT fp32 otherwise.  a_norm = (mean_ptr, istd_ptr,
    clip): X is normalised on the fly inside the tensor-core kernel (only valid when can_fuse_norm() said so)."""
    if tcw is not None and tc_ok(M, K, N, ldx, K, x_ptr, tcw.hiT.data_ptr()):
        mean_ptr, istd_ptr, clip = a_norm if a_norm is not None else (None, None, 0.0)
        ws_ptr, ws_n = _tc_workspace(M, K, N)                    # few output tiles + long reduction: split-K
        L.call("ppx_tc_linear_ws", x_ptr, ldx, tcw.hiT.data_ptr(), tcw.loT.data_ptr(), K, M, K, N, b_ptr, None, 0, act, 0,
               mean_ptr, istd_ptr, float(clip), y_ptr, ldy, ws_ptr, ws_n, L.stream())
    else:
        assert a_norm is None, "fused input normalisation needs the tensor-core path"
        linear_fwd(x_ptr, ldx, w_ptr, b_ptr, M, K, N, act, y_ptr, ldy)


def dense_bwd_data(dy_ptr, lddy, w_ptr, M, K, N, h_ptr, ldh, act, dx_ptr, lddx, tcw=None):
    """(dY @ W^T) * act'(H): tensor-core path when the shape allows it."""
    if tcw is not None and tc_ok(M, N, K, lddy, N, dy_ptr, tcw.hi.data_ptr()):
        L.call("ppx_tc_linear", dy_ptr, lddy, tcw.hi.data_ptr(), tcw.lo.data_ptr(), N, M, N, K, None, h_ptr, ldh, act, 1,
               None, None, 0.0, dx_ptr, lddx, L.stream())
    else:
        linear_bwd_data(dy_ptr, lddy, w_ptr, M, K, N, h_ptr, ldh, act, dx_ptr, lddx)


class _Scratch:
    """Named persistent device buffers that grow on demand (stable addresses between calls of equal size).

    `generation` (process-wide) counts every RE-allocation of an existing buffer: a captured CUDA graph that still
    points at the old block must not be replayed, so the learners compare the counter before every replay and drop
    their graphs when it moved (algorithms.BaseAlgorithm._graph_call)."""
    generation = 0

    def __init__(self, device):
        self.device, self.bufs = device, {}

    def get(self, name, numel, dtype=torch.float32):
        b = self.bufs.get(name)
        if b is None or b.numel() < numel or b.dtype != dtype:
            if b is not None:
                _Scratch.generation += 1
            b = torch.empty(max(int(numel), 1), dtype=dtype, device=self.device)
            self.bufs[name] = b
        return b


def linear_fwd(x_ptr, ldx, w_ptr, b_ptr, M, K, N, act, y_ptr, ldy, batch=1, sx=0, sw=0, sb=0, sy=0):
    L.call("ppx_linear_fwd", x_ptr, ldx, w_ptr, b_ptr, M, K, N, act, y_ptr, ldy, batch, sx, sw, sb, sy, L.stream())


def linear_bwd_data(dy_ptr, lddy, w_ptr, M, K, N, h_ptr, ldh, act, dx_ptr, lddx, batch=1, sdy=0, sw=0, sh=0, sdx=0):
    L.call("ppx_linear_bwd_data", dy_ptr, lddy, w_ptr, M, K, N, h_ptr, ldh, act, dx_ptr, lddx, batch, sdy, sw, sh, sdx,
           L.stream())


def linear_bwd_weight(scratch, x_ptr, ldx, dy_ptr, lddy, M, K, N, dw_ptr, db_ptr, batch=1, sx=0, sdy=0, sdw=0, sdb=0):
    # the tensor-core kernel tiles dW [K, N]: a gradient with only a handful of 128 x 128 tiles and a very long sample
    # dimension (conv layers: 256 x 32 over 1.6M rows) fills the GPU better on the SIMT kernel, which splits over the samples
    tiles = -(-K // 128) * -(-N // (64 if N <= 64 else 128))
    if (TC_ENABLED and batch == 1 and K >= TC_MIN_K and dw_ptr % 16 == 0 and tiles >= 12
            and L.call("ppx_tc_wgrad_supported", M, K, N, x_ptr, dy_ptr) == 1):
        # wide layer: samples as the reduction dimension of the tcgen05 3xTF32 kernel (tc_gemm.cu)
        ws = scratch.get("tc_wgrad_ws", L.call("ppx_tc_wgrad_workspace", M, K, N))
        L.call("ppx_tc_wgrad", x_ptr, ldx, dy_ptr, lddy, M, K, N, dw_ptr, db_ptr, ws.data_ptr(), L.stream())
        return
    need = L.call("ppx_linear_bwd_weight_workspace", M, K, N, batch)
    ws = scratch.get("wgrad_ws", need)
    L.call("ppx_linear_bwd_weight", x_ptr, ldx, dy_ptr, lddy, M, K, N, dw_ptr, db_ptr, ws.data_ptr(), batch, sx, sdy,
           sdw, sdb, L.stream())


class DenseStack:
    """A chain of Linear(+activation) layers living inside a ParamBank under `prefix`.

    layers: [(K, N, act_name)], last activation must be "none".  Reference state_dict names are
    f"{prefix}.{2*i}.weight/bias" (nn.Sequential indices with the activations interleaved)."""

    def __init__(self, bank, prefix, layers, scratch):
        self.bank, self.prefix, self.layers, self.scratch = bank, prefix, layers, scratch
        assert layers[-1][2] == "none"
        self.tc = {}                                  # layer index -> TcWeight (wide layers only)

    def enable_tc(self):
        """(Re)build the tensor-core weight shadows of the wide layers; call after the parameters were (re)loaded.
        They are refreshed after every optimiser step of the owning bank (ParamBank.adam_step)."""
        if not TC_ENABLED:
            return
        b, dev = self.bank, self.bank.device
        b.tc_weights = [t for t in b.tc_weights if t not in self.tc.values()]
        if self.tc:
            _Scratch.generation += 1               # captured refresh launches point at the shadows being dropped
        self.tc = {}
        for i, (K, N, _) in enumerate(self.layers):
            if K >= TC_MIN_K and K % 4 == 0 and N >= 16:
                self.tc[i] = TcWeight(b.p(f"{self.prefix}.{2 * i}.weight"), K, N, dev, transposed_only=True)
        b.tc_weights += list(self.tc.values())

    @staticmethod
    def specs(prefix, layers):
        out = []
        for i, (K, N, _) in enumerate(layers):
            out += [(f"{prefix}.{2 * i}.weight", (K, N)), (f"{prefix}.{2 * i}.bias", (N,))]
        return out

    def can_fuse_norm(self, x):
        """True when layer 0 runs on the tensor-core kernel for this input, i.e. an input normalisation can be fused."""
        K, N, _ = self.layers[0]
        t = self.tc.get(0)
        return t is not None and tc_ok(x.shape[0], K, N, x.stride(0), K, x.data_ptr(), t.hiT.data_ptr())

    def forward(self, x, tag="", a_norm=None):
        """x: [M, K0] contiguous f32 CUDA.  Returns the list of activations [x, h1, ..., y].  a_norm (layer 0 only):
        (mean_ptr, istd_ptr, clip) -> clip((x - mean) * istd) is applied to x inside the first layer's kernel."""
        M = x.shape[0]
        acts = [x]
        for i, (K, N, act) in enumerate(self.layers):
            y = self.scratch.get(f"{self.prefix}{tag}.h{i}", M * N)[:M * N].view(M, N)
            dense_fwd(acts[-1].data_ptr(), acts[-1].stride(0), self.bank.p(f"{self.prefix}.{2 * i}.weight"),
                      self.bank.p(f"{self.prefix}.{2 * i}.bias"), M, K, N, ACT[act], y.data_ptr(), N, self.tc.get(i),
                      a_norm if i == 0 else None)
            acts.append(y)
        return acts

    def backward(self, acts, d_y, need_dx=False, accumulate_tag=""):
        """Gradients into bank.grad (overwrites this stack's slices).  d_y: [M, N_last] contiguous.
        Returns dX ([M,K0]) if need_dx."""
        M = d_y.shape[0]
        d = d_y
        for i in range(len(self.layers) - 1, -1, -1):
            K, N, _ = self.layers[i]
            x = acts[i]
            linear_bwd_weight(self.scratch, x.data_ptr(), x.stride(0), d.data_ptr(), d.stride(0), M, K, N,
                              self.bank.g(f"{self.prefix}.{2 * i}.weight"), self.bank.g(f"{self.prefix}.{2 * i}.bias"))
            if i == 0 and not need_dx:
                return None
            prev_act = self.layers[i - 1][2] if i > 0 else "none"
            dx = self.scratch.get(f"{self.prefix}{accumulate_tag}.d{i}", M * K)[:M * K].view(M, K)
            linear_bwd_data(d.data_ptr(), d.stride(0), self.bank.p(f"{self.prefix}.{2 * i}.weight"), M, K, N,
                            x.data_ptr() if i > 0 else None, x.stride(0) if i > 0 else K, ACT[prev_act],
                            dx.data_ptr(), K)
            d = dx
        return d


class ConvTrunk:
    """Convolutional feature extractor for image observations (SURVEY §8f item 2): the Nature-CNN trunk of the reference's
    dead draft (.ipynb_checkpoints/models-checkpoint.py:48-66: Conv 8/4 -> 4/2 -> 3/1, each + activation -> Flatten ->
    Linear(7*7*64, hidden) + activation) or the RND conv stacks (:93-121), with forward AND backward, so it can sit in
    front of the MLP heads of `Policy` / `RndNetwork`.  The reference has no live conv arithmetic; parity is defined
    against torch.nn.Conv2d / nn.Linear in fp64 (tests/test_gpu_conv.py).

    Every layer is im2col + one of the library's dense layers (ppx_im2col / ppx_col2im + `dense_fwd` / `linear_bwd_*`:
    tcgen05 3xTF32 for reductions >= 256, split-K where the tiles are few), activations stay NHWC between layers; only
    layer 0 reads the caller's NCHW frames.  Parameters live in a ParamBank under `prefix` with nn.Sequential naming
    (f"{prefix}.{2*i}.weight" ...), stored in-major [K, Cout] with the patch order of the layer's im2col.

    in_shape: (C, H, W); convs: [(Cout, kernel, stride, act)]; fc: (hidden, act) or None."""

    def __init__(self, bank, prefix, in_shape, convs, fc, scratch):
        self.bank, self.prefix, self.scratch = bank, prefix, scratch
        self.geo, self.fc = self.geometry(in_shape, convs), fc
        C, H, W = self.geo[-1][8], self.geo[-1][6], self.geo[-1][7]
        self.flat_dim = C * H * W
        self.out_dim = fc[0] if fc else self.flat_dim
        self.tc = {}

    @staticmethod
    def geometry(in_shape, convs):
        """per conv layer: (Cin, H, W, k, stride, act, OH, OW, Cout)"""
        C, H, W = in_shape
        geo = []
        for Cout, k, s, act in convs:
            OH, OW = (H - k) // s + 1, (W - k) // s + 1
            geo.append((C, H, W, k, s, act, OH, OW, Cout))
            C, H, W = Cout, OH, OW
        return geo

    @staticmethod
    def specs(prefix, in_shape, convs, fc):
        geo, out = ConvTrunk.geometry(in_shape, convs), []
        for i, (C, H, W, k, s, act, OH, OW, Cout) in enumerate(geo):
            out += [(f"{prefix}.{2 * i}.weight", (C * k * k, Cout)), (f"{prefix}.{2 * i}.bias", (Cout,))]
        if fc:
            C, OH, OW = geo[-1][8], geo[-1][6], geo[-1][7]
            j = 2 * len(geo) + 1                       # nn.Sequential index after the Flatten module
            out += [(f"{prefix}.{j}.weight", (C * OH * OW, fc[0])), (f"{prefix}.{j}.bias", (fc[0],))]
        return out

    def _fc_name(self):
        return f"{self.prefix}.{2 * len(self.geo) + 1}"

    def load_torch(self, state_dict):
        """Weights of the equivalent torch nn.Sequential(Conv2d, act, ..., Flatten, Linear, act) state_dict -> the bank
        (patch / flatten orders converted: layer 0 keeps torch's (c, kh, kw), deeper layers and the Flatten are NHWC)."""
        for i, (C, H, W, k, s, act, OH, OW, Cout) in enumerate(self.geo):
            w = state_dict[f"{2 * i}.weight"].detach().to(torch.float32)           # [Cout, Cin, k, k]
            wm = w.reshape(Cout, -1) if i == 0 else w.permute(0, 2, 3, 1).reshape(Cout, -1)
            self.bank.view(f"{self.prefix}.{2 * i}.weight").copy_(wm.t())
            self.bank.view(f"{self.prefix}.{2 * i}.bias").copy_(state_dict[f"{2 * i}.bias"].detach().to(torch.float32))
        if self.fc:
            C, OH, OW = self.geo[-1][8], self.geo[-1][6], self.geo[-1][7]
            j = 2 * len(self.geo) + 1
            w = state_dict[f"{j}.weight"].detach().to(torch.float32)                # [hidden, C*OH*OW] over torch's (c, h, w)
            wm = w.reshape(-1, C, OH, OW).permute(0, 2, 3, 1).reshape(w.shape[0], -1)
            self.bank.view(f"{self._fc_name()}.weight").copy_(wm.t())
            self.bank.view(f"{self._fc_name()}.bias").copy_(state_dict[f"{j}.bias"].detach().to(torch.float32))
        self.enable_tc()

    def grads_as_torch(self):
        """The bank's gradients of this trunk in the torch state_dict layouts (tests, export)."""
        out = {}
        for i, (C, H, W, k, s, act, OH, OW, Cout) in enumerate(self.geo):
            g = self.bank.view(f"{self.prefix}.{2 * i}.weight", grad=True).t()      # [Cout, K]
            out[f"{2 * i}.weight"] = (g.reshape(Cout, C, k, k) if i == 0 else g.reshape(Cout, k, k, C).permute(0, 3, 1, 2)).contiguous()
            out[f"{2 * i}.bias"] = self.bank.view(f"{self.prefix}.{2 * i}.bias", grad=True).clone()
        if self.fc:
            C, OH, OW = self.geo[-1][8], self.geo[-1][6], self.geo[-1][7]
            j = 2 * len(self.geo) + 1
            g = self.bank.view(f"{self._fc_name()}.weight", grad=True).t()          # [hidden, OH*OW*C]
            out[f"{j}.weight"] = g.reshape(-1, OH, OW, C).permute(0, 3, 1, 2).reshape(g.shape[0], -1).contiguous()
            out[f"{j}.bias"] = self.bank.view(f"{self._fc_name()}.bias", grad=True).clone()
        return out

    def enable_tc(self):
        """tensor-core weight shadows of the layers whose reduction is wide enough (refreshed after every optimiser step)"""
        if not TC_ENABLED:
            return
        b = self.bank
        b.tc_weights = [t for t in b.tc_weights if t not in self.tc.values()]
        if self.tc:
            _Scratch.generation += 1
        self.tc = {}
        names = [(f"{self.prefix}.{2 * i}.weight", g[0] * g[3] * g[3], g[8]) for i, g in enumerate(self.geo)]
        if self.fc:
            names.append((f"{self._fc_name()}.weight", self.flat_dim, self.fc[0]))
        for i, (name, K, N) in enumerate(names):
            if K >= TC_MIN_K and K % 4 == 0 and N >= 16:
                self.tc[i] = TcWeight(b.p(name), K, N, b.device, transposed_only=True)
        b.tc_weights += list(self.tc.values())

    def forward(self, x, tag=""):
        """x: [N, C*H*W] (or [N,C,H,W]) contiguous f32 CUDA frames.  Returns (features [N, out_dim], saved) -- `saved`
        holds the im2col matrices and layer outputs the backward needs."""
        N = x.shape[0]
        cur, saved = x.reshape(N, -1), []
        for i, (C, H, W, k, s, act, OH, OW, Cout) in enumerate(self.geo):
            M, K = N * OH * OW, C * k * k
            cols = self.scratch.get(f"{self.prefix}{tag}.cols{i}", M * K)[:M * K].view(M, K)
            L.call("ppx_im2col", cur.data_ptr(), 1 if i == 0 else 0, N, C, H, W, k, k, s, cols.data_ptr(), L.stream())
            y = self.scratch.get(f"{self.prefix}{tag}.y{i}", M * Cout)[:M * Cout].view(M, Cout)
            dense_fwd(cols.data_ptr(), K, self.bank.p(f"{self.prefix}.{2 * i}.weight"), self.bank.p(f"{self.prefix}.{2 * i}.bias"),
                      M, K, Cout, ACT[act], y.data_ptr(), Cout, self.tc.get(i))
            saved.append((cols, y))
            cur = y
        feat = cur.view(N, self.flat_dim)
        if self.fc:
            hid, act = self.fc
            f = self.scratch.get(f"{self.prefix}{tag}.feat", N * hid)[:N * hid].view(N, hid)
            dense_fwd(feat.data_ptr(), self.flat_dim, self.bank.p(f"{self._fc_name()}.weight"), self.bank.p(f"{self._fc_name()}.bias"),
                      N, self.flat_dim, hid, ACT[act], f.data_ptr(), hid, self.tc.get(len(self.geo)))
            saved.append((feat, f))
            feat = f
        return feat, saved

    def backward(self, saved, d_feat, need_dx=False, tag=""):
        """Gradients of every layer into bank.grad (overwritten).  d_feat: [N, out_dim] gradient w.r.t. the returned
        features (AFTER their activation).  Returns dX [N, C*H*W] in the input's NCHW layout if need_dx."""
        N = d_feat.shape[0]
        sc = self.scratch
        d = d_feat
        if self.fc:
            hid, act = self.fc
            flat, f = saved[-1]
            dz = sc.get(f"{self.prefix}{tag}.dz_fc", N * hid)[:N * hid].view(N, hid)
            L.call("ppx_act_bwd_mul", d.data_ptr(), f.data_ptr(), N * hid, ACT[act], dz.data_ptr(), L.stream())
            name = self._fc_name()
            linear_bwd_weight(sc, flat.data_ptr(), self.flat_dim, dz.data_ptr(), hid, N, self.flat_dim, hid,
                              self.bank.g(f"{name}.weight"), self.bank.g(f"{name}.bias"))
            last_act = self.geo[-1][5]
            dflat = sc.get(f"{self.prefix}{tag}.dflat", N * self.flat_dim)[:N * self.flat_dim].view(N, self.flat_dim)
            # dY_conv_last = (dz W_fc^T) * act'(y_last): the producer's activation derivative fused into the dgrad epilogue
            linear_bwd_data(dz.data_ptr(), hid, self.bank.p(f"{name}.weight"), N, self.flat_dim, hid, flat.data_ptr(),
                            self.flat_dim, ACT[last_act], dflat.data_ptr(), self.flat_dim)
            d = dflat
        else:
            C, OH, OW, act = self.geo[-1][8], self.geo[-1][6], self.geo[-1][7], self.geo[-1][5]
            y = saved[len(self.geo) - 1][1]
            dz = sc.get(f"{self.prefix}{tag}.dz_last", N * self.flat_dim)[:N * self.flat_dim].view(N, self.flat_dim)
            L.call("ppx_act_bwd_mul", d.data_ptr(), y.data_ptr(), N * self.flat_dim, ACT[act], dz.data_ptr(), L.stream())
            d = dz
        # d: gradient w.r.t. the PRE-activation output of the last conv layer, [N*OH*OW, Cout] rows (NHWC)
        for i in range(len(self.geo) - 1, -1, -1):
            C, H, W, k, s, act, OH, OW, Cout = self.geo[i]
            M, K = N * OH * OW, C * k * k
            cols, _ = saved[i]
            dy = d.reshape(M, Cout)
            linear_bwd_weight(sc, cols.data_ptr(), K, dy.data_ptr(), Cout, M, K, Cout,
                              self.bank.g(f"{self.prefix}.{2 * i}.weight"), self.bank.g(f"{self.prefix}.{2 * i}.bias"))
            if i == 0 and not need_dx:
                return None
            dcols = sc.get(f"{self.prefix}{tag}.dcols{i}", M * K)[:M * K].view(M, K)
            linear_bwd_data(dy.data_ptr(), Cout, self.bank.p(f"{self.prefix}.{2 * i}.weight"), M, K, Cout, None, K, ACT["none"],
                            dcols.data_ptr(), K)
            dx = sc.get(f"{self.prefix}{tag}.dx{i}", N * C * H * W)[:N * C * H * W]
            L.call("ppx_col2im", dcols.data_ptr(), 1 if i == 0 else 0, N, C, H, W, k, k, s, dx.data_ptr(), L.stream())
            if i > 0:                                              # through the previous layer's activation
                y_prev = saved[i - 1][1]
                L.call("ppx_act_bwd_mul", dx.data_ptr(), y_prev.data_ptr(), dx.numel(), ACT[self.geo[i - 1][5]], dx.data_ptr(),
                       L.stream())
            d = dx
        return d.view(N, -1)


def _to_in_major(w):
    return w.detach().t().contiguous()


class _TorchInit:
    """CPU replay of the reference's module construction, only to consume the torch RNG identically."""

    @staticmethod
    def linear(i, o):
        return torch.nn.Linear(i, o)

    @staticmethod
    def orthogonal(lin):
        torch.nn.init.orthogonal_(lin.weight, math.sqrt(2))
        torch.nn.init.constant_(lin.bias, 0)


class ParallelMLP:
    """G independent D-h-h-out_g tanh MLPs sharing one input (actor | critic | int_critic), batched.

    Parameters (in `bank`): W1 [D, G*h], b1 [G*h], W2 [G,h,h], b2 [G,h], W3.g [h,out_g], b3.g [out_g]."""

    def __init__(self, bank, names, D, h, outs, scratch):
        self.bank, self.names, self.D, self.h, self.outs, self.scratch = bank, names, D, h, outs, scratch
        self.G = len(names)
        self.tc1 = self.tc2 = None
        self._fa = None

    def enable_tc(self):
        """(Re)build the tensor-core weight shadows; call after the parameters were (re)loaded.  The first layer takes
        the tcgen05 path when it is wide (Atari-shaped flat input, D >= TC_MIN_K); the h x h second layers only with
        PPX_TC_POLICY=1 (slower than SIMT at these widths)."""
        if not TC_ENABLED:
            return
        b, G, h, D, dev = self.bank, self.G, self.h, self.D, self.bank.device
        b.tc_weights = [t for t in b.tc_weights if t not in ([self.tc1] if self.tc1 else []) + (self.tc2 or [])]
        if self.tc1 is not None or self.tc2:
            _Scratch.generation += 1
        self.tc1 = self.tc2 = None
        if TC_POLICY or (D >= TC_MIN_K and D % 4 == 0):
            self.tc1 = TcWeight(b.p("W1"), D, G * h, dev, transposed_only=not TC_POLICY)
            b.tc_weights.append(self.tc1)
        if TC_POLICY:
            self.tc2 = [TcWeight(b.p("W2", g * h * h), h, h, dev) for g in range(G)]
            b.tc_weights += self.tc2

    @staticmethod
    def specs(names, D, h, outs):
        G = len(names)
        s = [("W1", (D, G * h)), ("b1", (G * h,)), ("W2", (G, h, h)), ("b2", (G, h))]
        for g, o in zip(names, outs):
            s += [(f"W3.{g}", (h, o)), (f"b3.{g}", (o,))]
        return s

    def _fused_args(self):
        """Host-side pointer tables for ppx_mlp3_* (built once; bank addresses never change)."""
        if self._fa is None:
            G, b = self.G, self.bank
            ia, pa = (C.c_int * G), (C.c_void_p * G)
            outs = ia(*self.outs)
            ok = FUSED_ENABLED and L.call("ppx_mlp3_supported", self.D, self.h, G, outs) == 1
            tc = ok and MLP_TC_ENABLED and L.call("ppx_mlp3_tc_supported", self.D, self.h, G, outs) == 1
            self._fa = dict(ok=ok, tc=tc, outs=outs, W3=pa(*[b.p(f"W3.{g}") for g in self.names]),
                            b3=pa(*[b.p(f"b3.{g}") for g in self.names]),
                            dW3=pa(*[b.g(f"W3.{g}") for g in self.names]), db3=pa(*[b.g(f"b3.{g}") for g in self.names]))
        return self._fa

    def forward(self, x):
        M, G, h, D, b = x.shape[0], self.G, self.h, self.D, self.bank
        fa = self._fused_args()
        if fa["tc"]:                                            # tensor-core pair: opaque tile-transposed activations
            n_act = L.call("ppx_mlp3_tc_act_elems", M, h, G)
            H1 = self.scratch.get("pmlp.H1t", n_act)[:n_act]
            H2 = self.scratch.get("pmlp.H2t", n_act)[:n_act]
            outs = [self.scratch.get(f"pmlp.out.{g}", M * o)[:M * o].view(M, o) for g, o in zip(self.names, self.outs)]
            L.call("ppx_mlp3_tc_fwd", x.data_ptr(), x.stride(0), M, D, h, G, fa["outs"], b.p("W1"), b.p("b1"), b.p("W2"),
                   b.p("b2"), fa["W3"], fa["b3"], H1.data_ptr(), H2.data_ptr(),
                   (C.c_void_p * G)(*[o.data_ptr() for o in outs]), L.stream())
            self._saved = (x, H1, H2)
            return outs
        H1 = self.scratch.get("pmlp.H1", M * G * h)[:M * G * h].view(M, G * h)
        H2 = self.scratch.get("pmlp.H2", M * G * h)[:M * G * h].view(M, G * h)
        if fa["ok"]:
            outs = [self.scratch.get(f"pmlp.out.{g}", M * o)[:M * o].view(M, o) for g, o in zip(self.names, self.outs)]
            L.call("ppx_mlp3_fwd", x.data_ptr(), x.stride(0), M, D, h, G, fa["outs"], b.p("W1"), b.p("b1"), b.p("W2"),
                   b.p("b2"), fa["W3"], fa["b3"], H1.data_ptr(), H2.data_ptr(),
                   (C.c_void_p * G)(*[o.data_ptr() for o in outs]), L.stream())
            self._saved = (x, H1, H2)
            return outs
        dense_fwd(x.data_ptr(), x.stride(0), b.p("W1"), b.p("b1"), M, D, G * h, ACT["tanh"], H1.data_ptr(), G * h, self.tc1)
        if self.tc2 is not None and tc_ok(M, h, h, G * h, h, H1.data_ptr(), self.tc2[0].hiT.data_ptr()):
            for g in range(G):
                dense_fwd(H1.data_ptr() + g * h * F4, G * h, b.p("W2", g * h * h), b.p("b2", g * h), M, h, h, ACT["tanh"],
                          H2.data_ptr() + g * h * F4, G * h, self.tc2[g])
        else:
            linear_fwd(H1.data_ptr(), G * h, b.p("W2"), b.p("b2"), M, h, h, ACT["tanh"], H2.data_ptr(), G * h,
                       batch=G, sx=h, sw=h * h, sb=h, sy=h)
        outs = []
        for gi, (g, o) in enumerate(zip(self.names, self.outs)):
            y = self.scratch.get(f"pmlp.out.{g}", M * o)[:M * o].view(M, o)
            linear_fwd(H2.data_ptr() + gi * h * F4, G * h, b.p(f"W3.{g}"), b.p(f"b3.{g}"), M, h, o, ACT["none"],
                       y.data_ptr(), o)
            outs.append(y)
        self._saved = (x, H1, H2)
        return outs

    def fused(self):
        return self._fused_args()["ok"]

    def backward(self, d_outs, value_heads=None, clip_range=0.0, B_total=0, with_sumsq=False, adam=None):
        """d_outs[g]: [M, out_g] contiguous (None for a net listed in `value_heads`).  Fills bank.grad for every
        MLP parameter.  value_heads (fused path only): {g_index: (values, old_values, returns, branch_ptr, scale)}
        -- the clipped-value-loss gradient of that head is evaluated inside the backward kernel."""
        x, H1, H2 = self._saved
        M, G, h, D, b, sc = x.shape[0], self.G, self.h, self.D, self.bank, self.scratch
        fa = self._fused_args()
        if fa["ok"]:
            sfx = "_tc" if fa["tc"] else ""
            ws = sc.get("pmlp.fused_ws" + sfx, L.call(f"ppx_mlp3{sfx}_bwd_workspace", M, D, h, G, fa["outs"]))
            vh = None
            if value_heads:
                vh = (L.ValueHead * G)()
                for gi, (v, ov, R, br, scale) in value_heads.items():
                    vh[gi] = L.ValueHead(v.data_ptr(), ov.data_ptr(), R.data_ptr(), br, float(scale))
            dptr = (C.c_void_p * G)(*[(d.data_ptr() if d is not None else None) for d in d_outs])
            ss = None
            if with_sumsq:                                      # clip_grad_norm_ partials come out of the reduce kernel
                n_ss = L.call("ppx_mlp3_sumsq_partials", D, h, G, fa["outs"])
                ss = sc.get("pmlp.sumsq", n_ss, torch.float64)
                self.sumsq = (ss, n_ss)
            L.call(f"ppx_mlp3{sfx}_bwd", x.data_ptr(), x.stride(0), M, D, h, G, fa["outs"], b.p("W2"), fa["W3"], H1.data_ptr(),
                   H2.data_ptr(), dptr, vh, float(clip_range), int(B_total), b.g("W1"), b.g("b1"), b.g("W2"),
                   b.g("b2"), fa["dW3"], fa["db3"], ws.data_ptr(), ss.data_ptr() if ss is not None else None,
                   b.step_dev.data_ptr() if ss is not None else None, C.byref(adam) if adam is not None else None, L.stream())
            return
        assert not value_heads, "value_heads needs the fused MLP path"
        dP2 = sc.get("pmlp.dP2", M * G * h)[:M * G * h].view(M, G * h)
        dP1 = sc.get("pmlp.dP1", M * G * h)[:M * G * h].view(M, G * h)
        for gi, (g, o) in enumerate(zip(self.names, self.outs)):
            d = d_outs[gi]
            linear_bwd_weight(sc, H2.data_ptr() + gi * h * F4, G * h, d.data_ptr(), o, M, h, o, b.g(f"W3.{g}"),
                              b.g(f"b3.{g}"))
            linear_bwd_data(d.data_ptr(), o, b.p(f"W3.{g}"), M, h, o, H2.data_ptr() + gi * h * F4, G * h, ACT["tanh"],
                            dP2.data_ptr() + gi * h * F4, G * h)
        linear_bwd_weight(sc, H1.data_ptr(), G * h, dP2.data_ptr(), G * h, M, h, h, b.g("W2"), b.g("b2"),
                          batch=G, sx=h, sdy=h, sdw=h * h, sdb=h)
        if self.tc2 is not None and tc_ok(M, h, h, G * h, h, dP2.data_ptr(), self.tc2[0].hi.data_ptr()):
            for g in range(G):
                dense_bwd_data(dP2.data_ptr() + g * h * F4, G * h, b.p("W2", g * h * h), M, h, h, H1.data_ptr() + g * h * F4,
                               G * h, ACT["tanh"], dP1.data_ptr() + g * h * F4, G * h, self.tc2[g])
        else:
            linear_bwd_data(dP2.data_ptr(), G * h, b.p("W2"), M, h, h, H1.data_ptr(), G * h, ACT["tanh"], dP1.data_ptr(),
                            G * h, batch=G, sdy=h, sw=h * h, sh=h, sdx=h)
        linear_bwd_weight(sc, x.data_ptr(), x.stride(0), dP1.data_ptr(), G * h, M, D, G * h, b.g("W1"), b.g("b1"))


class Policy:
    """models.py:15-124.  `env` only needs .observation_space.shape and .action_space (class name
    "Discrete" with .n, or "Box" with .shape)."""

    def __init__(self, env, hidden_size, intrinsic_model=False, device="cuda"):
        self.env = env
        self.device = torch.device(device)
        self.state_dim = env.observation_space.shape[0]
        self.action_type = env.action_space.__class__.__name__
        self.action_dim = env.action_space.n if self.action_type == "Discrete" else env.action_space.shape[0]
        self.intrinsic = intrinsic_model
        self.hidden_size = hidden_size
        self.names = ["actor", "critic"] + (["int_critic"] if intrinsic_model else [])
        self.outs = [self.action_dim, 1] + ([1] if intrinsic_model else [])
        specs = ParallelMLP.specs(self.names, self.state_dim, hidden_size, self.outs)
        specs.append(("action_log_std", (self.action_dim,)))
        self.bank = ParamBank(specs, self.device)
        self.scratch = _Scratch(self.device)
        self.mlp = ParallelMLP(self.bank, self.names, self.state_dim, hidden_size, self.outs, self.scratch)
        self.net = self                                           # reference code reaches policy.net.parameters()
        self._sample_seed, self._draws = int(torch.initial_seed()) & 0x7FFFFFFFFFFFFFFF, 0
        self._eval_draws = 0                                      # stochastic predict / evaluate_policy calls (EVAL_DRAW)
        self._init_like_reference()

    # ---- initialisation / weight exchange ----
    def _init_like_reference(self):
        """models.py:141-154 / 177-195: construct actor, critic(, int_critic) Linears in order, then
        init_weights(): orthogonal(sqrt 2) weights and zero biases in module order."""
        lins = {}
        D, h = self.state_dim, self.hidden_size
        for g, o in zip(self.names, self.outs):
            lins[g] = [_TorchInit.linear(D, h), _TorchInit.linear(h, h), _TorchInit.linear(h, o)]
        for g in self.names:
            for lin in lins[g]:
                _TorchInit.orthogonal(lin)
        sd = {"action_log_std": torch.zeros(1, self.action_dim)}
        for g in self.names:
            for li, lin in zip((0, 2, 4), lins[g]):
                sd[f"{g}.{li}.weight"], sd[f"{g}.{li}.bias"] = lin.weight.detach(), lin.bias.detach()
        self.load_state_dict(sd)

    def load_state_dict(self, sd):
        """Accepts the reference's MlpNetwork / MlpIntrinsic state_dict (torch tensors or numpy)."""
        t = lambda a: torch.as_tensor(np.asarray(a) if not isinstance(a, torch.Tensor) else a).float()
        h, b = self.hidden_size, self.bank
        W1, b1, W2, b2 = b.view("W1"), b.view("b1"), b.view("W2"), b.view("b2")
        for gi, g in enumerate(self.names):
            W1[:, gi * h:(gi + 1) * h].copy_(_to_in_major(t(sd[f"{g}.0.weight"])))
            b1[gi * h:(gi + 1) * h].copy_(t(sd[f"{g}.0.bias"]))
            W2[gi].copy_(_to_in_major(t(sd[f"{g}.2.weight"])))
            b2[gi].copy_(t(sd[f"{g}.2.bias"]))
            b.view(f"W3.{g}").copy_(_to_in_major(t(sd[f"{g}.4.weight"])))
            b.view(f"b3.{g}").copy_(t(sd[f"{g}.4.bias"]))
        b.view("action_log_std").copy_(t(sd["action_log_std"]).reshape(-1))
        self.mlp.enable_tc()

    def state_dict(self, grad=False):
        h, b = self.hidden_size, self.bank
        v = lambda n: b.view(n, grad=grad).detach().cpu()
        sd = {"action_log_std": v("action_log_std").reshape(1, -1).clone()}
        for gi, g in enumerate(self.names):
            sd[f"{g}.0.weight"] = v("W1")[:, gi * h:(gi + 1) * h].t().contiguous()
            sd[f"{g}.0.bias"] = v("b1")[gi * h:(gi + 1) * h].clone()
            sd[f"{g}.2.weight"] = v("W2")[gi].t().contiguous()
            sd[f"{g}.2.bias"] = v("b2")[gi].clone()
            sd[f"{g}.4.weight"] = v(f"W3.{g}").t().contiguous()
            sd[f"{g}.4.bias"] = v(f"b3.{g}").clone()
        return sd

    def parameters(self):
        return [self.bank.flat]

    # ---- forward passes ----
    def forward_raw(self, obs):
        """obs [B,D] f32 CUDA -> (actor_out [B,A] (pre-tanh means / logits), values [B,1](, int_values [B,1]))."""
        return self.mlp.forward(obs)

    def _dist(self, actor_out):
        if self.action_type == "Discrete":
            return torch.distributions.Categorical(torch.softmax(actor_out, dim=-1))
        mean = torch.tanh(actor_out)
        return torch.distributions.Normal(mean, torch.exp(self.bank.view("action_log_std").expand_as(mean)))

    def act(self, obs):
        """models.py:30-50 / 75-99 (rollout side).  Forward on the fused kernels, then ONE launch builds the action
        distribution, draws an action per env and evaluates its log-probability (sample.cu; Philox stream keyed by the
        torch seed at construction, one draw number per call) -- no torch.distributions kernels, and `obs` may already
        be a CUDA tensor (e.g. from ppx VecNormalize), in which case nothing crosses the host here.  Returns CUDA tensors
        shaped like the reference's: actions [N,A] (Box, f64 as the buffer stores them) / [N] int64 (Discrete),
        log-probs [N,A] / [N], values [N]."""
        obs = torch.as_tensor(np.asarray(obs) if not isinstance(obs, torch.Tensor) else obs).to(self.device).float()
        outs = self.forward_raw(obs.contiguous())
        N, A = outs[0].shape
        discrete = self.action_type == "Discrete"
        actions = torch.empty((N,) if discrete else (N, A), dtype=torch.float64, device=self.device)
        lp = torch.empty((N,) if discrete else (N, A), dtype=torch.float32, device=self.device)
        self._draws += 1
        L.call("ppx_policy_sample", outs[0].data_ptr(), None if discrete else self.bank.p("action_log_std"), N, A, int(discrete),
               self._sample_seed, self._draws, actions.data_ptr(), lp.data_ptr(), L.stream())
        if discrete:
            actions = actions.long()
        vals = [o.squeeze(-1).clone() for o in outs[1:]]
        if self.intrinsic:
            return actions, vals[0], vals[1], lp
        return actions, vals[0], lp

    def act_into(self, obs, rollout):
        """`act` for an env that lives on the GPU, writing straight into rollout step `rollout.pos`: the forward, then ONE
        launch (collect.cu) that draws the actions exactly as `act` would (same Philox stream, same draw numbers) and writes
        the observation, f64 actions, log-probs and value(s) rows.  obs: CUDA f32 [N,D].  Returns the actions for env.step
        in a buffer of their own (Box f64 [N,A], Discrete int64 [N]; the env may modify it) and views of the value rows:
        (actions, values) or, intrinsic, (actions, values, int_values)."""
        if not obs.is_cuda or tuple(obs.shape) != (rollout.n_envs, self.state_dim):
            raise RuntimeError(f"act_into: observations must be a CUDA tensor [{rollout.n_envs}, {self.state_dim}], got "
                               f"{tuple(obs.shape)} on {obs.device}")
        obs = obs.float().contiguous()
        outs = self.forward_raw(obs)
        N, A = outs[0].shape
        discrete = self.action_type == "Discrete"
        p = rollout.pos
        env_actions = torch.empty((N,) if discrete else (N, A), dtype=torch.int64 if discrete else torch.float64, device=self.device)
        vals = [rollout.values[p]] + ([rollout.int_values[p]] if self.intrinsic else [])
        self._draws += 1
        L.call("ppx_policy_act_record", outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr() if self.intrinsic else None,
               None if discrete else self.bank.p("action_log_std"), obs.data_ptr(), N, A, self.state_dim, int(discrete),
               self._sample_seed, self._draws, rollout.observations[p].data_ptr(), rollout.actions[p].data_ptr(),
               rollout.action_log_probs[p].data_ptr(), vals[0].data_ptr(), vals[1].data_ptr() if self.intrinsic else None,
               env_actions.data_ptr(), L.stream())
        return (env_actions, *vals)

    # Draw numbers of the evaluation stream: bit 63 set (the training stream counts up from 1, so the two never meet), the
    # evaluation call (`_eval_draws`) in bits 32-62 and the step within the call in bits 0-31.
    EVAL_DRAW = 1 << 63

    def eval_actions(self, obs, deterministic, draw=0, row_offset=0, out=None):
        """The env-facing actions for `obs` (CUDA f32 [N, D], contiguous): one forward, then ONE launch (evaluate.cu) --
        deterministic: Box tanh(mean) f64 [N, A], Discrete the argmax of the logits int64 [N]; otherwise one draw from the
        policy's distribution with the Philox counter (row_offset + n, draw).  No rollout row, log-prob or value is written
        and neither draw counter moves.  `out`: the action buffer to write (default a new one)."""
        outs = self.forward_raw(obs)
        N, A = outs[0].shape
        discrete = self.action_type == "Discrete"
        if out is None:
            out = torch.empty((N,) if discrete else (N, A), dtype=torch.int64 if discrete else torch.float64, device=self.device)
        L.call("ppx_policy_act_eval", outs[0].data_ptr(), None if discrete else self.bank.p("action_log_std"), N, A, int(discrete),
               int(bool(deterministic)), self._sample_seed, int(draw), int(row_offset), out.data_ptr(), L.stream())
        return out

    def predict(self, obs, deterministic=True):
        """Actions for observations `obs` ([N, D] or one [D]; numpy or a CUDA tensor), on the side they came from: a CUDA
        tensor gives a CUDA tensor, anything else numpy.  Box: f64 [N, A] ([A] for one observation); Discrete: int64 [N]
        (a scalar array for one).  deterministic=True: the distribution's mode as `eval_actions` forms it.  deterministic=False:
        one draw from the evaluation stream, a Philox stream of its own -- the training stream (`_draws`) is not touched, so
        calling predict() changes nothing in a run that goes on training."""
        on_gpu = isinstance(obs, torch.Tensor) and obs.is_cuda
        x = obs if isinstance(obs, torch.Tensor) else torch.as_tensor(np.asarray(obs, dtype=np.float32))
        if x.dim() not in (1, 2) or x.shape[-1] != self.state_dim:
            raise ValueError(f"predict: observations must be [N, {self.state_dim}] or [{self.state_dim}], got {tuple(x.shape)}")
        single = x.dim() == 1
        x = x.reshape(-1, self.state_dim).to(self.device, torch.float32).contiguous()
        draw = 0
        if not deterministic:
            self._eval_draws += 1
            draw = self.EVAL_DRAW | (self._eval_draws << 32)
        a = self.eval_actions(x, deterministic, draw)
        if single:
            a = a[0]
        return a if on_gpu else a.cpu().numpy()

    def evaluate(self, obs, actions):
        """models.py:52-73 / 101-124 as plain tensors (train() uses the fused loss kernel instead)."""
        obs = torch.as_tensor(np.asarray(obs) if not isinstance(obs, torch.Tensor) else obs).to(self.device).float()
        actions = actions.to(self.device)
        outs = self.forward_raw(obs.contiguous())
        dist = self._dist(outs[0])
        if self.action_type == "Discrete":
            lp = dist.log_prob(actions.flatten()).unsqueeze(1)
        else:
            lp = dist.log_prob(actions)
        ent = dist.entropy()
        vals = [o.squeeze(-1).clone() for o in outs[1:]]
        if self.intrinsic:
            return vals[0], vals[1], lp, ent
        return vals[0], lp, ent


class RndNetwork:
    """models.py:216-267: predictor D-h-h-h-1 (LeakyReLU, LeakyReLU, ELU), frozen target D-h-h-1
    (LeakyReLU x2); constant init (target w=.01 b=1, predictor w=1 b=.01).  Only the predictor lives in
    the optimiser bank."""

    def __init__(self, input_size, hidden_size=32, device="cuda"):
        self.device = torch.device(device)
        D, h = input_size, hidden_size
        self.input_size, self.hidden_size = D, h
        self.p_layers = [(D, h, "leaky_relu"), (h, h, "leaky_relu"), (h, h, "elu"), (h, 1, "none")]
        self.t_layers = [(D, h, "leaky_relu"), (h, h, "leaky_relu"), (h, 1, "none")]
        self.bank = ParamBank(DenseStack.specs("predictor", self.p_layers), self.device)
        self.target_bank = ParamBank(DenseStack.specs("target", self.t_layers), self.device)
        self.scratch = _Scratch(self.device)
        self.predictor = DenseStack(self.bank, "predictor", self.p_layers, self.scratch)
        self.target = DenseStack(self.target_bank, "target", self.t_layers, self.scratch)
        # the reference still constructs default-initialised Linears first (RNG consumption), models.py:220-234
        for (i, o, _) in self.p_layers + self.t_layers:
            _TorchInit.linear(i, o)
        for i in range(len(self.p_layers)):
            self.bank.view(f"predictor.{2 * i}.weight").fill_(1.0)
            self.bank.view(f"predictor.{2 * i}.bias").fill_(0.01)
        for i in range(len(self.t_layers)):
            self.target_bank.view(f"target.{2 * i}.weight").fill_(0.01)
            self.target_bank.view(f"target.{2 * i}.bias").fill_(1.0)
        self.predictor.enable_tc()
        self.target.enable_tc()

    def load_state_dict(self, sd):
        t = lambda a: torch.as_tensor(np.asarray(a) if not isinstance(a, torch.Tensor) else a).float()
        for name, bank, n in (("predictor", self.bank, 4), ("target", self.target_bank, 3)):
            for i in range(n):
                bank.view(f"{name}.{2 * i}.weight").copy_(_to_in_major(t(sd[f"{name}.{2 * i}.weight"])))
                bank.view(f"{name}.{2 * i}.bias").copy_(t(sd[f"{name}.{2 * i}.bias"]))
        self.predictor.enable_tc()
        self.target.enable_tc()

    def state_dict(self):
        sd = {}
        for name, bank, n in (("predictor", self.bank, 4), ("target", self.target_bank, 3)):
            for i in range(n):
                sd[f"{name}.{2 * i}.weight"] = bank.view(f"{name}.{2 * i}.weight").detach().cpu().t().contiguous()
                sd[f"{name}.{2 * i}.bias"] = bank.view(f"{name}.{2 * i}.bias").detach().cpu().clone()
        return sd

    def forward(self, x, a_norm=None, tag=""):
        """x [M,D] f32 CUDA contiguous -> (predict [M,1], target [M,1]); keeps predictor activations.  `tag` names the
        activation scratch: the train path (captured in CUDA graphs) and the bonus path (other batch sizes) never share
        buffers, so growing one cannot leave the other's graph with a dangling pointer."""
        self._p_acts = self.predictor.forward(x, tag=tag, a_norm=a_norm)
        t_acts = self.target.forward(x, tag=tag, a_norm=a_norm)
        return self._p_acts[-1], t_acts[-1]

    __call__ = forward

    def int_reward(self, obs, rms=None):
        """models.py:261-267: (pred - target)^2, squeezed -> [M] f32 CUDA.  With `rms` (a RunningMeanStd), `obs` are RAW
        observations and normalize_obs (algorithms.py:111-118) is applied on the way: fused into the first layers'
        tensor-core kernels when they take that path (the observations are then read from HBM by those two kernels
        only), as a separate pass otherwise."""
        obs = torch.as_tensor(np.asarray(obs) if not isinstance(obs, torch.Tensor) else obs).to(self.device).float()
        obs = obs.reshape(-1, self.input_size).contiguous()
        a_norm = None
        if rms is not None:
            if TC_FUSE_NORM and self.predictor.can_fuse_norm(obs) and self.target.can_fuse_norm(obs):
                a_norm = (rms.mean_dev.data_ptr(), rms.istd().data_ptr(), 5.0)
            else:
                from .util import normalize_obs
                obs = normalize_obs(obs, rms)
        pred, tgt = self.forward(obs, a_norm, tag=".bonus")
        r = torch.empty(obs.shape[0], dtype=torch.float32, device=self.device)
        L.call("ppx_rnd_sqerr", pred.data_ptr(), tgt.data_ptr(), obs.shape[0], r.data_ptr(), L.stream())
        return r

    def train_step(self, x, loss_accum, B_total=0):
        """MSE(pred, target) forward+backward into bank.grad (algorithms.py:495-500).  x already normalised.
        Sharded: B_total = rows of the global minibatch, so the mean (and its gradient) is global."""
        pred, tgt = self.forward(x, tag=".train")
        M = x.shape[0]
        d_pred = self.scratch.get("rnd.dpred", M)[:M].view(M, 1)
        L.call("ppx_mse_fwd_bwd", pred.data_ptr(), tgt.data_ptr(), M, float(M) / float(B_total) if B_total else 1.0,
               d_pred.data_ptr(), None,
               loss_accum.data_ptr(), L.stream())
        self.predictor.backward(self._p_acts, d_pred)


class ActionConverter:
    """util.py:47-78 (shape contract only)."""

    def __init__(self, action_space):
        self.action_type = action_space.__class__.__name__
        if self.action_type == "Discrete":
            self.num_actions, self.action_output = action_space.n, 1
        elif self.action_type == "Box":
            self.num_actions = action_space.shape[0]
            self.action_output = self.num_actions


class IntrinsicCuriosityModule:
    """models.py:270-320: state encoder D-h-f, forward model (n+f)-h-f, inverse model 2f-h-n,
    action encoder Embedding(n,n) / Linear(n,n); f = h; orthogonal(sqrt 2) Linears."""

    def __init__(self, input_size, action_converter, hidden_size, device="cuda"):
        self.device = torch.device(device)
        self.action_converter = action_converter
        self.discrete = action_converter.action_type == "Discrete"
        D, h = input_size, hidden_size
        f, n = hidden_size, action_converter.num_actions
        self.input_size, self.feature_size, self.n_actions, self.hidden = D, f, n, h
        self.enc_layers = [(D, h, "leaky_relu"), (h, f, "none")]
        self.fwd_layers = [(n + f, h, "leaky_relu"), (h, f, "none")]
        self.inv_layers = [(2 * f, h, "leaky_relu"), (h, n, "none")]
        specs = (DenseStack.specs("state_encoder", self.enc_layers) + DenseStack.specs("forward_model", self.fwd_layers)
                 + DenseStack.specs("inverse_model", self.inv_layers))
        specs += [("action_encoder.weight", (n, n))] + ([] if self.discrete else [("action_encoder.bias", (n,))])
        self.bank = ParamBank(specs, self.device)
        self.scratch = _Scratch(self.device)
        self.enc = DenseStack(self.bank, "state_encoder", self.enc_layers, self.scratch)
        self.fwd = DenseStack(self.bank, "forward_model", self.fwd_layers, self.scratch)
        self.inv = DenseStack(self.bank, "inverse_model", self.inv_layers, self.scratch)
        self._init_like_reference()

    def _init_like_reference(self):
        order = [("state_encoder", self.enc_layers), ("forward_model", self.fwd_layers), ("inverse_model", self.inv_layers)]
        lins = [(name, i, _TorchInit.linear(K, N)) for name, layers in order for i, (K, N, _) in enumerate(layers)]
        n = self.n_actions
        sd = {}
        if self.discrete:
            emb = torch.nn.Embedding(n, n)
        else:
            emb = _TorchInit.linear(n, n)
        for name, i, lin in lins:                                   # init_weights(): module order, Linears only
            _TorchInit.orthogonal(lin)
            sd[f"{name}.{2 * i}.weight"], sd[f"{name}.{2 * i}.bias"] = lin.weight.detach(), lin.bias.detach()
        if not self.discrete:
            _TorchInit.orthogonal(emb)
            sd["action_encoder.bias"] = emb.bias.detach()
        sd["action_encoder.weight"] = emb.weight.detach()
        self.load_state_dict(sd)

    def load_state_dict(self, sd):
        t = lambda a: torch.as_tensor(np.asarray(a) if not isinstance(a, torch.Tensor) else a).float()
        for name, layers in (("state_encoder", self.enc_layers), ("forward_model", self.fwd_layers),
                             ("inverse_model", self.inv_layers)):
            for i in range(len(layers)):
                self.bank.view(f"{name}.{2 * i}.weight").copy_(_to_in_major(t(sd[f"{name}.{2 * i}.weight"])))
                self.bank.view(f"{name}.{2 * i}.bias").copy_(t(sd[f"{name}.{2 * i}.bias"]))
        if self.discrete:
            self.bank.view("action_encoder.weight").copy_(t(sd["action_encoder.weight"]))      # table [n, n]
        else:
            self.bank.view("action_encoder.weight").copy_(_to_in_major(t(sd["action_encoder.weight"])))
            self.bank.view("action_encoder.bias").copy_(t(sd["action_encoder.bias"]))
        for st in (self.enc, self.fwd, self.inv):
            st.enable_tc()

    def state_dict(self):
        sd = {}
        for name, layers in (("state_encoder", self.enc_layers), ("forward_model", self.fwd_layers),
                             ("inverse_model", self.inv_layers)):
            for i in range(len(layers)):
                sd[f"{name}.{2 * i}.weight"] = self.bank.view(f"{name}.{2 * i}.weight").detach().cpu().t().contiguous()
                sd[f"{name}.{2 * i}.bias"] = self.bank.view(f"{name}.{2 * i}.bias").detach().cpu().clone()
        w = self.bank.view("action_encoder.weight").detach().cpu()
        sd["action_encoder.weight"] = w.clone() if self.discrete else w.t().contiguous()
        if not self.discrete:
            sd["action_encoder.bias"] = self.bank.view("action_encoder.bias").detach().cpu().clone()
        return sd

    # ---- pieces shared by int_reward and the training forward ----
    def _encode_action(self, action, M, out, ldo):
        """action_encoder into columns [0,n) of `out` (leading dim ldo).  Discrete: ids (f64 or i64, one per
        row); Box: f32 [M,n]."""
        n = self.n_actions
        if self.discrete:
            ids = action.reshape(-1).contiguous()
            is_f64 = ids.dtype == torch.float64
            if not is_f64:
                ids = ids.long()
            L.call("ppx_embedding_fwd", self.bank.p("action_encoder.weight"), n, ids.data_ptr(), int(is_f64), 1, M,
                   out, ldo, L.stream())
            return ids
        a = action.float().reshape(M, n).contiguous()
        linear_fwd(a.data_ptr(), n, self.bank.p("action_encoder.weight"), self.bank.p("action_encoder.bias"), M, n, n,
                   ACT["none"], out, ldo)
        return a

    def int_reward(self, state, next_state, action, rewards=None, eta=0.0):
        """models.py:311-320 (+ the reward blend of algorithms.py:630 when `rewards` is given, in place)."""
        dev, f, n = self.device, self.feature_size, self.n_actions
        s = torch.as_tensor(np.asarray(state) if not isinstance(state, torch.Tensor) else state).to(dev).float().contiguous()
        ns = torch.as_tensor(np.asarray(next_state) if not isinstance(next_state, torch.Tensor) else next_state).to(dev).float().contiguous()
        action = action.to(dev) if isinstance(action, torch.Tensor) else torch.as_tensor(np.asarray(action)).to(dev)
        M = s.shape[0]
        both = self.scratch.get("icm.both", 2 * M * self.input_size)[:2 * M * self.input_size].view(2 * M, self.input_size)
        both[:M].copy_(s)
        both[M:].copy_(ns)
        feats = self.enc.forward(both, tag=".bonus")[-1]                         # [2M, f]: phi(s) ; phi(s')
        fin = self.scratch.get("icm.bonus.fin", M * (f + n))[:M * (f + n)].view(M, f + n)
        fin[:, :f].copy_(feats[:M])
        self._encode_action(action, M, fin.data_ptr() + f * F4, f + n)
        pred = self.fwd.forward(fin, tag=".bonus")[-1]
        ri = torch.empty(M, dtype=torch.float32, device=dev)
        L.call("ppx_icm_bonus_tail", pred.data_ptr(), feats[M:].data_ptr(), M, f, float(eta),
               rewards.data_ptr() if rewards is not None else None, ri.data_ptr(), L.stream())
        return ri

    def train_step(self, obs, actions, beta, loss_accum, pairs_total=None):
        """Forward (models.py:300-309) + 0.8*inverse + 0.2*forward loss (algorithms.py:684-688) + backward into
        bank.grad, on the shuffled-consecutive rows obs[:-1] -> obs[1:], actions[:-1].  Sharded: `obs` holds this
        rank's slice of the global minibatch (plus its halo row) and `pairs_total` the pairs of the whole minibatch,
        so the means -- and their gradients -- are the global ones once summed over the ranks."""
        f, n, D = self.feature_size, self.n_actions, self.input_size
        B = obs.shape[0]
        M = B - 1
        share = 1.0 if not pairs_total else float(M) / float(pairs_total)
        sc = self.scratch
        feats_acts = self.enc.forward(obs, tag=".train")                         # encoder once over all B rows
        feats = feats_acts[-1]                                                   # [B, f]
        s_ft, ns_ft = feats[:M], feats[1:]
        fin = sc.get("icm.fin", M * (f + n))[:M * (f + n)].view(M, f + n)
        iin = sc.get("icm.iin", M * 2 * f)[:M * 2 * f].view(M, 2 * f)
        fin[:, :f].copy_(s_ft)
        iin[:, :f].copy_(s_ft)
        iin[:, f:].copy_(ns_ft)
        act_in = self._encode_action(actions[:M], M, fin.data_ptr() + f * F4, f + n)
        fwd_acts = self.fwd.forward(fin, tag=".train")
        inv_acts = self.inv.forward(iin, tag=".train")
        ns_hat, a_hat = fwd_acts[-1], inv_acts[-1]
        # losses + gradients w.r.t. the three heads
        d_ns_hat = sc.get("icm.d_ns_hat", M * f)[:M * f].view(M, f)
        d_ns_ft = sc.get("icm.d_ns_ft", M * f)[:M * f].view(M, f)
        d_a_hat = sc.get("icm.d_a_hat", M * n)[:M * n].view(M, n)
        ns_c = sc.get("icm.ns_c", M * f)[:M * f].view(M, f)
        ns_c.copy_(ns_ft)
        L.call("ppx_mse_fwd_bwd", ns_c.data_ptr(), ns_hat.data_ptr(), M * f, float(beta) * share, d_ns_ft.data_ptr(),
               d_ns_hat.data_ptr(), loss_accum.data_ptr(), L.stream())
        if self.discrete:
            tgt = actions[:M].reshape(-1).double().contiguous()
            L.call("ppx_xent_fwd_bwd", a_hat.data_ptr(), tgt.data_ptr(), 1, M, n, float(1 - beta) * share, d_a_hat.data_ptr(),
                   loss_accum.data_ptr(), L.stream())
        else:
            tgt = actions[:M].float().reshape(M, n).contiguous()
            L.call("ppx_mse_fwd_bwd", a_hat.data_ptr(), tgt.data_ptr(), M * n, float(1 - beta) * share, d_a_hat.data_ptr(),
                   None, loss_accum.data_ptr(), L.stream())
        # backward through the two heads down to their inputs
        d_fin = self.fwd.backward(fwd_acts, d_ns_hat, need_dx=True)              # [M, f+n]
        d_iin = self.inv.backward(inv_acts, d_a_hat, need_dx=True)               # [M, 2f]
        # action encoder gradient
        if self.discrete:
            d_act = d_fin[:, f:].contiguous()
            L.call("ppx_embedding_bwd", d_act.data_ptr(), n, act_in.data_ptr(), int(act_in.dtype == torch.float64), 1, M,
                   n, self.bank.g("action_encoder.weight"), L.stream())
        else:
            d_act = d_fin[:, f:].contiguous()
            linear_bwd_weight(sc, act_in.data_ptr(), n, d_act.data_ptr(), n, M, n, n, self.bank.g("action_encoder.weight"),
                              self.bank.g("action_encoder.bias"))
        # gradient w.r.t. the encoder output rows: row i gets s_ft grads (i < M) and ns_ft grads (i >= 1)
        d_feats = sc.get("icm.d_feats", B * f)[:B * f].view(B, f)
        d_feats.zero_()
        d_feats[:M].add_(d_fin[:, :f]).add_(d_iin[:, :f])
        d_feats[1:].add_(d_iin[:, f:]).add_(d_ns_ft)
        self.enc.backward(feats_acts, d_feats)
