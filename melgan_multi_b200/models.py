"""Drop-in replacement for the reference's ``models`` module (/root/reference/models.py).

``train.py:13`` does ``from models import Generator, MultiScaleDiscriminator, feature_loss,
generator_loss, discriminator_loss``; this module exports the same five names with the same
constructor and ``forward`` signatures, the same ``state_dict`` keys, shapes and parameter
registration order (so reference checkpoints and Adam state load, SURVEY 8b), and leaves
``weight_g`` / ``weight_v`` / ``bias`` as ordinary leaf parameters so the reference's gradient
all-reduce wrapper (distributed.py:90-142) hooks them unchanged.

What runs where
  * ``Generator.forward`` (models.py:61-71 in the reference): eight hand-written sm_100a tcgen05 kernels in
    libmelgan_b200.so -- conv_pre, then LeakyReLU -> ConvTranspose1d and the fused six-conv ResBlock of each stage,
    the last stage as ONE kernel (its stride-2 ConvT, the ResBlock and LeakyReLU -> conv_post -> tanh) -- plus one launch that folds weight-norm for all 30 layers
    whenever the parameters changed.  CUDA only; a CPU tensor raises (the reference's CPU path lives in oracle/ as
    test infrastructure).
  * ``MultiScaleDiscriminator.forward`` (models.py:119-135, Discriminator.forward :87-103) on CUDA: real and generated
    audio are stacked into one batch and run through hand-written kernels -- AvgPool chain fused into each scale's
    conv_pre, grouped k41 convs and conv_post1 on tcgen05 -- after one launch that folds weight-norm for the 21 layers.
  * ``feature_loss`` / ``generator_loss`` / ``discriminator_loss`` (models.py:138-167) on CUDA tensors: every term of a
    loss is a row of one fused reduction launch (forward) and one gradient launch (backward).
  * Backward: the generator's runs as recomputation through stock PyTorch ops; the discriminators' walks the saved
    feature maps layer by layer on hand-written kernels only (grouped convs, conv_post1 dgrad / wgrad on tcgen05,
    conv_pre / conv_post2, LeakyReLU, weight-norm): no cuDNN call in a discriminator's backward.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import AvgPool1d, Conv1d, ConvTranspose1d
from torch.nn.utils import weight_norm

from . import engine as _engine
from .synth import DISCRIMINATOR_LAYERS, GENERATOR_LAYERS

_RES_DILATIONS = (1, 3, 9)


def get_padding(kernel_size, dilation=1):
    """'same' padding for an odd kernel (reference models.py:8-9)."""
    return (kernel_size * dilation - dilation) // 2


def _wn_conv(cin, cout, k, **kw):
    return weight_norm(Conv1d(cin, cout, k, **kw))


class ResBlock(nn.Module):
    """Parameter container with the reference's layout (models.py:12-30).  ``forward`` is the stock
    PyTorch restatement used only by the autograd (backward) path."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.convs1 = nn.ModuleList(
            [_wn_conv(in_channels, out_channels, 3, dilation=d, padding=get_padding(3, d)) for d in _RES_DILATIONS])
        self.convs2 = nn.ModuleList(
            [_wn_conv(in_channels, out_channels, 3, dilation=1, padding=get_padding(3, 1)) for _ in _RES_DILATIONS])

    def forward(self, x):
        for first, second in zip(self.convs1, self.convs2):
            x = second(F.leaky_relu(first(F.leaky_relu(x)))) + x
        return x


def _layer_modules(gen):
    """The 30 weight-normed modules of a Generator in reference registration order."""
    mods = [gen.conv_pre] + list(gen.ups)
    for rb in gen.resblocks:
        mods += list(rb.convs1) + list(rb.convs2)
    mods.append(gen.conv_post)
    return mods


class _GeneratorFunction(torch.autograd.Function):
    """Forward on the fused sm_100a kernels; backward by recomputation through stock PyTorch ops (open row: native
    backward).  The recomputation -- 30 convs forward, their backward, weight-norm: ~600 launches that cost the host more
    than the GPU -- is captured ONCE per input shape as a pair of CUDA graphs (torch.cuda.make_graphed_callables) and
    replayed, so the step is no longer bound by eager launch overhead (MG_GEN_BWD_GRAPH=0: eager).
    Inputs: mel, then 30 x (weight_v, weight_g, bias)."""

    @staticmethod
    def forward(ctx, gen, mel, *params):
        ctx.gen = gen
        ctx.save_for_backward(mel, *params)
        ctx.graphed = gen._graphed_recompute(mel, params)  # built here (not inside backward): capture needs a quiet device
        return gen._engine_forward(mel)

    @staticmethod
    def backward(ctx, grad_out):
        gen = ctx.gen
        mel, *params = ctx.saved_tensors
        need_mel = ctx.needs_input_grad[1]
        with torch.enable_grad():
            mel_ = mel.detach().requires_grad_(need_mel)
            leaves = [p.detach().requires_grad_(True) for p in params]
            if ctx.graphed is not None and need_mel == ctx.graphed[1]:
                y = ctx.graphed[0](mel_, *leaves)
            else:
                y = gen._torch_forward(mel_, leaves)
            wanted = ([mel_] if need_mel else []) + leaves
            grads = torch.autograd.grad(y, wanted, grad_out.contiguous(), allow_unused=True)
        grads = list(grads)
        gmel = grads.pop(0) if need_mel else None
        return (None, gmel, *grads)


class Generator(nn.Module):
    """mel [B, 80, T] fp32 CUDA -> audio [B, 1, 256*T] (reference models.py:43-71)."""

    def __init__(self):
        super().__init__()
        self.conv_pre = _wn_conv(80, 512, 7, padding=3)
        self.ups = nn.ModuleList([
            weight_norm(ConvTranspose1d(cin, cout, k, k // 2, padding=k // 4))
            for _n, kind, cin, cout, k in GENERATOR_LAYERS if kind == "convT"])
        self.resblocks = nn.ModuleList([ResBlock(c, c) for c in (256, 128, 64, 32)])
        self.conv_post = _wn_conv(32, 1, 7, padding=3)
        self._dev = None          # engine.GeneratorDevice, created lazily on the parameters' device
        self._packed_key = None   # (data_ptr, _version) of every parameter at the last pack

    # -- parameter plumbing -----------------------------------------------------------------
    def _param_triplets(self):
        mods = _layer_modules(self)
        return [m.weight_v for m in mods], [m.weight_g for m in mods], [m.bias for m in mods]

    def _ensure_packed(self):
        vs, gs, bs = self._param_triplets()
        dev = vs[0].device
        if dev.type != "cuda":
            raise _engine.EngineError(
                "melgan_multi_b200.Generator runs on CUDA (sm_100a) only; move the module with .to('cuda'). "
                "There is deliberately no CPU fallback.")
        if self._dev is None or self._dev.device != dev:
            self._dev = _engine.GeneratorDevice(dev)
            self._packed_key = None
        key = tuple((t.data_ptr(), t._version) for t in vs + gs + bs)
        if key != self._packed_key:
            self._dev.pack(vs, gs, bs)
            self._packed_key = key
        return self._dev

    def _engine_forward(self, mel):
        return self._ensure_packed().forward(mel)

    def _graphed_recompute(self, mel, params):
        """(graphed stock-op forward+backward, mel_requires_grad) for this input shape, or None.  Cached per shape / dtype
        policy; the graphs own static copies of nothing but activations -- parameters are call arguments."""
        import os
        if os.environ.get("MG_GEN_BWD_GRAPH", "1") == "0" or torch.cuda.is_current_stream_capturing():
            return None
        need_mel = bool(mel.requires_grad)
        key = (tuple(mel.shape), mel.device, need_mel, torch.backends.cudnn.conv.fp32_precision, torch.backends.cudnn.benchmark)
        cache = self.__dict__.setdefault("_bwd_graphs", {})
        if key not in cache:
            if len(cache) >= 4:  # shapes keep changing (e.g. whole-utterance validation): stay eager for new ones
                return None
            sample = [mel.detach().clone().requires_grad_(need_mel)] + [p.detach().clone().requires_grad_(True) for p in params]
            try:
                with torch.enable_grad():  # (we are inside autograd.Function.forward, where grad mode is off)
                    fn = torch.cuda.make_graphed_callables(lambda m, *leaves: self._torch_forward(m, list(leaves)), tuple(sample))
            except Exception:  # capture refused (e.g. allocator / library state): the eager recompute still works
                fn = None
            cache[key] = fn
        return (cache[key], need_mel) if cache[key] is not None else None

    # -- stock-PyTorch restatement, used ONLY to differentiate (backward) ---------------------
    def _torch_forward(self, x, leaves):
        # (the same graph on channels_last 4-D tensors through conv2d saves cuDNN's nchw<->nhwc conversions -- 0.7 ms eager,
        #  ~0.2 ms under the CUDA graph, scripts/gen_bwd_layout_ab.py -- but picks TF32 kernels whose rounding puts the deepest
        #  layers' weight_g gradients AT the 5e-3 digest tolerance of tests/test_train_gpu.py on the small case: not taken)
        ws = [torch._weight_norm(leaves[3 * i], leaves[3 * i + 1], 0) for i in range(30)]
        bs = [leaves[3 * i + 2] for i in range(30)]
        x = F.conv1d(x, ws[0], bs[0], padding=3)
        for i in range(4):
            k = ws[1 + i].shape[2]
            x = F.conv_transpose1d(F.leaky_relu(x), ws[1 + i], bs[1 + i], stride=k // 2, padding=k // 4)
            for j, d in enumerate(_RES_DILATIONS):
                a, b = 5 + 6 * i + j, 5 + 6 * i + 3 + j
                h = F.conv1d(F.leaky_relu(x), ws[a], bs[a], padding=d, dilation=d)
                x = F.conv1d(F.leaky_relu(h), ws[b], bs[b], padding=1) + x
        return torch.tanh(F.conv1d(F.leaky_relu(x), ws[29], bs[29], padding=3))

    def forward(self, x, lengths=None):
        """lengths (optional): ragged batch -- one mel length in [1, T] per item (list, tuple or integer tensor; a CUDA
        tensor costs one host synchronisation to read).  Item b is then x[b, :, :lengths[b]]; its audio fills the first
        256 * lengths[b] samples, bit-identical to a forward of that item alone, and is exactly 0 after them.  Inference
        only: a call that would need autograd raises EngineError (training uses fixed-length segments)."""
        if not x.is_cuda:
            raise _engine.EngineError("melgan_multi_b200.Generator.forward needs a CUDA tensor (no CPU fallback)")
        if x.dtype != torch.float32:
            x = x.float()
        vs, gs, bs = self._param_triplets()
        needs_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in vs + gs + bs))
        if lengths is not None:
            if needs_grad:
                raise _engine.EngineError("Generator.forward(x, lengths): ragged batches are inference-only; call it under "
                                          "torch.no_grad() / torch.inference_mode() or with parameters that need no grad")
            return self._ensure_packed().forward(x, lengths=lengths)
        if not needs_grad:
            return self._engine_forward(x)
        flat = []
        for v, g, b in zip(vs, gs, bs):
            flat += [v, g, b]
        return _GeneratorFunction.apply(self, x, *flat)


class Discriminator(nn.Module):
    """One discriminator (reference models.py:74-103).  Inside ``MultiScaleDiscriminator`` (its only caller in the
    reference, models.py:109-113) the three of them run as one fused pipeline on the stacked real + generated batch;
    called on its own, ``forward(x)`` runs the same sm_100a kernels on this module's weights and returns
    ``(flattened logits, [7 feature maps])`` like the reference's.  CUDA only, no stock-op fallback."""

    def __init__(self):
        super().__init__()
        spec = {n: (cin, cout, k, s, g, p) for n, cin, cout, k, s, g, p in DISCRIMINATOR_LAYERS}
        def mk(n):
            cin, cout, k, s, g, p = spec[n]
            return weight_norm(Conv1d(cin, cout, k, s, groups=g, padding=p))
        self.conv_pre = mk("conv_pre")
        self.grouped_convs = nn.ModuleList([mk("grouped_convs.%d" % i) for i in range(4)])
        self.conv_post1 = mk("conv_post1")
        self.conv_post2 = mk("conv_post2")

    def layers(self):
        return [self.conv_pre] + list(self.grouped_convs) + [self.conv_post1, self.conv_post2]

    meanpools = ()   # what _MSDFunction walks for scale 0: no pooling

    def _param_triplets(self):
        mods = self.layers()
        return [m.weight_v for m in mods], [m.weight_g for m in mods], [m.bias for m in mods]

    def _engine_forward(self, x):
        vs, gs, bs = self._param_triplets()
        dev = vs[0].device
        if getattr(self, "_dev", None) is None or self._dev.device != dev:
            self._dev = _engine.DiscriminatorDevice(dev, ndisc=1)
            self._packed_key = None
        key = tuple((t.data_ptr(), t._version) for t in vs + gs + bs)
        if key != self._packed_key:
            self._dev.pack(vs, gs, bs)
            self._packed_key = key
        return self._dev.forward(x)

    def forward(self, x):
        if not x.is_cuda:
            raise _engine.EngineError("melgan_multi_b200.Discriminator.forward needs a CUDA tensor (no CPU fallback)")
        x = x.float()
        vs, gs, bs = self._param_triplets()
        needs_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in vs + gs + bs))
        if needs_grad:
            flat = []
            for v, g, b in zip(vs, gs, bs):
                flat += [v, g, b]
            fmap = list(_MSDFunction.apply(self, 0, {}, x, *flat))
        else:
            fmap = self._engine_forward(x)[0]
        return torch.flatten(fmap[6], 1, -1), fmap


class _MSDFunction(torch.autograd.Function):
    """ONE discriminator of the stack as an autograd node: forward on the fused sm_100a kernels, backward layer by layer on
    the saved feature maps without recomputing the forward -- the grouped k41 convs (layers 1..4) and weight-norm on the
    hand-written kernels of csrc/mg_disc_bwd.cu (cuDNN launches one kernel per group for them), conv_post1 (88 % of the
    FLOPs) on the tcgen05 kernels of csrc/mg_conv_tc.cu (dgrad, transposed weight copy) and csrc/mg_wgrad_tc.cu (wgrad),
    conv_pre / conv_post2 on the bandwidth-bound kernels of csrc/mg_disc_edge_bwd.cu.  No aten / cuDNN call is left.

    The three scales of a MultiScaleDiscriminator are three nodes that share one forward: the first node to run launches the
    whole fused stack (real and generated stacked as one batch, the scales on forked streams) and parks the feature maps
    in ``cache``; the other two pick theirs up.  Separate nodes mean each discriminator's parameter gradients exist as soon
    as ITS backward is done, so the data-parallel wrapper (distributed.py) all-reduces them while the other scales'
    backward is still running.
    Inputs: scale index, cache dict, stacked audio [2B,1,L], then 7 x (weight_v, weight_g, bias) of that discriminator;
    outputs: its 7 feature maps."""

    @staticmethod
    def forward(ctx, host, s, cache, y2, *params):
        ctx.host, ctx.s = host, s
        if "fmaps" not in cache:
            cache["fmaps"] = host._engine_forward(y2)
        fm = tuple(cache["fmaps"][s])
        ctx.save_for_backward(y2, *params, *fm)
        return fm

    @staticmethod
    def backward(ctx, *grads):
        host, s, dev = ctx.host, ctx.s, ctx.host._dev
        saved = ctx.saved_tensors
        y2, params, fm = saved[0], saved[1:22], saved[22:]
        need_y = ctx.needs_input_grad[3]
        x0 = y2
        for k in range(s):  # the scale's input: the AvgPool chain of models.py:114-117,125-127
            x0 = host.meanpools[k](x0)
        # one host call walks the seven layers and enqueues every kernel (csrc/mg_disc_bwd_chain.cu): LeakyReLU', grouped convs,
        # conv_post1 dgrad / wgrad on tcgen05, conv_pre / conv_post2 -- the step was bound by per-kernel Python launches
        g, dws, dbs = dev.scale_backward(s, x0, fm, grads, need_y)
        gy = None
        if need_y and g is not None:  # back through the (linear) AvgPool chain: differentiate it on zeros
            gy = g
            lens = [y2.shape[2], y2.shape[2] // 2 + 1]  # input lengths of pools 0, 1: AvgPool1d(4, 2, pad 2) gives L // 2 + 1
            for k in range(s - 1, -1, -1):
                with torch.enable_grad():
                    a = torch.zeros((y2.shape[0], 1, lens[k]), dtype=y2.dtype, device=y2.device).requires_grad_(True)
                    (gy,) = torch.autograd.grad(host.meanpools[k](a), a, gy)
        dvs, dgs = dev.wn_backward([params[3 * l] for l in range(7)], [params[3 * l + 1] for l in range(7)], dws)
        out = []
        for l in range(7):
            out += [dvs[l], dgs[l], dbs[l]]
        return (None, None, None, gy, *out)


class MultiScaleDiscriminator(nn.Module):
    """Reference models.py:106-135: three Discriminators on y, pool(y), pool(pool(y)); returns
    (y_d_rs, y_d_gs, fmap_rs, fmap_gs).  On CUDA the whole stack runs in the hand-written kernels of
    libmelgan_b200.so with y and y_hat stacked into one batch (the reference calls each discriminator twice)."""

    def __init__(self):
        super().__init__()
        self.discriminators = nn.ModuleList([Discriminator() for _ in range(3)])
        self.meanpools = nn.ModuleList([AvgPool1d(4, 2, padding=2), AvgPool1d(4, 4, padding=2)])
        self._dev = None
        self._packed_key = None

    def _param_triplets(self):
        mods = [m for d in self.discriminators for m in d.layers()]
        return [m.weight_v for m in mods], [m.weight_g for m in mods], [m.bias for m in mods]

    def _engine_forward(self, y2):
        vs, gs, bs = self._param_triplets()
        dev = vs[0].device
        if self._dev is None or self._dev.device != dev:
            self._dev = _engine.DiscriminatorDevice(dev)
            self._packed_key = None
        key = tuple((t.data_ptr(), t._version) for t in vs + gs + bs)
        if key != self._packed_key:
            self._dev.pack(vs, gs, bs)
            self._packed_key = key
        return self._dev.forward(y2)

    # -- stock-PyTorch restatement on folded weights, used ONLY to differentiate (backward) -----------------
    def _torch_forward(self, y2, leaves):
        outs = []
        x_in = y2
        for s in range(3):
            if s > 0:
                x_in = self.meanpools[s - 1](x_in)
            x = x_in
            for l, (_n, _cin, _cout, _k, stride, groups, pad) in enumerate(DISCRIMINATOR_LAYERS):
                i = 3 * (7 * s + l)
                w = torch._weight_norm(leaves[i], leaves[i + 1], 0)
                x = F.conv1d(x, w, leaves[i + 2], stride=stride, padding=pad, groups=groups)
                if l < 6:
                    x = F.leaky_relu(x)
                outs.append(x)
        return outs

    def forward(self, y, y_hat):
        if not (y.is_cuda and y_hat.is_cuda):
            raise _engine.EngineError(
                "melgan_multi_b200.MultiScaleDiscriminator.forward needs CUDA tensors (no CPU fallback)")
        B = y.shape[0]
        y2 = torch.cat([y, y_hat], dim=0).float()
        vs, gs, bs = self._param_triplets()
        needs_grad = torch.is_grad_enabled() and (y2.requires_grad or any(p.requires_grad for p in vs + gs + bs))
        if needs_grad:
            cache, fmaps = {}, []
            for s in range(3):  # three autograd nodes, one fused forward launch (see _MSDFunction)
                flat = []
                for i in range(7 * s, 7 * s + 7):
                    flat += [vs[i], gs[i], bs[i]]
                fmaps.append(list(_MSDFunction.apply(self, s, cache, y2, *flat)))
        else:
            fmaps = self._engine_forward(y2)
        # The reference's four lists.  Every element is an ordinary autograd slice of the stacked map (any use of it
        # differentiates correctly), and is also tagged with the stacked tensor it is a half of: the package's own loss
        # functions then work on the stacked tensors directly -- one gradient tensor per map instead of two zero-padded
        # slice gradients and their sum (SliceBackward + add_: ~1000 launches and 3 ms per training step).
        def half(f, h, flat=False):
            t = f[h * B:(h + 1) * B]
            if flat:
                t = torch.flatten(t, 1, -1)
            t._mg_half = (f, h)
            return t
        y_d_rs, y_d_gs, fmap_rs, fmap_gs = [], [], [], []
        for s in range(3):
            fmap_rs.append([half(f, 0) for f in fmaps[s]])
            fmap_gs.append([half(f, 1) for f in fmaps[s]])
            y_d_rs.append(half(fmaps[s][6], 0, True))
            y_d_gs.append(half(fmaps[s][6], 1, True))
        return y_d_rs, y_d_gs, fmap_rs, fmap_gs


class _LossRows(torch.autograd.Function):
    """Row means of a loss table on the fused kernels (csrc/mg_loss.cu): forward = one reduction launch over every row +
    a fixed-order combine, backward = one launch writing every input gradient.  Inputs: rows of (a, b) CUDA tensors
    (b ignored unless the row is an L1 pair)."""

    @staticmethod
    def forward(ctx, modes, *tensors):
        k = len(modes)
        a, b = list(tensors[:k]), list(tensors[k:])
        ctx.modes, ctx.k = modes, k
        ctx.save_for_backward(*[t.detach() for t in tensors])
        return _engine.loss_forward(a, b, list(modes))

    @staticmethod
    def backward(ctx, grad_out):
        k, modes = ctx.k, ctx.modes
        saved = ctx.saved_tensors
        a, b = list(saved[:k]), list(saved[k:])
        need_b = [ctx.needs_input_grad[1 + k + i] and modes[i] == _engine.LOSS_L1 for i in range(k)]
        ga, gb = _engine.loss_backward(a, b, list(modes), grad_out, need_b)
        ga = [g if ctx.needs_input_grad[1 + i] else None for i, g in enumerate(ga)]
        return (None, *[g.view_as(t) if g is not None else None for g, t in zip(ga, a)],
                *[g.view_as(t) if g is not None else None for g, t in zip(gb, b)])


class _StackedLossRows(torch.autograd.Function):
    """The same row means, for rows that are halves (real / generated) of stacked discriminator outputs: forward reads the
    halves in place, backward writes each row's gradient straight into its half of ONE gradient tensor per stacked map.
    rows: tuple of (parent index, half of a, half of b or None, mode)."""

    @staticmethod
    def forward(ctx, rows, *parents):
        ctx.rows = rows
        ctx.save_for_backward(*parents)
        a, b = _StackedLossRows._views(rows, [p.detach() for p in parents])
        return _engine.loss_forward(a, [u if u is not None else t for t, u in zip(a, b)], [r[3] for r in rows])

    @staticmethod
    def _views(rows, tensors):
        a, b = [], []
        for pi, ha, hb, _mode in rows:
            t = tensors[pi]
            n = t.shape[0] // 2
            a.append(t[ha * n:(ha + 1) * n])
            b.append(t[hb * n:(hb + 1) * n] if hb is not None else None)
        return a, b

    @staticmethod
    def backward(ctx, grad_out):
        rows, parents = ctx.rows, ctx.saved_tensors
        covered = [set() for _ in parents]
        for pi, ha, hb, _mode in rows:
            covered[pi].add(ha)
            if hb is not None:
                covered[pi].add(hb)
        grads = [(torch.empty_like(p) if len(c) == 2 else torch.zeros_like(p)) if ctx.needs_input_grad[1 + i] else None
                 for i, (p, c) in enumerate(zip(parents, covered))]
        scratch = [g if g is not None else torch.empty_like(p) for g, p in zip(grads, parents)]
        a, b = _StackedLossRows._views(rows, [p.detach() for p in parents])
        ga, gb = _StackedLossRows._views(rows, scratch)
        modes = [r[3] for r in rows]
        _engine.loss_backward(a, [u if u is not None else t for t, u in zip(a, b)], modes, grad_out,
                              [u is not None for u in b], out_a=ga, out_b=gb)
        return (None, *grads)


def _stacked_rows(a, b, modes):
    """If every row is a tagged half of a stacked discriminator output (MultiScaleDiscriminator.forward), the table in
    (parent index, halves, mode) form plus the distinct parents; else None."""
    parents, index, rows = [], {}, []
    for t, u, m in zip(a, b, modes):
        ti = getattr(t, "_mg_half", None)
        ui = getattr(u, "_mg_half", None) if u is not None else None
        if ti is None or (u is not None and (ui is None or ui[0] is not ti[0])) or not ti[0].requires_grad:
            return None
        if id(ti[0]) not in index:
            index[id(ti[0])] = len(parents)
            parents.append(ti[0])
        rows.append((index[id(ti[0])], ti[1], ui[1] if ui is not None else None, m))
    return tuple(rows), parents


def _row_means(a, b, modes):
    """Row means of a loss table on the fused kernels.  CUDA tensors only, like the modules: there is no CPU path."""
    if not all(t.is_cuda for t in a):
        raise _engine.EngineError("melgan_multi_b200 loss functions need CUDA tensors (no CPU fallback)")
    st = _stacked_rows(a, b, modes) if torch.is_grad_enabled() else None
    if st is not None:
        return _StackedLossRows.apply(st[0], *st[1])
    b = [u if u is not None else t for t, u in zip(a, b)]  # placeholder rows keep the argument list rectangular
    return _LossRows.apply(tuple(modes), *a, *b)


def feature_loss(fmap_r, fmap_g):
    """10 * sum over the 21 feature-map pairs of mean |r - g| (reference models.py:138-144)."""
    rs = [r for maps in fmap_r for r in maps]
    gs = [g for maps in fmap_g for g in maps]
    return _row_means(rs, gs, [_engine.LOSS_L1] * len(rs)).sum() * 10


def discriminator_loss(disc_real_outputs, disc_generated_outputs):
    """LSGAN discriminator loss; returns (loss, real terms, generated terms) like models.py:147-159 (the two lists are
    Python floats, as in the reference -- read back with ONE host sync instead of six)."""
    k = len(disc_real_outputs)
    rows = list(disc_real_outputs) + list(disc_generated_outputs)
    means = _row_means(rows, [None] * (2 * k), [_engine.LOSS_ONE_MINUS_SQ] * k + [_engine.LOSS_SQ] * k)
    vals = means.detach().tolist()
    # the read-back above synchronised the stream: every forward enqueued before it has finished, so its pipeline status
    # word (engine._StatusWatch) can be inspected here at no cost -- a stalled tcgen05 pipeline raises instead of training on
    _engine.poll_status()
    return means.sum(), vals[:k], vals[k:]


def generator_loss(disc_generated_outputs):
    """LSGAN generator loss (reference models.py:162-167)."""
    rows = list(disc_generated_outputs)
    return _row_means(rows, [None] * len(rows), [_engine.LOSS_ONE_MINUS_SQ] * len(rows)).sum()
