"""Training step of the reference (SURVEY §8 f2, BASELINE configs[4]) composed from this library's kernels.

What the reference does per step (train_utils.py:137-166, ``Trainer.loss`` / ``Trainer.step``):

    t ~ U{1..T}/T or U[0, 1) (fp64), noise ~ N(0, I)            # Trainer.loss, generator seeded 8191 + rank
    loss = diffusion.train_loss(model, x_0, t, y, noise)        # q_sample -> UNet.forward (.train()) -> re-weighted MSE
    loss.mean().div(num_accum).backward()                       # autograd through the whole UNet
    [DistributedDataParallel averages the gradients over ranks]
    clip_grad_norm_ -> AdamW.step -> EMA.update                 # train_utils.py:159-166

Here the UNet's forward AND backward are an explicit list of kernel calls over NHWC tensors -- no autograd graph:
``UNetTrainGraph.forward`` records one closure per block (the tape), ``UNetTrainGraph.backward`` replays it in reverse.
Every contraction, normalisation and attention call goes through the C ABI (``vdt_op_*``, the entry points the kernel
parity tests exercise one by one): conv forward / dgrad / wgrad on tcgen05, the fused GroupNorm -> FiLM -> SiLU -> dropout
forward and backward, the attention core forward (tcgen05) and backward (fp32), the fp32 linear kernel for the embedding
MLP and the FiLM projections (also used for their backward products, with transposed operands).  PyTorch supplies device
memory and the glue between the calls that a production version would fold into the kernels' epilogues: 16-bit casts of the
gradient tensors, the residual / skip adds, ``torch.cat`` of the concat blocks' inputs, the 2x2 resample adjoints, SiLU and
its derivative on the [B, E] embedding, bias-gradient column sums of the tiny linears.  This slice is about a complete,
reference-matching training step; it is not tuned (the kernel-level hooks allocate and synchronise per call).

fp16 gradients: a gradient tensor handed to dgrad / wgrad is rounded to the 16-bit operand format.  With fp16 operands
each such tensor is first multiplied by a power of two that brings its largest magnitude to ~2^10 and the results are
multiplied back (exact, no host sync: the factor lives on the device), so d loss.mean() / d activations of order 1e-7 do
not flush to zero; bf16 operands need no scaling.

There is no CPU fallback and no backend switch: ``KernelOps`` is what every graph constructs.  (tests/test_training_graph.py
checks the *orchestration* -- which gradient flows where -- against autograd by monkeypatching this module's ``KernelOps``
name with a stand-in that models each call's contract in fp64; nothing in the package can select another backend.)
"""
import ctypes as C

import torch
import torch.nn.functional as F

from . import _lib

_PAD = 128            # in_conv's im2col depth and out_conv's channel count are padded to this (tested GEMM shapes)


def pow2_scale_for_16bit(x, target_log2=10):
    """Power-of-two factor s (0-dim tensor on x's device, no host sync) with max|x * s| in [2^target, 2^(target+1));
    1 when x is all zero or not finite."""
    amax = x.detach().abs().amax().to(torch.float32)
    e = torch.floor(torch.log2(amax))
    ok = torch.isfinite(e)
    e = torch.where(ok, e, torch.zeros_like(e)).clamp(-100.0, 100.0)
    return torch.where(ok, torch.exp2(float(target_log2) - e), torch.ones_like(e))


class KernelOps:
    """ctypes calls into libvdt_b200.so (include/vdt_b200.h), one method per kernel-level entry point.  Tensors are
    contiguous CUDA tensors: activations NHWC, fp32 unless the name says 16."""

    def __init__(self, operand_dtype="fp16"):
        if operand_dtype not in ("fp16", "bf16"):
            raise NotImplementedError("the training step runs with fp16 or bf16 tensor-core operands "
                                      f"(got {operand_dtype!r}; fp16x3 is a sampling-only validation mode)")
        self.f16 = 1 if operand_dtype == "fp16" else 0
        self.dt = torch.float16 if self.f16 else torch.bfloat16
        self.acc = torch.float32
        self.L = _lib.lib()                                  # raises when the CUDA library is missing

    # ---- helpers
    @staticmethod
    def _cuda32(*ts):
        for t in ts:
            if t is not None and (t.device.type != "cuda" or t.dtype != torch.float32 or not t.is_contiguous()):
                raise ValueError("expected contiguous fp32 CUDA tensors (there is no CPU fallback)")

    def _call(self, fn, *args):
        _lib.check(fn(*args, _lib.current_stream_ptr()))

    def to16(self, x):
        return x.to(self.dt)

    def grad16(self, g):
        """16-bit copy of a gradient tensor for dgrad / wgrad and the factor to multiply their results by (None: 1)."""
        if not self.f16:
            return g.to(self.dt), None
        s = pow2_scale_for_16bit(g)
        return (g * s).to(self.dt), 1.0 / s

    # ---- forward kernels
    def groupnorm(self, src1, src2, gamma, beta, film, silu, resample, want_raw, want_res):
        self._cuda32(src1, src2, gamma, beta, film)
        B, H, W, c1 = src1.shape
        c2 = 0 if src2 is None else src2.shape[3]
        Cc = c1 + c2
        Ho, Wo = (H // 2, W // 2) if resample == 1 else (H * 2, W * 2) if resample == 2 else (H, W)
        act = torch.empty((B, Ho, Wo, Cc), device=src1.device, dtype=self.dt)
        raw = torch.empty((B, H, W, Cc), device=src1.device, dtype=self.dt) if want_raw else None
        res = torch.empty((B, Ho, Wo, Cc), device=src1.device, dtype=torch.float32) if want_res else None
        self._call(self.L.vdt_op_groupnorm, _lib.ptr(src1), c1, _lib.ptr(src2), c2, B, H, W, _lib.ptr(gamma), _lib.ptr(beta),
                   _lib.ptr(film), 2 * Cc if film is not None else 0, 0, int(bool(silu)), int(resample), _lib.ptr(act),
                   _lib.ptr(raw), _lib.ptr(res), self.f16, None, None, 4, 0)
        return act, raw, res

    def groupnorm_train(self, src, gamma, beta, film, drop_p, seed, layer):
        self._cuda32(src, gamma, beta, film)
        B, H, W, Cc = src.shape
        act = torch.empty((B, H, W, Cc), device=src.device, dtype=self.dt)
        self._call(self.L.vdt_op_groupnorm_train, _lib.ptr(src), Cc, B, H, W, _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(film),
                   2 * Cc, 0, 1, _lib.ptr(act), self.f16, C.c_float(drop_p), C.c_uint64(seed), int(layer))
        return act

    def conv(self, a16, w, b, residual, ksize, out16=False):
        self._cuda32(w, b, residual)
        B, H, W, cin = a16.shape
        cout = w.shape[0]
        assert a16.dtype == self.dt and a16.is_contiguous() and tuple(w.shape) == (cout, cin, ksize, ksize)
        out = torch.empty((B, H, W, cout), device=a16.device, dtype=self.dt if out16 else torch.float32)
        self._call(self.L.vdt_op_conv, _lib.ptr(a16), B, H, W, cin, _lib.ptr(w), cout, ksize, _lib.ptr(b), _lib.ptr(residual),
                   None if out16 else _lib.ptr(out), self.f16, _lib.ptr(out) if out16 else None, None, 4)
        return out

    def attention(self, qkv16, B, N, heads, d):
        assert qkv16.dtype == self.dt and qkv16.is_contiguous() and tuple(qkv16.shape) == (B * N, 3 * heads * d)
        out = torch.empty((B * N, heads * d), device=qkv16.device, dtype=self.dt)
        self._call(self.L.vdt_op_attention, _lib.ptr(qkv16), _lib.ptr(out), B, N, heads, d, self.f16)
        return out

    def linear(self, x, w, b, silu=False):
        self._cuda32(x, w, b)
        rows, K = x.shape
        N = w.shape[0]
        assert tuple(w.shape) == (N, K) and tuple(b.shape) == (N,)
        out = torch.empty((rows, N), device=x.device, dtype=torch.float32)
        self._call(self.L.vdt_op_linear, _lib.ptr(x), _lib.ptr(w), _lib.ptr(b), _lib.ptr(out), rows, K, N, int(bool(silu)))
        return out

    def timestep_embedding(self, t, dim):
        if t.device.type != "cuda" or t.dtype != torch.float64 or not t.is_contiguous():
            raise ValueError("t must be a contiguous fp64 CUDA tensor")
        out = torch.empty((t.numel(), dim), device=t.device, dtype=torch.float32)
        self._call(self.L.vdt_op_timestep_embedding, _lib.ptr(t), _lib.ptr(out), t.numel(), dim)
        return out

    # ---- backward kernels
    def conv_backward(self, a16, dy16, w, ksize, need_dx=True):
        """(dX fp32 NHWC or None, dW fp32 OIHW, dbias fp32) of conv(a16, w) given dY in 16 bits."""
        self._cuda32(w)
        B, H, W, cin = a16.shape
        cout = w.shape[0]
        assert dy16.dtype == self.dt and dy16.is_contiguous() and tuple(dy16.shape) == (B, H, W, cout)
        dx = None
        if need_dx:
            dx = torch.empty((B, H, W, cin), device=a16.device, dtype=torch.float32)
            self._call(self.L.vdt_op_conv_dgrad, _lib.ptr(dy16), B, H, W, cin, _lib.ptr(w), cout, ksize, _lib.ptr(dx), self.f16)
        dw = torch.empty_like(w)
        db = torch.empty((cout,), device=w.device, dtype=torch.float32)
        self._call(self.L.vdt_op_conv_wgrad, _lib.ptr(a16), _lib.ptr(dy16), B, H, W, cin, cout, ksize, _lib.ptr(dw), _lib.ptr(db),
                   self.f16)
        return dx, dw, db

    def groupnorm_backward(self, x, dact, gamma, beta, film, silu, drop_p, seed, layer):
        self._cuda32(x, dact, gamma, beta, film)
        B, H, W, Cc = x.shape
        assert dact.shape == x.shape
        dx = torch.empty_like(x)
        dg = torch.empty((Cc,), device=x.device, dtype=torch.float32)
        db = torch.empty((Cc,), device=x.device, dtype=torch.float32)
        df = torch.empty_like(film) if film is not None else None
        self._call(self.L.vdt_op_groupnorm_backward, _lib.ptr(x), _lib.ptr(dact), Cc, B, H, W, _lib.ptr(gamma), _lib.ptr(beta),
                   _lib.ptr(film), int(bool(silu)), C.c_float(drop_p), C.c_uint64(seed), int(layer), _lib.ptr(dx), _lib.ptr(dg),
                   _lib.ptr(db), _lib.ptr(df))
        return dx, dg, db, df

    def attention_backward(self, qkv, do, B, N, heads, d):
        self._cuda32(qkv, do)
        dqkv = torch.empty_like(qkv)
        self._call(self.L.vdt_op_attention_backward, _lib.ptr(qkv), _lib.ptr(do), _lib.ptr(dqkv), B, N, heads, d)
        return dqkv


def _silu_grad(x):
    s = torch.sigmoid(x)
    return s * (1 + x * (1 - s))


def _resample_adjoint(g, mode):
    """Adjoint of the 2x2 resampling between act1 and conv1 / on the skip path (unet.py:127-130, 138, 141), NHWC."""
    if mode == 1:                                   # AvgPool2d(2): every input pixel receives a quarter of its cell's gradient
        return (g.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2) * 0.25).contiguous()
    if mode == 2:                                   # nearest x2: an input pixel collects its four copies
        B, H2, W2, Cc = g.shape
        return g.reshape(B, H2 // 2, 2, W2 // 2, 2, Cc).sum(dim=(2, 4)).contiguous()
    return g


def block_list(model):
    """Execution order of the UNet's blocks (unet.py:230-283, 297-321) read off the module tree: dicts with kind
    ("res" | "attn"), the parameter-name prefix, the module, resample (0 none / 1 avg-pool / 2 nearest), concat (input is
    cat[h, hs.pop()]) and push (output appended to hs)."""
    out = []

    def add(prefix, mod, resample=0, concat=False, push=False):
        if isinstance(mod, torch.nn.ModuleList):                       # Sequential(ResidualBlock, AttentionBlock)
            out.append(dict(kind="res", name=prefix + ".0", module=mod[0], resample=resample, concat=concat, push=False))
            out.append(dict(kind="attn", name=prefix + ".1", module=mod[1], resample=0, concat=False, push=push))
        else:
            out.append(dict(kind="res", name=prefix, module=mod, resample=resample, concat=concat, push=push))

    nrb, levels = model.num_res_blocks, model.levels
    for i in range(levels):
        for j, mod in enumerate(model.downsamples[f"level_{i}"]):
            add(f"downsamples.level_{i}.{j}", mod, resample=1 if j == nrb else 0, push=True)
    out.append(dict(kind="res", name="middle.0", module=model.middle[0], resample=0, concat=False, push=False))
    out.append(dict(kind="attn", name="middle.1", module=model.middle[1], resample=0, concat=False, push=False))
    out.append(dict(kind="res", name="middle.2", module=model.middle[2], resample=0, concat=False, push=False))
    for i in range(levels - 1, -1, -1):
        for j, mod in enumerate(model.upsamples[f"level_{i}"]):
            if j != nrb + 1:
                add(f"upsamples.level_{i}.{j}", mod, concat=True)
            else:
                add(f"upsamples.level_{i}.{j}", mod, resample=2)
    return out


class UNetTrainGraph:
    """``UNet.forward`` in .train() mode with everything the backward needs kept, and the matching backward pass.

        graph = UNetTrainGraph(model)
        out = graph.forward(x_t, t, y)              # fp32 NCHW, like UNet.forward(x, t, y) (unet.py:286-322)
        grads = graph.backward(grad_out)            # {state_dict key: fp32 gradient}, what autograd leaves in .grad
    """

    def __init__(self, model):
        self.model = model
        self.ops = KernelOps(model.operand_dtype)
        self.blocks = block_list(model)
        if model.in_channels * 9 > _PAD or model.out_channels > _PAD:
            raise NotImplementedError(f"in_channels * 9 and out_channels must not exceed {_PAD}")
        self._tape = None

    # ------------------------------------------------------------------ bookkeeping
    def _acc(self, name, g):
        g = g.reshape(self._P[name].shape)
        self._grads[name] = g if name not in self._grads else self._grads[name] + g

    def _zeros(self, n, like):
        return torch.zeros((n,), device=like.device, dtype=like.dtype)

    def _scaled(self, g):
        return self.ops.grad16(g)

    @staticmethod
    def _unscale(inv, *ts):
        return tuple(t if (inv is None or t is None) else t * inv for t in ts)

    def _conv_backward(self, a16, dy, w, ksize, need_dx=True, scaled=None):
        """``scaled``: the (16-bit copy, inverse factor) pair of ``dy`` when the caller already made it (a block's output
        gradient feeds both conv2's and the 1x1 skip conv's backward)."""
        dy16, inv = scaled if scaled is not None else self._scaled(dy.contiguous())
        return self._unscale(inv, *self.ops.conv_backward(a16, dy16, w, ksize, need_dx))

    def _linear_nobias(self, x, w):
        return self.ops.linear(x.contiguous(), w.contiguous(), self._zeros(w.shape[0], x))

    # ------------------------------------------------------------------ forward
    def forward(self, x, t, y=None, drop_rate=None, seed=None):
        model, ops = self.model, self.ops
        if x.ndim != 4 or x.shape[1] != model.in_channels or x.shape[2] != x.shape[3]:
            raise ValueError(f"expected x of shape (B, {model.in_channels}, R, R), got {tuple(x.shape)}")
        B, dev = x.shape[0], x.device
        self._P = P = {k: v.detach() for k, v in model.named_parameters()}
        self._grads = {}
        self._tape = []
        if drop_rate is None:
            drop_rate = float(model.drop_rate) if model.training else 0.0
        if seed is None:                                               # nn.Dropout draws from the global generator
            seed = int(torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64).item()) if drop_rate > 0 else 0
        self._drop, self._seed = float(drop_rate), int(seed)
        pdt = P["in_conv.weight"].dtype

        # ---- time / class embedding (unet.py:287-295)
        t = t.reshape(-1).to(device=dev, dtype=torch.float64).contiguous()
        if t.numel() != B:
            raise ValueError("t must have one entry per batch row")
        temb0 = ops.timestep_embedding(t, model.hid_channels).to(pdt)
        e1 = ops.linear(temb0, P["time_embed.0.weight"], P["time_embed.0.bias"])
        a1 = F.silu(e1)
        emb = ops.linear(a1, P["time_embed.2.weight"], P["time_embed.2.bias"])
        cls_in, cls_key = None, None
        if model.num_classes and y is not None:
            if model.multitags:
                assert y.ndim == 2                                     # unet.py:291
                yy = y.to(device=dev, dtype=pdt)
                cls_in = yy / torch.count_nonzero(yy, dim=1).clamp(min=1.).sqrt().unsqueeze(1)
                cls_key = "class_embed"
            else:
                yl = y.to(device=dev, dtype=torch.int64).reshape(-1)   # OneHot(exclude_zero=True), modules.py:190-199
                if int(yl.min()) < 0 or int(yl.max()) > model.num_classes:
                    raise RuntimeError(f"class ids must lie in [0, {model.num_classes}] (0 = unconditional)")
                cls_in = F.one_hot((yl - 1).clamp(min=0), model.num_classes).to(pdt)
                cls_in[yl == 0] = 0
                cls_key = "class_embed.1"
            cls_in = cls_in.contiguous()
            emb = emb + ops.linear(cls_in, P[cls_key + ".weight"], P[cls_key + ".bias"])
        emb_act = F.silu(emb).contiguous()                             # ResidualBlock.fc(act1(t_emb)), unet.py:142
        self._emb = dict(temb0=temb0, e1=e1, a1=a1, emb=emb, emb_act=emb_act, cls_in=cls_in, cls_key=cls_key)
        self._d_emb_act = torch.zeros_like(emb_act)

        # ---- in_conv (unet.py:297) as a pointwise GEMM over 3x3 patches: K = in_channels * 9 padded to _PAD
        R = x.shape[2]
        hid, cin9 = model.hid_channels, model.in_channels * 9
        cols = F.unfold(x.to(pdt), 3, padding=1).transpose(1, 2)        # [B, R*R, cin*9], (c, ky, kx) like weight.reshape(hid, -1)
        cols = F.pad(cols, (0, _PAD - cin9)).reshape(B, R, R, _PAD)
        cols16 = ops.to16(cols.contiguous())
        w_in = F.pad(P["in_conv.weight"].reshape(hid, cin9), (0, _PAD - cin9)).reshape(hid, _PAD, 1, 1).contiguous()
        h = ops.conv(cols16, w_in, P["in_conv.bias"], None, 1)
        self._in_conv = dict(cols16=cols16, w=w_in)

        vals = [h]
        hs = [0]
        cur = 0
        for layer, blk in enumerate(self.blocks):
            ins = [cur, hs.pop()] if blk["concat"] else [cur]
            xs = [vals[i] for i in ins]
            out, bwd = (self._res_forward(blk, xs, emb_act, layer) if blk["kind"] == "res" else self._attn_forward(blk, xs))
            vals.append(out)
            cur = len(vals) - 1
            self._tape.append((ins, cur, bwd))
            if blk["push"]:
                hs.append(cur)
        assert not hs, len(hs)
        self._num_vals = len(vals)

        # ---- out_conv (unet.py:246-249, 321): GroupNorm -> SiLU -> conv 3x3 to out_channels (padded to _PAD GEMM columns)
        h_last = vals[cur]
        oc = model.out_channels
        g, be = P["out_conv.0.weight"], P["out_conv.0.bias"]
        a_out = ops.groupnorm(h_last, None, g, be, None, True, 0, False, False)[0]
        w_out = F.pad(P["out_conv.2.weight"], (0, 0, 0, 0, 0, 0, 0, _PAD - oc)).contiguous()
        b_out = F.pad(P["out_conv.2.bias"], (0, _PAD - oc)).contiguous()
        o = ops.conv(a_out, w_out, b_out, None, 3)
        self._out_conv = dict(h=h_last, a=a_out, w=w_out, last=cur)
        return o[..., :oc].permute(0, 3, 1, 2).contiguous()

    def _res_forward(self, blk, xs, emb_act, layer):
        """ResidualBlock.forward (unet.py:137-148)."""
        ops, P, n, r = self.ops, self._P, blk["name"], blk["resample"]
        x1 = xs[0]
        x2 = xs[1] if len(xs) > 1 else None
        c1 = x1.shape[3]
        has_skip = (n + ".skip.weight") in P
        if has_skip and r:
            raise NotImplementedError("a resampling ResidualBlock that also changes the channel count")
        g1, be1, w1, b1 = P[n + ".norm1.weight"], P[n + ".norm1.bias"], P[n + ".conv1.weight"], P[n + ".conv1.bias"]
        g2, be2, w2, b2 = P[n + ".norm2.weight"], P[n + ".norm2.bias"], P[n + ".conv2.weight"], P[n + ".conv2.bias"]
        wfc, bfc = P[n + ".fc.weight"], P[n + ".fc.bias"]
        drop, seed = self._drop, self._seed
        a1, raw16, res = ops.groupnorm(x1, x2, g1, be1, None, True, r, has_skip, bool(r))    # norm1 -> act1 -> resample
        h1 = ops.conv(a1, w1, b1, None, 3)
        film = ops.linear(emb_act, wfc, bfc)                               # [B, 2 cout]: shift | scale (unet.py:145)
        a2 = ops.groupnorm_train(h1, g2, be2, film, drop, seed, layer)     # norm2 -> FiLM -> act2 -> dropout
        if has_skip:
            ws, bs = P[n + ".skip.weight"], P[n + ".skip.bias"]
            skip = ops.conv(raw16, ws, bs, None, 1)
        else:
            skip = res if r else x1
        out = ops.conv(a2, w2, b2, skip, 3)

        def backward(dout):
            dout16 = self._scaled(dout.contiguous())
            da2, dw2, db2 = self._conv_backward(a2, dout, w2, 3, scaled=dout16)
            self._acc(n + ".conv2.weight", dw2); self._acc(n + ".conv2.bias", db2)
            dh1, dg2, dbe2, dfilm = ops.groupnorm_backward(h1, da2.contiguous(), g2, be2, film, True, drop, seed, layer)
            self._acc(n + ".norm2.weight", dg2); self._acc(n + ".norm2.bias", dbe2)
            # fc: film = emb_act W^T + b
            self._d_emb_act += self._linear_nobias(dfilm, wfc.t())
            self._acc(n + ".fc.weight", self._linear_nobias(dfilm.t(), emb_act.t()))
            self._acc(n + ".fc.bias", dfilm.sum(dim=0))
            da1, dw1, db1 = self._conv_backward(a1, dh1, w1, 3)
            self._acc(n + ".conv1.weight", dw1); self._acc(n + ".conv1.bias", db1)
            da1 = _resample_adjoint(da1, r)
            xcat = x1 if x2 is None else torch.cat([x1, x2], dim=3)
            dx, dg1, dbe1, _ = ops.groupnorm_backward(xcat.contiguous(), da1.contiguous(), g1, be1, None, True, 0.0, 0, 0)
            self._acc(n + ".norm1.weight", dg1); self._acc(n + ".norm1.bias", dbe1)
            if has_skip:
                ds, dws, dbs = self._conv_backward(raw16, dout, ws, 1, scaled=dout16)
                self._acc(n + ".skip.weight", dws); self._acc(n + ".skip.bias", dbs)
                dx = dx + ds
            else:
                dx = dx + _resample_adjoint(dout, r)
            if x2 is None:
                return [dx]
            return [dx[..., :c1].contiguous(), dx[..., c1:].contiguous()]

        return out, backward

    def _attn_forward(self, blk, xs):
        """AttentionBlock.forward (unet.py:73-81)."""
        ops, P, n, model = self.ops, self._P, blk["name"], self.model
        x = xs[0]
        B, H, W, Cc = x.shape
        N = H * W
        hid = P[n + ".proj_out.weight"].shape[1]
        if model.head_dim is None:                                       # unet.py:43-49
            heads = model.num_heads
            d = Cc // heads
        else:
            d = model.head_dim
            heads = model.num_heads if model.num_heads is not None else Cc // d
        assert heads * d == hid
        g, be = P[n + ".norm.weight"], P[n + ".norm.bias"]
        w_in, b_in, w_o, b_o = P[n + ".proj_in.weight"], P[n + ".proj_in.bias"], P[n + ".proj_out.weight"], P[n + ".proj_out.bias"]
        a = ops.groupnorm(x, None, g, be, None, False, 0, False, False)[0]
        qkv16 = ops.conv(a, w_in, b_in, None, 1, out16=True)             # q | k | v thirds, heads contiguous (unet.py:76-78)
        o16 = ops.attention(qkv16.reshape(B * N, 3 * hid), B, N, heads, d).reshape(B, H, W, hid)
        out = ops.conv(o16, w_o, b_o, x, 1)

        def backward(dout):
            do, dwo, dbo = self._conv_backward(o16, dout, w_o, 1)
            self._acc(n + ".proj_out.weight", dwo); self._acc(n + ".proj_out.bias", dbo)
            qkv = qkv16.to(ops.acc).reshape(B * N, 3 * hid).contiguous()
            dqkv = ops.attention_backward(qkv, do.reshape(B * N, hid).contiguous(), B, N, heads, d).reshape(B, H, W, 3 * hid)
            da, dwi, dbi = self._conv_backward(a, dqkv, w_in, 1)
            self._acc(n + ".proj_in.weight", dwi); self._acc(n + ".proj_in.bias", dbi)
            dx, dg, dbe, _ = ops.groupnorm_backward(x, da.contiguous(), g, be, None, False, 0.0, 0, 0)
            self._acc(n + ".norm.weight", dg); self._acc(n + ".norm.bias", dbe)
            return [dx + dout]

        return out, backward

    # ------------------------------------------------------------------ backward
    def backward(self, grad_out):
        """``grad_out``: d loss / d output, fp32 NCHW like the output.  Returns {parameter name: gradient}."""
        if self._tape is None:
            raise RuntimeError("backward() needs a forward() first")
        ops, P, model = self.ops, self._P, self.model
        oc = model.out_channels
        oc_ = self._out_conv
        # out_conv
        g_nhwc = F.pad(grad_out.to(oc_["h"].dtype).permute(0, 2, 3, 1), (0, _PAD - oc)).contiguous()
        da, dwp, dbp = self._conv_backward(oc_["a"], g_nhwc, oc_["w"], 3)
        self._acc("out_conv.2.weight", dwp[:oc]); self._acc("out_conv.2.bias", dbp[:oc])
        dh, dg, dbe, _ = ops.groupnorm_backward(oc_["h"], da.contiguous(), P["out_conv.0.weight"], P["out_conv.0.bias"], None, True,
                                                0.0, 0, 0)
        self._acc("out_conv.0.weight", dg); self._acc("out_conv.0.bias", dbe)
        pending = {oc_["last"]: dh}
        # blocks, last to first
        for ins, oid, bwd in reversed(self._tape):
            dins = bwd(pending.pop(oid).contiguous())
            for i, d in zip(ins, dins):
                pending[i] = d if i not in pending else pending[i] + d
        # in_conv: parameters only (no gradient w.r.t. the images)
        ic = self._in_conv
        hid, cin9 = model.hid_channels, model.in_channels * 9
        _, dwi, dbi = self._conv_backward(ic["cols16"], pending.pop(0), ic["w"], 1, need_dx=False)
        self._acc("in_conv.weight", dwi.reshape(hid, _PAD)[:, :cin9]); self._acc("in_conv.bias", dbi)
        assert not pending, sorted(pending)
        # embedding MLP (unet.py:287-295, 201-215)
        E = self._emb
        d_emb = self._d_emb_act * _silu_grad(E["emb"])
        if E["cls_in"] is not None:
            k = E["cls_key"]
            self._acc(k + ".weight", self._linear_nobias(d_emb.t(), E["cls_in"].t()))
            self._acc(k + ".bias", d_emb.sum(dim=0))
        self._acc("time_embed.2.weight", self._linear_nobias(d_emb.t(), E["a1"].t()))
        self._acc("time_embed.2.bias", d_emb.sum(dim=0))
        d_e1 = self._linear_nobias(d_emb, P["time_embed.2.weight"].t()) * _silu_grad(E["e1"])
        self._acc("time_embed.0.weight", self._linear_nobias(d_e1.t(), E["temb0"].t()))
        self._acc("time_embed.0.bias", d_e1.sum(dim=0))
        grads, self._grads, self._tape = self._grads, {}, None
        for k, p in P.items():                                          # e.g. class_embed when y is None: autograd leaves None
            if k not in grads:
                grads[k] = torch.zeros_like(p)
        return grads


class _UNetFunction(torch.autograd.Function):
    """One autograd node for the whole UNet: forward = UNetTrainGraph.forward, backward = UNetTrainGraph.backward (the kernel
    tape), handing each parameter its gradient.  No gradient flows to the images, times or labels (training never needs one)."""

    @staticmethod
    def forward(ctx, graph, names, x, t, y, *params):
        ctx.graph, ctx.names = graph, names
        return graph.forward(x, t, y)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        grads = ctx.graph.backward(grad_out.contiguous())
        return (None, None, None, None, None) + tuple(grads[n] for n in ctx.names)


def unet_autograd_forward(model, x, t, y=None):
    """``UNet.forward`` with ``UNet.autograd = True`` under grad mode: a fresh graph (tape) per call, so several forwards may
    be outstanding before their backwards, like any autograd graph."""
    graph = UNetTrainGraph(model)
    named = list(model.named_parameters())
    return _UNetFunction.apply(graph, tuple(k for k, _ in named), x.detach(), t, y, *(p for _, p in named))


class GradBucketReducer:
    """What DistributedDataParallel does to the gradients (train.py wraps the model in DDP; the reference relies on its
    bucketed all-reduce): average them over the ranks.  Gradients are packed into flat buckets of ``bucket_bytes`` in the
    order they are handed over; every full bucket starts an asynchronous all-reduce (NCCL over NVLink on the GPUs, gloo in
    the CPU tests) while the caller keeps producing gradients; ``finish`` waits, divides by the world size and unpacks.
    The only collective of the training step; nothing else crosses ranks."""

    def __init__(self, world_size, bucket_bytes=64 << 20, group=None):
        self.world_size, self.bucket_bytes, self.group = int(world_size), int(bucket_bytes), group
        self._open, self._open_bytes, self._inflight = [], 0, []

    def add(self, name, g):
        self._open.append((name, g))
        self._open_bytes += g.numel() * g.element_size()
        if self._open_bytes >= self.bucket_bytes:
            self._launch()

    def _launch(self):
        if not self._open:
            return
        import torch.distributed as dist
        items, self._open, self._open_bytes = self._open, [], 0
        flat = torch.cat([g.reshape(-1) for _, g in items])
        work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True) if self.world_size > 1 else None
        self._inflight.append((items, flat, work))

    def finish(self):
        """-> {name: averaged gradient}; resets the reducer."""
        self._launch()
        out = {}
        for items, flat, work in self._inflight:
            if work is not None:
                work.wait()
            if self.world_size > 1:
                flat.div_(self.world_size)
            off = 0
            for name, g in items:
                out[name] = flat[off:off + g.numel()].view(g.shape)
                off += g.numel()
        self._inflight = []
        return out


class ema_weights:
    """``with self.ema:`` of the reference trainer (utils.py:151-166, used by Trainer.sample_fn train_utils.py:173-176): inside
    the block the model's parameters hold the EMA shadow, afterwards the live weights are back.  Plain device copies; the
    model's sampling plans are told to re-pack on both edges."""

    def __init__(self, model, shadow):
        self.model, self.shadow, self.backup = model, shadow, None

    def _mark(self):
        if hasattr(self.model, "mark_weights_changed"):
            self.model.mark_weights_changed()

    @torch.no_grad()
    def __enter__(self):
        if not self.shadow:
            raise RuntimeError("this rank keeps no EMA shadow (use_ema=False, or not the leader: train_utils.py:127-130)")
        self.backup = {k: p.detach().clone() for k, p in self.model.named_parameters()}
        for k, p in self.model.named_parameters():
            p.copy_(self.shadow[k])
        self._mark()
        return self.model

    @torch.no_grad()
    def __exit__(self, *exc):
        for k, p in self.model.named_parameters():
            p.copy_(self.backup[k])
        self.backup = None
        self._mark()
        return False


class TrainingStep:
    """``Trainer.loss`` + ``Trainer.step`` (train_utils.py:137-166) for one rank.

        step = TrainingStep(model, diffusion, timesteps=0, lr=2e-4, grad_norm=1.0, use_ema=True)
        loss = step.step(x, y)          # x fp32 NCHW in [-1, 1] on the GPU, y class ids / multi-hot rows / None

    ``model`` is a ``v_diffusion_b200.UNet`` on the GPU, ``diffusion`` a ``v_diffusion_b200.GaussianDiffusion``.  The
    learning-rate schedule stays with the caller (``step(..., lr=...)``), like LambdaLR in train.py:161-162.
    """

    def __init__(self, model, diffusion, timesteps=0, lr=2e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_norm=1.0,
                 num_accum=1, use_ema=True, ema_decay=0.9999, distributed=False, rank=0, world_size=1, device=None):
        from .optim import AdamWEMA
        self.model, self.diffusion = model, diffusion
        self.timesteps, self.num_accum = int(timesteps), int(num_accum)
        self.distributed, self.rank, self.world_size = bool(distributed), int(rank), int(world_size)
        self.is_leader = rank == 0
        self.device = torch.device(device) if device is not None else next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 trains on CUDA (sm_100a) only; there is no CPU fallback")
        self.graph = UNetTrainGraph(model)
        # EMA lives on the leader only (train_utils.py:127-130)
        self.optimizer = AdamWEMA(model.named_parameters(), lr=lr, betas=betas, eps=eps, weight_decay=weight_decay,
                                  grad_norm=grad_norm, ema_decay=ema_decay, use_ema=bool(use_ema and self.is_leader))
        self.generator = torch.Generator(self.device).manual_seed(8191 + rank)          # train_utils.py:121
        self._accum, self._micro = None, 0
        self.last_grad_sq = None

    def ema(self):
        """Context manager: sample / evaluate with the EMA weights (``with self.ema:``, train_utils.py:173)."""
        return ema_weights(self.model, self.optimizer.shadow)

    @torch.no_grad()
    def sample_fn(self, shape, label=None, use_ddim=False, seed=None, use_ema=True):
        """Trainer.sample_fn (train_utils.py:168-186): ``p_sample`` of ``shape`` images on this rank with the EMA weights (where this
        rank keeps them), gathered over the ranks when distributed.  Returns CPU fp32 images."""
        import contextlib
        import torch.distributed as dist
        was_training = self.model.training
        self.model.eval()
        try:
            with (self.ema() if (use_ema and self.optimizer.shadow) else contextlib.nullcontext()):
                sample = self.diffusion.p_sample(denoise_fn=self.model, shape=tuple(shape), device=self.device, noise=None,
                                                 label=label, seed=131071 + self.rank if seed is None else seed, use_ddim=use_ddim)
        finally:
            self.model.train(was_training)
        if self.distributed:
            parts = [torch.zeros(tuple(shape), device=self.device) for _ in range(self.world_size)]
            dist.all_gather(parts, sample.to(self.device))
            sample = torch.cat(parts, dim=0).cpu()
        return sample

    # ---- checkpoints in the reference trainer's format (train_utils.py:309-352): {"model", "optimizer", "ema", "epoch", "rng"}
    def checkpoint(self, epoch=0, **extra_info):
        """``extra_info`` is merged in like Trainer.save_checkpoint(ckpt_path, **extra_info) does -- e.g. ``scheduler=
        lr_scheduler.state_dict()`` (the learning-rate schedule is the caller's) or ``rng=[...]``."""
        ckpt = {"model": {k: v.detach().cpu() for k, v in self.model.state_dict().items()},
                "optimizer": self.optimizer.state_dict(), "epoch": int(epoch)}
        if self.optimizer.shadow:
            ckpt["ema"] = self.optimizer.ema_state_dict()
        ckpt.update(extra_info)
        return ckpt

    def save_checkpoint(self, path, epoch=0, **extra_info):
        if self.is_leader:
            torch.save(self.checkpoint(epoch, **extra_info), path)

    @torch.no_grad()
    def load_checkpoint(self, path_or_dict, map_location="cpu"):
        """Resume from a checkpoint written by this class or by the reference's Trainer.save_checkpoint (DDP "module." prefixes
        accepted).  Returns the stored epoch."""
        from .optim import strip_module_prefix
        ckpt = path_or_dict if isinstance(path_or_dict, dict) else torch.load(path_or_dict, map_location=map_location)
        if "rng" in ckpt:
            self.generator.set_state(ckpt["rng"][int(self.rank)])
        self.model.load_state_dict(strip_module_prefix(ckpt["model"]), strict=True)
        if hasattr(self.model, "mark_weights_changed"):
            self.model.mark_weights_changed()
        self.optimizer.load_state_dict(ckpt["optimizer"])
        if "ema" in ckpt and self.is_leader:
            self.optimizer.load_ema_state_dict(ckpt["ema"])
        return int(ckpt.get("epoch", 0))

    def draw(self, x):
        """The random draws of Trainer.loss (train_utils.py:137-147): continuous or discrete fp64 times, then the noise."""
        B, T = x.shape[0], self.timesteps
        if T > 0:
            t = torch.randint(T, size=(B,), dtype=torch.float64, device=self.device, generator=self.generator).add(1).div(T)
        else:
            t = torch.rand((B,), dtype=torch.float64, device=self.device, generator=self.generator)
        noise = torch.empty_like(x).normal_(generator=self.generator)
        return t, noise

    @torch.no_grad()
    def loss_and_grads(self, x, y, t=None, noise=None):
        """Per-sample loss (B,) and the gradients of ``loss.mean()`` w.r.t. every parameter."""
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if t is None or noise is None:
            t, noise = self.draw(x)
        loss, grad_out = self.diffusion.train_loss(self.graph.forward, x_0=x, t=t, y=y, noise=noise, return_grad=True)
        assert loss.shape == (x.shape[0],)
        return loss, self.graph.backward(grad_out)

    @torch.no_grad()
    def step(self, x, y, update=True, lr=None):
        import torch.distributed as dist
        per_sample, grads = self.loss_and_grads(x, y)
        loss = per_sample.mean()
        if self.num_accum != 1:                                         # loss.div(num_accum).backward()
            grads = {k: g / self.num_accum for k, g in grads.items()}
        if self._accum is None:
            self._accum = grads
        else:
            for k, g in grads.items():
                self._accum[k] += g
        if self.distributed:
            dist.reduce(loss, dst=0, op=dist.ReduceOp.SUM)             # train_utils.py:155-157
            loss = loss / self.world_size
        if update:
            grads, self._accum = self._accum, None
            if self.distributed:
                red = GradBucketReducer(self.world_size)
                for k, g in grads.items():
                    red.add(k, g)
                grads = red.finish()
            self.last_grad_sq = self.optimizer.step(grads, lr=lr)
            if hasattr(self.model, "mark_weights_changed"):
                self.model.mark_weights_changed()                       # sampling plans re-pack the updated weights
        return loss


class DistillationStep(TrainingStep):
    """One stage of progressive distillation (Salimans & Ho, 2022): ``student`` learns to sample in N =
    ``diffusion.sample_timesteps`` DDIM steps what ``teacher`` does in 2N (GaussianDiffusion.distill_loss).  Only ``draw`` and
    ``loss_and_grads`` differ from TrainingStep, so ``step()``, gradient accumulation, the all-reduce, clip + AdamW + EMA and the
    checkpoints are the training step's own.

        ds = DistillationStep(student, teacher, diffusion, w_guide=0., lr=1e-4, ema_decay=0.9995)
        loss = ds.step(x, y)

    The teacher runs in ``.eval()`` on the sampling (plan) path.  With ``w_guide`` = 0 the labels are dropped (set to 0, "no
    class") with probability ``diffusion.p_uncond`` before either network sees them, so the student keeps its unconditional
    branch and can still be sampled with CFG.  With ``w_guide`` > 0 the teacher is guided, no label is dropped, and the student
    learns the guided prediction: sample it with ``w_guide`` = 0."""

    def __init__(self, student, teacher, diffusion, w_guide=0., **kwargs):
        super().__init__(student, diffusion, **kwargs)
        self.teacher = teacher.eval()
        self.w_guide = float(w_guide)
        if self.w_guide < 0:
            raise ValueError(f"w_guide must be >= 0, got {w_guide}")

    def draw(self, x):
        """From the step's generator, in this order: the student step indices i ~ U{0 .. N-1}, the noise, then the label-keep
        mask (uniforms >= p_uncond; drawn every step, so the stream does not depend on the labels or on w_guide)."""
        B, N = x.shape[0], int(self.diffusion.sample_timesteps)
        step = torch.randint(N, size=(B,), device=self.device, generator=self.generator)
        noise = torch.empty_like(x).normal_(generator=self.generator)
        keep = torch.rand((B,), device=self.device, generator=self.generator) >= float(self.diffusion.p_uncond or 0.)
        return step, noise, keep

    @torch.no_grad()
    def loss_and_grads(self, x, y, step=None, noise=None, keep=None):
        """Per-sample distillation loss (B,) and the gradients of ``loss.mean()`` w.r.t. every student parameter."""
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if step is None or noise is None or keep is None:
            step, noise, keep = self.draw(x)
        if y is not None and self.w_guide == 0:
            y = y.to(self.device)
            y = y * keep.to(y.dtype).reshape((-1,) + (1,) * (y.ndim - 1))
        loss, grad_out = self.diffusion.distill_loss(self.teacher, self.graph.forward, x, step, y, noise=noise,
                                                     w_guide=self.w_guide, return_grad=True)
        return loss, self.graph.backward(grad_out)
