"""Decoder 1152-latents -> 1x96x60 bar (reference: graph/decoder.py:8-222).

Latent head (embedding, two Linears, ReLU, Dropout) -> two k==stride ConvTranspose stems to 1024x6x3 -> fit1 ->
four up-sampling blocks (strided ConvTranspose pairs, sub-pixel decomposed) -> fit2 + sigmoid.  Contractions run
as tcgen05 implicit GEMMs, every InstanceNorm/CBAM/ReLU site as one fused norm block, fit2+sigmoid as one
memory-bound kernel.  Embedding lookup and the dropout mask stay in PyTorch (tiny [B,1152] tensors; keeps the
Philox dropout stream a torch one).  Replicated defect: DeConvPitchPadding applies bn2 to both branches and never
uses bn1 (decoder.py:137,142)."""
import torch
import torch.nn as nn

from .. import _lib
from ..engine import BF16, Act, async_wgrad, fork, fork_enabled, grad_ptr, raw_dtype, saving
from .cbam import CBAM
from .encodingBlock import _norm, gemm_of, norm_block
from .weights_initializer import weights_init


class _HeadModule(nn.Module):
    """ConvT(2304->1024, k=s) -> ReLU -> ConvT(1024->1024, k=s) -> IN -> out + CBAM(out) -> ReLU  (decoder.py:25-36,55-66)"""
    FIRST = SECOND = None

    def _build(self, first, second):
        spec = {"time": dict(kernel_size=(6, 1), stride=(6, 1)), "pitch": dict(kernel_size=(1, 3), stride=(1, 3))}
        setattr(self, first, nn.ConvTranspose2d(2304, 1024, bias=False, **spec[first]))
        setattr(self, second, nn.ConvTranspose2d(1024, 1024, bias=False, **spec[second]))
        self.bn = _norm(1024)
        self.cbam = CBAM(1024)
        self.apply(weights_init)

    def fwd(self, x: Act, out: Act):
        g1, g2 = gemm_of(getattr(self, self.FIRST)), gemm_of(getattr(self, self.SECOND))
        h1, w1 = g1.out_hw(x.H, x.W)
        t1 = Act.empty(x.N, h1, w1, 1024)
        g1.forward(x, t1, act=True, slope=0.0)
        y = Act.empty(x.N, out.H, out.W, 1024, dtype=raw_dtype())
        st = g2.forward(t1, y, want_stats=True)
        nb = norm_block(self.bn, self.cbam, 1, 0.0)
        return (x, t1, nb, nb.forward(y, out, stats=st))

    def bwd(self, ctx, dout: Act, dx: Act, accumulate: bool):
        x, t1, nb, nctx = ctx
        g1, g2 = gemm_of(getattr(self, self.FIRST)), gemm_of(getattr(self, self.SECOND))
        dy = Act.empty(dout.N, dout.H, dout.W, 1024)
        nb.backward(nctx, dout, dy)
        g2.wgrad(t1, dy)
        dt1 = Act.empty(t1.N, t1.H, t1.W, 1024)
        g2.dgrad(dy, dt1, mask=t1, mask_slope=0.0)
        g1.wgrad(x, dt1)
        g1.dgrad(dt1, dx, addend=dx if accumulate else None)


class TimePitchModule(_HeadModule):
    FIRST, SECOND = "time", "pitch"

    def __init__(self):
        super().__init__()
        self._build("time", "pitch")


class PitchTimeModule(_HeadModule):
    FIRST, SECOND = "pitch", "time"

    def __init__(self):
        super().__init__()
        self._build("pitch", "time")


class _UpBlock(nn.Module):
    """Two transposed-conv branches -> IN -> ReLU, concatenated -> 1x1 conv -> IN -> out + CBAM(out) -> ReLU."""

    def _branches(self):
        raise NotImplementedError

    def out_shape(self, H, W):
        h, w = gemm_of(self.deConv1).out_hw(H, W)
        return h, w, self.conv.out_channels

    def fwd(self, x: Act, out: Act):
        Cc = out.C
        cat = Act.empty(out.N, out.H, out.W, 2 * Cc)

        def branch(i, deconv, bn, cbam, mode):
            g = gemm_of(deconv)
            y = Act.empty(out.N, out.H, out.W, Cc, dtype=raw_dtype())
            st = g.forward(x, y, want_stats=True)
            nb = norm_block(bn, cbam, mode, 0.0)
            return (g, nb, nb.forward(y, cat.slice(i * Cc, Cc), stats=st))

        b0, b1 = self._branches()
        if fork_enabled():                      # engine.fork: second branch on the companion stream
            with fork() as f:
                c1 = branch(1, *b1)
            bctx = [branch(0, *b0), c1]
            f.join()
        else:
            bctx = [branch(0, *b0), branch(1, *b1)]
        g3 = gemm_of(self.conv)
        y3 = Act.empty(out.N, out.H, out.W, Cc, dtype=raw_dtype())
        st3 = g3.forward(cat, y3, want_stats=True)
        nb3 = norm_block(self.bn3, self._last_cbam(), 1, 0.0)
        return (x, cat, bctx, g3, nb3, nb3.forward(y3, out, stats=st3))

    def bwd(self, ctx, dout: Act) -> Act:
        x, cat, bctx, g3, nb3, n3ctx = ctx
        Cc = dout.C
        dy3 = Act.empty(dout.N, dout.H, dout.W, Cc)
        nb3.backward(n3ctx, dout, dy3)
        g3.wgrad(cat, dy3)
        dcat = Act.empty(dout.N, dout.H, dout.W, 2 * Cc)
        g3.dgrad(dy3, dcat)
        dx = Act.empty(x.N, x.H, x.W, x.C)
        # DeConvPitchPadding applies ONE InstanceNorm (bn2) to both branches: their backward passes accumulate into the
        # same d-gamma / d-beta and must stay ordered on one stream
        if not fork_enabled() or bctx[0][1].gamma is bctx[1][1].gamma:
            for i, (g, nb, nctx) in enumerate(bctx):
                dy = Act.empty(dout.N, dout.H, dout.W, Cc)
                nb.backward(nctx, dcat.slice(i * Cc, Cc), dy)
                g.wgrad(x, dy)
                g.zero_bias_grad()          # bias feeds an InstanceNorm: gradient is identically zero
                g.dgrad(dy, dx, addend=dx if i > 0 else None)
            return dx
        # engine.fork: norm-block backward of the second branch on the companion stream; its weight /
        # data gradients follow after the join (no weight-gradient launch inside a fork)
        dys = [None, None]
        with fork() as f:
            dys[1] = Act.empty(dout.N, dout.H, dout.W, Cc)
            bctx[1][1].backward(bctx[1][2], dcat.slice(Cc, Cc), dys[1])
        dys[0] = Act.empty(dout.N, dout.H, dout.W, Cc)
        bctx[0][1].backward(bctx[0][2], dcat.slice(0, Cc), dys[0])
        for i, (g, nb, nctx) in enumerate(bctx):
            if i == 1:
                f.join()
            g.wgrad(x, dys[i])
            g.zero_bias_grad()
            g.dgrad(dys[i], dx, addend=dx if i > 0 else None)
        return dx


class DeConvModule(_UpBlock):
    """decoder.py:69-109 (layers 2, 3)."""

    def __init__(self, in_channel, out_channel):
        super().__init__()
        self.deConv1 = nn.ConvTranspose2d(in_channel, out_channel, 4, 2, 1, bias=False)
        self.deConv2 = nn.ConvTranspose2d(in_channel, out_channel, 3, 2, 1, output_padding=1, bias=True)
        self.conv = nn.Conv2d(in_channel, out_channel, 1, 1, bias=False)
        self.bn1, self.bn2, self.bn3 = _norm(out_channel), _norm(out_channel), _norm(out_channel)
        self.cbam = CBAM(out_channel)
        self.apply(weights_init)

    def _branches(self):
        return ((self.deConv1, self.bn1, None, 0), (self.deConv2, self.bn2, None, 0))

    def _last_cbam(self):
        return self.cbam


class DeConvPitchPadding(_UpBlock):
    """decoder.py:112-154 (layers 0, 1): odd output width via output_padding=(0,1); bn2 shared by both branches."""

    def __init__(self, in_channel, out_channel):
        super().__init__()
        self.deConv1 = nn.ConvTranspose2d(in_channel, out_channel, 4, 2, 1, output_padding=(0, 1), bias=True)
        self.deConv2 = nn.ConvTranspose2d(in_channel, out_channel, 4, 2, 1, output_padding=(0, 1), bias=True)
        self.conv = nn.Conv2d(in_channel, out_channel, 1, 1, bias=False)
        self.bn1, self.bn2, self.bn3 = _norm(out_channel), _norm(out_channel), _norm(out_channel)
        self.cbam1 = CBAM(out_channel)
        self.cbam2 = CBAM(out_channel)
        self.apply(weights_init)

    def _branches(self):
        return ((self.deConv1, self.bn2, self.cbam1, 1), (self.deConv2, self.bn2, None, 0))

    def _last_cbam(self):
        return self.cbam2


class _DecoderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, z, pre_z, phrase_feature, position, masks, *params):
        need = any(ctx.needs_input_grad)
        with saving(need):
            recon, saved = module._fwd(z, pre_z, phrase_feature, position, masks, need)
        ctx.module, ctx.saved = module, saved
        if getattr(module, "_bvae_keep_state", False):      # parity tests read the stored forward state (tests/gpu_util.py)
            module._bvae_state = (recon, saved)
        return recon

    @staticmethod
    def backward(ctx, drecon):
        with async_wgrad():
            dz, dpz, dpf = ctx.module._bwd(ctx.saved, drecon)
        ctx.saved = None
        cb = getattr(ctx.module, "_bvae_on_bwd_done", None)  # parallel.GradReducer: decoder gradients are complete
        if cb is not None:                                   # (after the weight-gradient stream has been joined)
            cb()
        return (None, dz, dpz, dpf, None, None) + (None,) * len(ctx.module._plist)


class Decoder(nn.Module):
    def __init__(self, layers):      # [1024, 512, 256, 128, 64]
        super().__init__()
        self.dropout = nn.Dropout(p=0.3)
        self.bar_linear = nn.Linear(1152 * 2, 1152)
        self.phrase_linear = nn.Linear(1152 * 2, 1152)
        self.time = TimePitchModule()
        self.pitch = PitchTimeModule()
        self.fit1 = nn.Conv2d(2048, 1024, 1, 1, bias=False)
        self.bn = _norm(1024)
        self.fit2 = nn.Conv2d(64, 1, 1, 1, bias=False)
        blocks = []
        for i in range(1, len(layers)):
            cls = DeConvPitchPadding if i < 3 else DeConvModule
            blocks.append(cls(layers[i - 1], layers[i]))
        self.layers = nn.ModuleList(blocks)
        self.cbam = CBAM(1024)
        self.position_embedding = nn.Embedding(332, 1152)
        nn.init.uniform_(self.position_embedding.weight, -1.0, 1.0)
        self.apply(weights_init)

    def forward(self, z, pre_z, phrase_feature, position, dropout_masks=None):
        """Same call as the reference (decoder.py:192).  ``dropout_masks`` = (phrase_keep, bar_keep) 0/1 tensors
        lets a test inject the Dropout(0.3) draws; by default they are drawn with torch's CUDA generator in the
        reference's order (phrase branch first, decoder.py:196,201) when the module is in training mode."""
        if not z.is_cuda:
            raise RuntimeError("the B200 path needs CUDA tensors; there is no CPU fallback")
        if dropout_masks is None and self.training:
            ones = torch.ones(z.shape[0], 1152, device=z.device)
            dropout_masks = ((self.dropout(ones) != 0).float(), (self.dropout(ones) != 0).float())
        self._plist = list(self.parameters())
        return _DecoderFn.apply(self, z, pre_z, phrase_feature, position, dropout_masks, *self._plist)

    # ---------------------------------------------------------------------------------------------------
    def forward_logits(self, z, pre_z, phrase_feature, position):
        """Inference only (no dropout, nothing saved for a backward pass): ``(probs, logits)``, both [B,1,96,60] fp32
        from ONE fit2 + sigmoid launch, so ``probs`` is what ``forward`` returns and ``logits`` the values it squashed.
        The sampling loop's Bernoulli mode draws from the logits at a temperature (data/packed.bernoulli_sample)."""
        if torch.is_grad_enabled():
            raise RuntimeError("Decoder.forward_logits is inference-only: call it under torch.no_grad()")
        if self.training:
            raise RuntimeError("Decoder.forward_logits is inference-only: put the module in eval() mode (no dropout)")
        if not z.is_cuda:
            raise RuntimeError("the B200 path needs CUDA tensors; there is no CPU fallback")
        logits = torch.empty((z.shape[0], 1, 96, 60), dtype=torch.float32, device=z.device)
        with saving(False):
            probs, _ = self._fwd(z, pre_z, phrase_feature, position, None, False, logits=logits)
        return probs, logits

    def _fwd(self, z, pre_z, pf, position, masks, save, logits=None):
        B = z.shape[0]
        emb = self.position_embedding.weight.detach()[position]
        pcat = Act(torch.cat((pf.detach().float(), emb), 1).to(BF16), B, 1, 1, 2304)
        bcat = Act(torch.cat((z.detach().float(), pre_z.detach().float()), 1).to(BF16), B, 1, 1, 2304)
        lin = Act.empty(B, 1, 1, 2304)                      # [relu(bar_linear) | relu(phrase_linear)]
        gb, gp = gemm_of(self.bar_linear), gemm_of(self.phrase_linear)
        gb.forward(bcat, lin.slice(0, 1152), act=True, slope=0.0)
        gp.forward(pcat, lin.slice(1152, 1152), act=True, slope=0.0)
        if masks is not None:
            # nn.Dropout scales the kept values by 1/(1-p) in fp32 (decoder.py:196,201); the product is rounded once
            keep = torch.cat((masks[1], masks[0]), 1).float() * (1.0 / 0.7)      # bar first in the concat
            x = Act((lin.t.view(B, 2304).float() * keep).to(BF16), B, 1, 1, 2304)
        else:
            keep, x = None, lin
        hcat = Act.empty(B, 6, 3, 2048)                     # torch.cat((pitch, time), 1)
        if fork_enabled():                      # engine.fork: the two head stems are independent
            with fork() as f:
                c_t = self.time.fwd(x, hcat.slice(1024, 1024))
            c_p = self.pitch.fwd(x, hcat.slice(0, 1024))
            f.join()
        else:
            c_p = self.pitch.fwd(x, hcat.slice(0, 1024))
            c_t = self.time.fwd(x, hcat.slice(1024, 1024))
        g1 = gemm_of(self.fit1)
        y = Act.empty(B, 6, 3, 1024, dtype=raw_dtype())
        st1 = g1.forward(hcat, y, want_stats=True)
        nb = norm_block(self.bn, self.cbam, 1, 0.0)
        h = Act.empty(B, 6, 3, 1024)
        c_f = nb.forward(y, h, stats=st1)
        ctxs = []
        for layer in self.layers:
            oh, ow, oc = layer.out_shape(h.H, h.W)
            out = Act.empty(B, oh, ow, oc)
            ctxs.append(layer.fwd(h, out))
            h = out
        rows = B * h.H * h.W
        recon = torch.empty((B, 1, h.H, h.W), dtype=torch.float32, device=z.device)
        if logits is not None:
            assert logits.dtype == torch.float32 and logits.is_contiguous() and logits.numel() == rows
        _lib.check(_lib.lib().bvae_fit_sigmoid_fwd(h.ptr, h.pitch, self.fit2.weight.data_ptr(), rows, 64,
                                                   None if logits is None else logits.data_ptr(),
                                                   recon.data_ptr(), _lib.stream_ptr()), "fit_sigmoid_fwd")
        saved = (position, pcat, bcat, lin, keep, x, hcat, c_p, c_t, nb, c_f, ctxs, h, recon) if save else None
        return recon, saved

    def _bwd(self, saved, drecon):
        position, pcat, bcat, lin, keep, x, hcat, c_p, c_t, nb, c_f, ctxs, h, recon = saved
        B = recon.shape[0]
        rows = B * h.H * h.W
        drecon = drecon.contiguous().float()
        d = Act.empty(B, h.H, h.W, 64)
        _lib.check(_lib.lib().bvae_fit_sigmoid_bce_bwd(h.ptr, h.pitch, self.fit2.weight.data_ptr(), recon.data_ptr(),
                                                       None, drecon.data_ptr(), 1.0, 0, rows, 64, d.ptr, d.pitch,
                                                       grad_ptr(self.fit2.weight), _lib.stream_ptr()),
                   "fit_sigmoid_bce_bwd")
        for layer, c in zip(reversed(self.layers), reversed(ctxs)):
            d = layer.bwd(c, d)
        g1 = gemm_of(self.fit1)
        dy = Act.empty(B, 6, 3, 1024)
        nb.backward(c_f, d, dy)
        g1.wgrad(hcat, dy)
        dh = Act.empty(B, 6, 3, 2048)
        g1.dgrad(dy, dh)
        dx = Act.empty(B, 1, 1, 2304)
        self.pitch.bwd(c_p, dh.slice(0, 1024), dx, accumulate=False)
        self.time.bwd(c_t, dh.slice(1024, 1024), dx, accumulate=True)
        # dropout + ReLU backward on the [B,2304] latent features (tiny; PyTorch glue)
        dl = dx.t.view(B, 2304)
        if keep is not None:
            dl = (dl.float() * keep).to(BF16)
        dl = (dl * (lin.t.view(B, 2304) > 0)).contiguous()
        dlin = Act(dl, B, 1, 1, 2304)
        gb, gp = gemm_of(self.bar_linear), gemm_of(self.phrase_linear)
        dbar, dphr = dlin.slice(0, 1152), dlin.slice(1152, 1152)
        gb.wgrad(bcat, dbar)
        gb.bias_grad(dbar)
        gp.wgrad(pcat, dphr)
        gp.bias_grad(dphr)
        dbc = Act.empty(B, 1, 1, 2304)
        dpc = Act.empty(B, 1, 1, 2304)
        gb.dgrad(dbar, dbc)
        gp.dgrad(dphr, dpc)
        dbc_f = dbc.t.view(B, 2304).float()
        dpc_f = dpc.t.view(B, 2304).float()
        emb_w = self.position_embedding.weight
        if emb_w.requires_grad:
            grad_ptr(emb_w)
            emb_w.grad.index_add_(0, position, dpc_f[:, 1152:])
        return dbc_f[:, :1152].contiguous(), dbc_f[:, 1152:].contiguous(), dpc_f[:, :1152].contiguous()
