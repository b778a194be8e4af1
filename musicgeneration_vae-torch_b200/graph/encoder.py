"""Bar encoder 1x96x60 -> 1152 (reference: graph/encoder.py:8-40) and the shared trunk used by the phrase encoder
(graph/phrase_encoder.py:8-41).  One autograd node per call: forward keeps bf16 NHWC activations, backward runs
the hand-written data/weight-gradient kernels and accumulates straight into the parameters' .grad buffers."""
import torch
import torch.nn as nn

from ..engine import BF16, Act, async_wgrad, saving
from .encodingBlock import PitchTimeModule, PoolingModule, ResidualModule, TimePitchModule, gemm_of
from .weights_initializer import weights_init


class _TrunkFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, *params):
        need = any(ctx.needs_input_grad)
        with saving(need):
            z, saved = module._fwd(x, need)
        ctx.module, ctx.saved = module, saved
        ctx.stream = torch.cuda.current_stream()
        if getattr(module, "_bvae_keep_state", False):      # parity tests read the stored forward state (tests/gpu_util.py)
            module._bvae_state = (z, saved)
        return z

    @staticmethod
    def backward(ctx, dz):
        cur0 = torch.cuda.current_stream()
        if cur0 != torch.cuda.default_stream(cur0.device) and not torch.cuda.is_current_stream_capturing():
            dz.record_stream(cur0)       # produced on the decoder's stream, dropped by autograd when this node returns
        with async_wgrad():
            ctx.module._bwd(ctx.saved, dz)
        ctx.saved = None
        cb = getattr(ctx.module, "_bvae_on_bwd_done", None)  # parallel.GradReducer: this segment's gradients are complete
        if cb is not None:                                   # (after the weight-gradient stream has been joined)
            cb()
        # The parameter gradients are written by our kernels on THIS node's stream (autograd replays the forward
        # stream) and are not returned to autograd, so its end-of-backward stream sync does not cover them: when the
        # node ran on a side stream, make the stream that called backward() wait for it.
        cur = torch.cuda.current_stream()
        if cur != torch.cuda.default_stream(cur.device):
            ev = torch.cuda.Event()
            ev.record(cur)
            torch.autograd.Variable._execution_engine.queue_callback(lambda: torch.cuda.current_stream().wait_event(ev))
        return (None, None) + (None,) * len(ctx.module._plist)


class _EncoderTrunk(nn.Module):
    def _build(self, layers, linear_bias):
        self.time_pitch = TimePitchModule()
        self.pitch_time = PitchTimeModule()
        blocks = []
        for i in range(1, len(layers)):
            blocks.append(ResidualModule(layers[i - 1]))
            blocks.append(PoolingModule(layers[i - 1], layers[i]))
        self.layers = nn.ModuleList(blocks)
        self.linear = nn.Linear(1024, 1152, bias=linear_bias)
        self.apply(weights_init)

    def forward(self, x):
        if not x.is_cuda:
            raise RuntimeError("the B200 path needs CUDA tensors; there is no CPU fallback")
        self._plist = list(self.parameters())
        return _TrunkFn.apply(self, x, *self._plist)

    def encode(self, x):
        """Inference only: ``forward(x)`` without the autograd node and with nothing saved for a backward pass (under
        ``torch.no_grad`` the node would still save, because the parameters require grad).  ``x`` may be fp32 or bf16."""
        if torch.is_grad_enabled():
            raise RuntimeError("encode is inference-only: call it under torch.no_grad()")
        if not x.is_cuda:
            raise RuntimeError("the B200 path needs CUDA tensors; there is no CPU fallback")
        with saving(False):
            return self._fwd(x, False)[0]

    # ---- fused forward / backward over engine.Act views ------------------------------------------------
    def _fwd(self, x, save):
        B, _, H, W = x.shape
        xb = Act(x.detach().to(BF16).contiguous(), B, H, W, 1)      # C == 1: NCHW is NHWC
        cat = Act.empty(B, H // 2, W // 2, 64)                       # torch.cat((pitch, time), 1) never materialised
        c_pt = self.pitch_time.fwd(xb, cat.slice(0, 32))
        c_tp = self.time_pitch.fwd(xb, cat.slice(32, 32))
        h, ctxs = cat, []
        for layer in self.layers:
            oh, ow, oc = layer.out_shape(h.H, h.W)
            out = Act.empty(B, oh, ow, oc)
            ctxs.append(layer.fwd(h, out))
            h = out
        HW = h.H * h.W                                                # AvgPool2d((3,2)) / ((12,2)): the whole map
        pooled = h.t.view(B, HW, 1024).float().mean(1).to(BF16)
        pa = Act(pooled, B, 1, 1, 1024)
        z = Act.empty(B, 1, 1, 1152, dtype=torch.float32)
        gemm_of(self.linear).forward(pa, z)
        saved = (c_pt, c_tp, ctxs, pa, (h.H, h.W), cat) if save else None
        return z.t.view(B, 1152), saved

    def _bwd(self, saved, dz):
        c_pt, c_tp, ctxs, pa, (fh, fw), cat = saved
        B = dz.shape[0]
        lin = gemm_of(self.linear)
        dz = dz.contiguous().float()
        dzb = Act(dz.to(BF16), B, 1, 1, 1152)
        lin.wgrad(pa, dzb)
        lin.bias_grad(Act(dz, B, 1, 1, 1152))
        dp = Act.empty(B, 1, 1, 1024)
        lin.dgrad(dzb, dp)
        HW = fh * fw
        dh = (dp.t.view(B, 1, 1024).float() / HW).to(BF16).expand(B, HW, 1024).contiguous()
        d = Act(dh, B, fh, fw, 1024)
        for layer, c in zip(reversed(self.layers), reversed(ctxs)):
            d = layer.bwd(c, d)
        self.time_pitch.bwd(c_tp, d.slice(32, 32))
        self.pitch_time.bwd(c_pt, d.slice(0, 32))


class Encoder(_EncoderTrunk):
    def __init__(self, layers):
        super().__init__()
        self._build(layers, linear_bias=True)
