"""Training path of the drop-in backbone (SURVEY §8 row f-3 / BASELINE config 5): ``torch.autograd.Function`` around
``madm_extract(MADM_FLAG_TRAIN)`` / ``madm_backward``.

The reference's student passes call the backbone under grad (``modeling/meta_arch/mtmadise.py:240-256, :286-302``) and
``AMPTrainer.run_step`` back-propagates the summed losses through it (``engine/train_loop.py:277-302``).  Here the same call returns
feature maps that carry a ``grad_fn``; ``loss.backward()`` then runs the CUDA engine's backward pass and hands autograd the gradients of

* the ACTIVE adapter's ``lora_A`` / ``lora_B`` factors (128 wrapped projections),
* ``backbone.feature_projections`` (conv weights + GroupNorm affines),
* ``cond_inputs`` / ``cond_emb`` — from which autograd itself reaches the learned prompt / time parameters through the tiny
  ``tanh(alpha) * embed`` arithmetic that stays in PyTorch (``ldm_base.py:675-717``).

In the ``vae_decoder_loss`` / s0 variant the VAE decoder runs under ``no_grad`` and its image is detached before it becomes the first
feature (``ldm_diffusers.py:191-201``): ``s0`` back-propagates into ``feature_projections.0`` only.  With ``return_unet_final_output=True``
the UNet's final output ``before_vae.decoder`` carries grad (the meta-arch's ``vae_decoder_loss`` differentiates it) and
``after_vae.decoder`` does not.

Everything else must be frozen: BASELINE.json narrows the training configuration to LoRA gradients, so a call under grad with trainable
BASE UNet weights (``finetune_unet='all'`` without freezing them) raises instead of silently dropping their gradients.  Several forwards
may be in flight before one ``backward()`` (source pass + mixed pass, different adapters): each holds its own training workspace and
input-gradient weight arena until its backward has run.  torch tensors are device memory only; there is no eager fallback.
"""
import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import MadmBackwardArgs, MadmExtractArgs, MadmTensor
from .engine import OUT_SHAPES

_UNSUPPORTED = ("madm_b200's backward pass covers the LoRA training step's trainable set (active adapter's lora_A / lora_B, "
                "feature_projections, prompt / time conditioning; BASELINE config 5). {} Freeze them (requires_grad_(False)) or wrap "
                "inference in torch.no_grad().")


class _Slot:
    """Resources one in-flight training forward owns until its backward has run."""

    def __init__(self):
        self.ws: Optional[torch.Tensor] = None
        self.dgrad: Optional[torch.Tensor] = None
        self.dgrad_sig = None
        self.busy = False


class TrainContext:
    """Per-backbone state of the training path: slots, the registered gradient buffers."""

    def __init__(self, backbone):
        self.backbone = backbone
        self.slots: List[_Slot] = []
        self.grad_sig = None
        self.grad_src = None
        self.grad_flat: Optional[torch.Tensor] = None
        self.grad_views: Dict[str, torch.Tensor] = {}
        self.grad_slices: Dict[str, Tuple[int, int, Tuple[int, ...]]] = {}

    # ------------------------------------------------------------------ gradient buffers (one flat fp32 buffer, views per parameter)
    def ensure_grads(self, eng, named: Sequence[Tuple[str, torch.Tensor]]):
        if named is self.grad_src:  # the cached list object: nothing can have changed
            return
        sig = tuple((n, tuple(t.shape)) for n, t in named)
        if sig == self.grad_sig:
            self.grad_src = named
            return
        total = sum(t.numel() for _, t in named)
        self.grad_flat = torch.zeros(total, dtype=torch.float32, device=eng.device)
        self.grad_views = {}
        self.grad_slices = {}
        arr = (MadmTensor * len(named))()
        keep = [n.encode() for n, _ in named]
        off = 0
        for i, (n, t) in enumerate(named):
            v = self.grad_flat[off:off + t.numel()].view(t.shape)
            off += t.numel()
            self.grad_views[n] = v
            self.grad_slices[n] = (off - t.numel(), t.numel(), tuple(t.shape))
            arr[i].name, arr[i].data, arr[i].ndim = keep[i], v.data_ptr(), t.dim()
            for k, s in enumerate(t.shape):
                arr[i].shape[k] = s
        _lib.check(eng.lib.madm_set_grad_tensors(eng.ctx, arr, len(named)), eng.ctx, "madm_set_grad_tensors")
        self.grad_sig, self.grad_src = sig, named
        for s in self.slots:  # plans were dropped; sizes may have changed
            s.ws = None

    def acquire(self) -> _Slot:
        for s in self.slots:
            if not s.busy:
                s.busy = True
                return s
        s = _Slot()
        s.busy = True
        self.slots.append(s)
        return s


def _context(backbone) -> TrainContext:
    tc = getattr(backbone, "_train_ctx", None)
    if tc is None:
        tc = TrainContext(backbone)
        object.__setattr__(backbone, "_train_ctx", tc)
    return tc


def trainable_sets(backbone, grad_inputs: Sequence[Tuple[str, torch.Tensor]]):
    """Split the parameters that require grad into (engine-side trainables of this call, conditioning parameters); raise for the rest."""
    ldm = backbone.feature_extractor.ldm_extractor
    adapter = ldm.unet.active_adapter()
    upre, ppre = "feature_extractor.ldm_extractor.unet.", "feature_projections."
    engine_side, cond_side, bad = [], [], []
    for n, p in grad_inputs:
        if n.startswith(upre):
            if ".lora_A." in n or ".lora_B." in n:
                if adapter is not None and f".{adapter}." in n:
                    engine_side.append((n, p))
                # factors of the other adapters do not take part in this forward: no gradient (the reference adds explicit zeros,
                # mtmadise.py:149-157; optim.allreduce_grads materialises them)
            else:
                bad.append(n)
        elif n.startswith(ppre):
            engine_side.append((n, p))
        else:
            cond_side.append((n, p))
    if bad:
        raise NotImplementedError(_UNSUPPORTED.format(f"{len(bad)} base UNet weights require grad (e.g. {bad[0]})."))
    return adapter, engine_side, cond_side


class _ExtractFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, backbone, slot, eng, adapter, scaling, loss_scale, names, want_final, img, cond_inputs, cond_emb, timesteps, *params):
        dev = eng.device
        B = img.shape[0]
        lib = eng.lib
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        ad = (adapter or "").encode()
        # input-gradient operands of this slot: repacked when a parameter or the adapter changed
        need = lib.madm_dgrad_packed_bytes(eng.ctx)
        if need == 0:
            _lib.check(-1, eng.ctx, "madm_dgrad_packed_bytes")
        sig = (eng._version_vector(), adapter, id(eng._named))
        if slot.dgrad is None or slot.dgrad.numel() != need:
            slot.dgrad, slot.dgrad_sig = torch.empty(need, dtype=torch.uint8, device=dev), None
        if slot.dgrad_sig != sig:
            old = slot.dgrad_sig
            partial = old is not None and old[2] == sig[2] and eng.only_trainables_changed(old[0], sig[0])
            _lib.check(lib.madm_pack_dgrad_weights(eng.ctx, C.c_void_p(slot.dgrad.data_ptr()), ad, float(scaling), 1 if partial else 0, st),
                       eng.ctx, "madm_pack_dgrad_weights")
            slot.dgrad_sig = sig
        wneed = lib.madm_train_workspace_bytes(eng.ctx, B, ad)
        if wneed == 0:
            _lib.check(-1, eng.ctx, "madm_train_workspace_bytes")
        if slot.ws is None or slot.ws.numel() < wneed:
            slot.ws = torch.empty(wneed, dtype=torch.uint8, device=dev)
        img = img.detach().to(torch.float32).contiguous()
        ci = cond_inputs.detach().to(torch.float32).expand(B, 77, 768).contiguous()
        ce = cond_emb.detach().to(torch.float32).reshape(-1, 1280).expand(B, 1280).contiguous()
        ts = timesteps.to(device=dev, dtype=torch.int64).contiguous()
        noise = backbone.feature_extractor.ldm_extractor.shared_noise
        outs = [torch.empty(B, ch, side, side, dtype=torch.float32, device=dev) for ch, side in OUT_SHAPES[eng.variant]]
        a = MadmExtractArgs()
        a.B, a.stages, a.ema, a.flags = B, eng.stage_all, 0, _lib.FLAG_TRAIN
        a.img, a.cond_inputs, a.cond_emb, a.timesteps = img.data_ptr(), ci.data_ptr(), ce.data_ptr(), ts.data_ptr()
        a.shared_noise = noise.data_ptr()
        for i, t in enumerate(outs):
            a.out[i] = t.data_ptr()
        a.packed = eng._packed.data_ptr()
        a.workspace, a.workspace_bytes = slot.ws.data_ptr(), slot.ws.numel()
        a.range_flag = eng.range_flag.data_ptr()
        a.packed_dgrad = slot.dgrad.data_ptr()
        a.train_adapter, a.train_lora_scale, a.train_loss_scale = ad, float(scaling), float(loss_scale)
        final = ()
        if want_final:  # 'before_vae.decoder' (differentiable), 'after_vae.decoder' (not: the decoder runs under no_grad)
            final = (torch.empty(B, 4, 64, 64, dtype=torch.float32, device=dev), torch.empty(B, 3, 512, 512, dtype=torch.float32, device=dev))
            a.unet_sample, a.decoded = final[0].data_ptr(), final[1].data_ptr()
            ctx.mark_non_differentiable(final[1])
        eng._range_poll()
        _lib.check(lib.madm_extract(eng.ctx, C.byref(a), st), eng.ctx, "madm_extract(train)")
        eng._range_publish()
        ctx.backbone, ctx.slot, ctx.eng, ctx.names = backbone, slot, eng, names
        ctx.adapter, ctx.scaling, ctx.loss_scale = ad, float(scaling), float(loss_scale)
        ctx.packed_ptr = eng._packed.data_ptr()
        ctx.keep = (img, ci, ts)
        ctx.cond_shapes = (tuple(cond_inputs.shape), tuple(cond_emb.shape))
        ctx.save_for_backward(ce, *outs)
        ctx.set_materialize_grads(False)
        return tuple(outs) + final

    @staticmethod
    def backward(ctx, *douts):
        eng, slot = ctx.eng, ctx.slot
        saved = ctx.saved_tensors
        ce, outs = saved[0], saved[1:]
        B = outs[0].shape[0]
        dev = eng.device
        tc = _context(ctx.backbone)
        try:
            d_ci = torch.empty(B, 77, 768, dtype=torch.float32, device=dev)
            d_ce = torch.empty(B, 1280, dtype=torch.float32, device=dev)
            b = MadmBackwardArgs()
            b.B = B
            keep = []
            for i in range(4):
                g = douts[i] if douts[i] is not None else torch.zeros_like(outs[i])
                g = g.to(torch.float32).contiguous()
                keep.append(g)
                b.dout[i], b.out[i] = g.data_ptr(), outs[i].data_ptr()
            if len(douts) > 4 and douts[4] is not None:  # gradient of 'before_vae.decoder'; none: the UNet-output backward does no work
                g = douts[4].to(torch.float32).contiguous()
                keep.append(g)
                b.d_unet_sample = g.data_ptr()
            b.cond_emb, b.d_cond_inputs, b.d_cond_emb = ce.data_ptr(), d_ci.data_ptr(), d_ce.data_ptr()
            b.adapter, b.lora_alpha_over_r, b.loss_scale = ctx.adapter, ctx.scaling, ctx.loss_scale
            b.packed, b.packed_dgrad = ctx.packed_ptr, slot.dgrad.data_ptr()
            b.workspace, b.workspace_bytes = slot.ws.data_ptr(), slot.ws.numel()
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(eng.lib.madm_backward(eng.ctx, C.byref(b), st), eng.ctx, "madm_backward")
            # the flat buffer is overwritten by the next backward: ONE copy of it, the returned gradients are views of that copy
            # (306 per-tensor clones were 306 small launches per pass)
            snap = tc.grad_flat.clone()
            grads = []
            for n in ctx.names:
                off, cnt, shape = tc.grad_slices[n]
                grads.append(snap[off:off + cnt].view(shape))
        finally:
            slot.busy = False
        ci_shape, ce_shape = ctx.cond_shapes
        g_ci = d_ci if ci_shape[0] == B else d_ci.sum(0, keepdim=True)
        g_ce = d_ce.reshape(B, *ce_shape[1:]) if ce_shape[0] == B else d_ce.sum(0, keepdim=True).reshape(1, *ce_shape[1:])
        return (None,) * 8 + (None, g_ci, g_ce, None) + tuple(grads)


def extract_with_grad(backbone, img, input_modal, ema_forward, timestep, grad_inputs, want_taps=False, timesteps=None, **kwargs):
    """``AttentionFeatureExtractorBackbone._extract`` under grad: returns ``{'features': [s2, s3, s4, s5]}`` (s0 variant: s0, s3, s4, s5)
    with a grad_fn, plus ``unet_sample`` / ``decoded`` under ``return_unet_final_output`` (s0 variant)."""
    gen = backbone.feature_extractor
    ldm = gen.ldm_extractor
    if ema_forward:
        raise NotImplementedError(_UNSUPPORTED.format("ema_forward=True under grad (the teacher runs under no_grad, mtmadise.py:335-349)."))
    want_final = bool(kwargs.get("return_unet_final_output"))
    if want_final and backbone.variant != "s0":
        raise NotImplementedError("return_unet_final_output needs vae_decoder_loss=True (the reference raises on decoder_output too)")
    if want_taps or "modality_mask" in kwargs:
        raise NotImplementedError(_UNSUPPORTED.format("Taps / modality_mask are not available under grad."))
    if tuple(img.shape[1:]) != (3, 512, 512):
        raise ValueError(f"the training path expects [B,3,512,512] images, got {tuple(img.shape)}")
    if img.shape[0] > 8:
        raise ValueError("the training path supports up to 8 images per call")
    adapter, engine_side, _ = trainable_sets(backbone, grad_inputs)
    batched = dict(img=img)
    gen.conditioning(batched, input_modal, ema_forward, timestep)  # under grad: autograd reaches the prompt / time parameters
    if timesteps is None:
        timesteps = ldm.sample_timesteps(batched, img.shape[0])
    eng = ldm.prepare(backbone._projection_tensors())
    tc = _context(backbone)
    # gradient buffers for EVERY engine-side trainable (all adapters' factors + projections), so one registration serves all passes
    tc.ensure_grads(eng, _all_engine_trainables(backbone))
    slot = tc.acquire()
    scaling = ldm.unet.scaling_of(adapter) if adapter else 0.0
    loss_scale = float(getattr(ldm, "train_loss_scale", None) or (1.0 if ldm.compute_dtype == "bf16" else 4096.0))
    names = [n for n, _ in engine_side]
    try:
        outs = _ExtractFn.apply(backbone, slot, eng, adapter, scaling, loss_scale, names, want_final, img, batched["cond_inputs"],
                                batched["cond_emb"], timesteps, *[p for _, p in engine_side])
    except Exception:
        slot.busy = False
        raise
    if not any(o.requires_grad for o in outs):  # nothing to back-propagate (e.g. only frozen inputs): release the slot now
        slot.busy = False
    res = {"features": list(outs[:4])}
    if want_final:
        res["unet_sample"], res["decoded"] = outs[4], outs[5]
    return res


def _all_engine_trainables(backbone):
    """Every parameter the engine can produce a gradient for (all adapters' factors + the projections), from the cached name lists."""
    ldm = backbone.feature_extractor.ldm_extractor
    base = ldm.named_engine_tensors(False)
    proj = backbone._projection_tensors()
    hit = getattr(backbone, "_trainables_cache", None)
    if hit is not None and hit[0] is base and hit[1] is proj:
        return hit[2]
    out = [(n, p) for n, p in base if ".lora_A." in n or ".lora_B." in n]
    out += [(n, p) for n, p in proj if n.startswith("feature_projections.")]
    object.__setattr__(backbone, "_trainables_cache", (base, proj, out))
    return out
