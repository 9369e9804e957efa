"""Counterpart of vq_ae/model.py: ``VQAE``, ``Encoder``, ``Decoder`` with the reference's
constructor signatures, attribute names, ``state_dict`` keys and return tuples.

``Encoder.forward`` / ``Decoder.forward`` in eval mode run a packed, NHWC, kernel-by-kernel
plan over the C-ABI library instead of dispatching module by module.  The shipped topology (one VQ
level, no shortcut blocks: conf/model/vq_ae.yaml) runs one fused plan; the multi-level hierarchy of
model.py:144-148,203-215 (row (f)-4 of the scope table) runs the same kernels level by level
(plan.encoder_forward_levels / decoder_forward_levels).  Training (``shared_step``, SAM, logging) is
out of scope.
"""
from __future__ import annotations

from typing import Any, List, Optional, Sequence, Tuple

import torch
from torch import Tensor, nn

from . import engine as E
from . import plan as P
from ._instantiate import instantiate


def maybe_repeat_layer(layer, repetitions: int):
    """utils/train_helpers.py:27-32."""
    if not isinstance(layer, (list, tuple)):
        return [layer] * repetitions
    assert len(layer) == repetitions
    return layer


_flat_blocks = P.flat_blocks      # kept under its round-1 name for profiles/ scripts


class Encoder(nn.Module):
    """in_stem -> DownBlock pyramid -> trunk of 'same' blocks -> quantiser (model.py:129-217)."""

    def __init__(self, stem_conf, down_block_conf, n_pre_enc_layers, vq_conf, conv_block_conf,
                 shortcut_block_conf):
        super().__init__()
        self.in_stem = instantiate(stem_conf)
        vq_layers = instantiate(vq_conf)

        n_pre_enc_layers, down_block_conf, shortcut_block_conf = (
            maybe_repeat_layer(n_pre_enc_layers, len(vq_layers)),
            maybe_repeat_layer(down_block_conf, len(vq_layers)),
            maybe_repeat_layer(shortcut_block_conf, len(vq_layers) - 1),
        )
        pre_enc_conf = [[{**conv_block_conf, **{'mode': 'same'}}] * n for n in n_pre_enc_layers]

        down_layers, pre_enc_layers, shortcut_layers = [], [], []
        current_in = self.in_stem.out_channels
        for down_layer, pre_enc_layer, shortcut_layer in zip(
                down_block_conf, pre_enc_conf, (None, *shortcut_block_conf)):
            down_block = instantiate(down_layer, in_channels=current_in)
            down_layers.append(down_block)
            current_in = down_block.out_channels
            shortcut_layers.append(instantiate(shortcut_layer, in_channels=current_in)
                                   if shortcut_layer is not None else None)
            pre_enc_layers.append(nn.Sequential(*(
                instantiate(layer, in_channels=current_in, out_channels=current_in)
                for layer in pre_enc_layer)))
        del shortcut_layers[0]
        shortcut_layers.append(None)

        # stored low-res first, like the reference (model.py:182-187)
        self.down_layers = nn.ModuleList(down_layers)
        self.pre_enc_layers = nn.ModuleList(reversed(pre_enc_layers))
        self.shortcut_layers = nn.ModuleList(reversed(shortcut_layers))
        self.vq_layers = nn.ModuleList(reversed(vq_layers))
        #: None = follow torch.autocast like the reference (fp32 unless autocast is active);
        #: "fp32" / "fp16" / ... pin the arithmetic (vqae_b200.set_precision)
        self.precision = None

    # -- B200 path -------------------------------------------------------------------------
    def encode(self, x: Tensor, mean=None, std=None, want_quantized: bool = True,
               want_latents: bool = False):
        """(enc or None, indices int64 [B,h,w], loss 0-dim, near_ties 0-dim int32, z or None);
        x: float [B,3,H,W] (NCHW or channels_last) or uint8 [B,H,W,3] -- see plan.encoder_encode."""
        out = P.encoder_encode(self, x, mean, std, want_quantized, want_latents)
        self.vq_layers[0].last_near_ties = out[3]
        return out

    def forward(self, x: Tensor) -> Tuple[Sequence[Tensor], Sequence[Tensor], Sequence[Tensor]]:
        """((enc,), (indices,), (loss,)) -- low-res to high-res order (model.py:189-217)."""
        # one fused plan for the shipped topology; multi-level hierarchies and MBConv pyramids (scope row
        # f-4) run level by level
        out = P.encoder_forward(self, x)
        for vq in self.vq_layers:
            vq.last_near_ties = P.state(vq).last_near_ties
        return out


class Decoder(nn.Module):
    """trunk of 'same' blocks -> UpBlock pyramid -> out_stem (model.py:220-291)."""

    def __init__(self, n_enc_layers: int, stem_conf, up_block_conf, n_post_enc_layers,
                 conv_block_conf, shortcut_block_conf):
        super().__init__()
        self.out_stem = instantiate(stem_conf)
        n_post_enc_layers, up_block_conf, shortcut_block_conf = (
            maybe_repeat_layer(n_post_enc_layers, n_enc_layers),
            maybe_repeat_layer(up_block_conf, n_enc_layers),
            maybe_repeat_layer(shortcut_block_conf, n_enc_layers - 1),
        )
        post_enc_conf = [[{**conv_block_conf, **{'mode': 'same'}}] * n
                         for n in n_post_enc_layers]

        up_layers, post_enc_layers, shortcut_layers = [], [], []
        current_out = self.out_stem.in_channels
        for up_layer, post_enc_layer, shortcut_layer in zip(
                up_block_conf, post_enc_conf, (None, *shortcut_block_conf)):
            up_block = instantiate(up_layer, out_channels=current_out)
            up_layers.append(up_block)
            current_out = up_block.in_channels
            shortcut_layers.append(instantiate(shortcut_layer, out_channels=current_out)
                                   if shortcut_layer is not None else None)
            post_enc_layers.append(nn.Sequential(*(
                instantiate(layer, in_channels=current_out, out_channels=current_out)
                for layer in post_enc_layer)))
        del shortcut_layers[0]
        shortcut_layers.append(None)

        self.up_layers = nn.ModuleList(reversed(up_layers))
        self.post_enc_layers = nn.ModuleList(reversed(post_enc_layers))
        self.shortcut_layers = nn.ModuleList(reversed(shortcut_layers))
        self.precision = None

    def forward(self, x: Sequence[Tensor]) -> Tensor:
        return P.decoder_forward(self, x)


class VQAE(nn.Module):
    """Encoder + decoder assembly (model.py:13-48).  ``optim_conf`` / ``loss_f_conf`` are kept
    for signature and checkpoint compatibility; the loss module is instantiated (it owns no
    parameters in the shipped config) but nothing trains here."""

    def __init__(self, optim_conf, loss_f_conf, encoder_conf, decoder_conf, **kwargs: Any):
        super().__init__()
        self.optim_conf = optim_conf
        self.hparams_conf = dict(optim_conf=optim_conf, loss_f_conf=loss_f_conf,
                                 encoder_conf=encoder_conf, decoder_conf=decoder_conf, **kwargs)
        for attr_name, attr_conf in (('loss_f', loss_f_conf), ('encoder', encoder_conf),
                                     ('decoder', decoder_conf)):
            setattr(self, attr_name, instantiate(attr_conf))
        for key, value in kwargs.items():
            setattr(self, key, value)

    def forward(self, data: Tensor) -> Tuple[Tensor, Sequence[Tensor]]:
        encodings, *_, encoding_loss = self.encoder(data)
        out = self.decoder(encodings)
        return out, encoding_loss

    @torch.no_grad()
    def decode_codes(self, indices: Tensor, channels_last: bool = False) -> Tensor:
        """Decompress stored code maps: embed_code -> proj_out -> Decoder (scope row f-2).  A sequence of
        index maps (low-res first, like the encoder returns them) decodes a multi-level hierarchy."""
        if isinstance(indices, (list, tuple)):
            return self.decoder(tuple(P.decode_codes(vq, idx, channels_last)
                                      for vq, idx in zip(self.encoder.vq_layers, indices)))
        enc = self.encoder.vq_layers[0].decode_codes(indices, channels_last)
        return self.decoder((enc,))

    @torch.no_grad()
    def decode_codes_u8(self, indices: Tensor, mean=None, std=None) -> Tensor:
        """Decompress stored codes [B,h,w] (int64 or uint8, CUDA) to uint8 RGB pixels [B,H,W,3]: the
        decoder of ``decode_codes`` with the normalisation undone inside out_stem's kernel,
        ``rint(v * 255 std_c + 255 mean_c)`` clamped to [0, 255].  ``mean`` / ``std`` default to the
        CAMELYON16 constants, as in ``Encoder.encode``, so ``encoder.encode(decode_codes_u8(idx))`` is a
        round trip.  Precision follows the decoder (``set_precision``, ``torch.autocast``)."""
        return P.decode_codes_u8(self.encoder.vq_layers[0], self.decoder, indices, mean, std)

    def transfer_batch_to_device(self, batch: Tensor, device: torch.device,
                                 dataloader_idx: int = 0) -> Tensor:
        return batch.to(device, non_blocking=True, memory_format=torch.channels_last)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path: str, map_location=None, strict: bool = True,
                             **overrides: Any) -> "VQAE":
        """Load a Lightning checkpoint written by the reference (``hyper_parameters`` holds the
        conf dicts saved by ``save_hyperparameters()``, model.py:25; ``state_dict`` the weights)."""
        ckpt = torch.load(checkpoint_path, map_location=map_location or "cpu",
                          weights_only=False)
        hparams = _plain(ckpt.get("hyper_parameters", {}))
        hparams.update(overrides)
        model = cls(**hparams)
        model.load_state_dict(ckpt["state_dict"], strict=strict)
        return model


def _plain(obj: Any) -> Any:
    """DictConfig/ListConfig (if omegaconf objects were pickled) -> plain containers."""
    if hasattr(obj, "items"):
        return {k: _plain(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)) or type(obj).__name__ == "ListConfig":
        return [_plain(v) for v in obj]
    return obj
