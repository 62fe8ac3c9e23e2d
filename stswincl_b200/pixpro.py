"""``PixPro``-side wrapper of the contrastive pre-training model (pixcontrast_18/contrast/models/PixPro_swin_v5.py:138-561).

The reference's ``PixPro`` builds two copies of the whole segmentor (ResNet-18 OS8 -> Swin head -> ASPP, three 1x1
projections, a ``Proj_Head``) from a hard-coded checkpoint path, keeps one as the momentum ("key") encoder, and its
forward runs 2 query passes with gradients and, under ``no_grad``, the momentum update followed by 6 key passes.
ResNet / ASPP / projection heads are the caller's components (SURVEY.md section 8b: out of scope here); this module is
the part of that class that touches the two hot paths:

  * it takes the caller's built encoder pair (any ``nn.Module`` with the segmentor's attribute names) and replaces
    ``swin`` in both by ``stswincl_b200.swin.SwinTransformerLayerv5`` (``encoder_2`` / ``encoder_k_2``, :166,181),
    loading the reference weights strictly;
  * ``_momentum_update_key_encoder`` (:258-289) is one multi-tensor EMA launch per 48 tensors over ALL parameter
    pairs (``optim.momentum_update``), with the cosine momentum schedule of :262 kept on the device (a table of the
    per-iteration momenta and a device step counter), so a CUDA-graph-captured ``forward`` follows the schedule;
  * the 6 key passes run through the forward-only block path (no activations kept, no GELU-derivative output);
  * ``forward`` returns the reference's 8-tuple; with ``fuse_normalize=True`` the embeddings are returned
    un-normalised for ``contrast.consistency_loss_tail(normalize=True)``, which fuses ``F.normalize`` (:330,...).

``state_dict`` keys follow the reference (``encoder_1.*``, ``encoder_2.*``, ``encoder_3.*``, ``proj1-3.*``,
``projector.*``, the ``*_k_*`` twins and ``value_transform.*``, :146-151,236-243), so reference checkpoints load.
"""
from __future__ import annotations

import math
from typing import Callable, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import optim as soptim
from . import swin as sswin


def swap_swin_head(segmentor: nn.Module, attr: str = "swin") -> nn.Module:
    """``segmentor.swin = stswincl_b200.swin.SwinTransformerLayerv5(...)`` with the old head's weights (strict load)."""
    old = getattr(segmentor, attr)
    if isinstance(old, sswin.SwinTransformerLayerv5):
        return segmentor
    new = sswin.SwinTransformerLayerv5(dim=old.dim, input_resolution=tuple(old.input_resolution), num_heads=old.num_heads)
    new.load_state_dict(old.state_dict(), strict=True)
    p = next(old.parameters())
    setattr(segmentor, attr, new.to(p.device))
    return segmentor


def momentum_table(base_momentum: float, K: int) -> torch.Tensor:
    """fp32 [K + 1, 2]: row k < K is (m_k, 1 - m_k) with m_k = 1 - (1 - base) (cos(pi k / K) + 1) / 2 evaluated in
    double, as PixPro_swin_v5.py:262 does, and each entry rounded to fp32 once -- the values the eager expression
    ``k * m + q * (1. - m)`` multiplies by.  Row K is (1, 0), the expression's own value at k = K; every k >= K reads
    it, so past the end of the schedule the key encoder stays where it is (the expression would start a second cosine
    period there, which no recipe reaches: K is the recipe's iteration count)."""
    rows = []
    for k in range(K):
        m = 1. - (1. - base_momentum) * (math.cos(math.pi * k / K) + 1) / 2.
        rows.append((m, 1. - m))
    rows.append((1., 0.))
    return torch.tensor(rows, dtype=torch.float32)


class PixPro(nn.Module):
    """Drop-in for the reference ``PixPro`` around caller-built encoders.

    ``args`` carries the reference's options (``pixpro_momentum``, ``pixpro_transform_layer``, ``num_instances``,
    ``batch_size``, ``epochs``, ``start_epoch``; :143-150,230-231).  ``make_segmentor() -> nn.Module`` builds ONE
    segmentor with attributes ``resnet``, ``swin``, ``aspp``, ``project1..3`` (``TswinPlusv5`` in the reference, :164);
    ``make_projector() -> nn.Module`` builds the ``Proj_Head`` (:130).  Both are called twice (query / key copy)."""

    def __init__(self, args, make_segmentor: Optional[Callable[[], nn.Module]] = None,
                 make_projector: Optional[Callable[[], nn.Module]] = None, world_size: int = 1, fuse_normalize: bool = False):
        super().__init__()
        if make_segmentor is None or make_projector is None:
            raise ValueError("PixPro needs make_segmentor and make_projector: the ResNet / ASPP / projection heads are the "
                             "caller's components (see INTEGRATION.md)")
        self.pixpro_momentum = args.pixpro_momentum
        self.pixpro_transform_layer = getattr(args, "pixpro_transform_layer", 0)
        self.fuse_normalize = fuse_normalize
        q, k = swap_swin_head(make_segmentor()), swap_swin_head(make_segmentor())
        self.encoder_1, self.encoder_2, self.encoder_3 = q.resnet, q.swin, q.aspp
        self.proj1, self.proj2, self.proj3 = q.project1, q.project2, q.project3
        self.projector = make_projector()
        self.encoder_k_1, self.encoder_k_2, self.encoder_k_3 = k.resnet, k.swin, k.aspp
        self.proj_k_1, self.proj_k_2, self.proj_k_3 = k.project1, k.project2, k.project3
        self.projector_k = make_projector()
        for pq, pk in self._pairs():
            pk.data.copy_(pq.data)
            pk.requires_grad = False
        if self.pixpro_transform_layer == 0:
            self.value_transform = nn.Identity()
        elif self.pixpro_transform_layer == 1:
            self.value_transform = nn.Conv2d(256, 256, kernel_size=1, stride=1, padding=0, bias=True)
        else:
            raise NotImplementedError("pixpro_transform_layer 2 (MLP2d) is the caller's module: assign value_transform")
        # momentum schedule length and position (:230-231)
        self.K = int(args.num_instances * 1. / world_size / args.batch_size * args.epochs)
        if self.K < 1:
            raise ValueError(f"PixPro: the momentum schedule needs at least one iteration, got K = {self.K}")
        # the schedule on the device (momentum_table) and its position; the counter advances inside the update.  Not
        # part of state_dict (the reference's keys only); .to() / .cuda() move them with the module.
        p = next(self.parameters())
        self.register_buffer("_m_table", momentum_table(self.pixpro_momentum, self.K).to(p.device), persistent=False)
        self.register_buffer("_k_t", torch.zeros(1, dtype=torch.int64, device=p.device), persistent=False)
        self.k = int(args.num_instances * 1. / world_size / args.batch_size * (args.start_epoch - 1))

    @property
    def k(self) -> int:
        """The schedule position (:231): iterations taken so far.  Reading it synchronises with the device."""
        return int(self._k_t.item())

    @k.setter
    def k(self, value: int) -> None:
        if value < 0:
            raise ValueError(f"PixPro.k must be >= 0, got {value}")
        self._k_t.fill_(int(value))

    def _pairs(self):
        mods = [(self.encoder_1, self.encoder_k_1), (self.encoder_2, self.encoder_k_2), (self.encoder_3, self.encoder_k_3),
                (self.proj1, self.proj_k_1), (self.proj2, self.proj_k_2), (self.proj3, self.proj_k_3),
                (self.projector, self.projector_k)]
        for mq, mk in mods:
            yield from zip(mq.parameters(), mk.parameters())

    @torch.no_grad()
    def _momentum_update_key_encoder(self):
        """:258-289 -- cosine schedule, then every parameter pair in multi-tensor launches.  The momentum pair is read
        from the device table at the device counter, which then advances: no host read, so the update can be
        captured in a CUDA graph and each replay takes the next step of the schedule."""
        m = self._m_table.index_select(0, self._k_t.clamp(max=self.K)).view(2)
        self._k_t.add_(1)
        pairs = list(self._pairs())
        soptim.momentum_update([p for p, _ in pairs], [p for _, p in pairs], m)

    def _embed(self, seq, key: bool):
        enc1, enc2, enc3 = (self.encoder_k_1, self.encoder_k_2, self.encoder_k_3) if key else (self.encoder_1, self.encoder_2, self.encoder_3)
        p1, p2, p3 = (self.proj_k_1, self.proj_k_2, self.proj_k_3) if key else (self.proj1, self.proj2, self.proj3)
        projector = self.projector_k if key else self.projector
        feats = torch.cat([enc1(seq[:, i]).unsqueeze(1) for i in range(seq.shape[1])], dim=1)      # :303-308
        res_output = feats[:, -1]
        tem1, tem2 = enc2(feats)                                                                      # the Swin head (:311)
        t1, t2 = tem1[:, -1], tem2[:, -1]
        aspp = enc3(t2)
        r, a, b = p1(res_output), p2(t1), p3(t2)
        b = F.interpolate(b, size=r.shape[2:], mode="bilinear", align_corners=False)
        aspp = F.interpolate(aspp, size=r.shape[2:], mode="bilinear", align_corners=False)
        proj = projector(torch.cat([r, a, b, aspp], dim=1))                                           # :326-328
        return proj if self.fuse_normalize else F.normalize(proj, dim=1)                              # :330

    def forward(self, seq_1, seq_2, seq_3, seq_4, seq_5, seq_6):
        pred_1 = self._embed(seq_1, key=False)
        pred_2 = self._embed(seq_2, key=False)
        with torch.no_grad():                                   # no gradient to keys (:366)
            self._momentum_update_key_encoder()
            keys = [self._embed(s, key=True) for s in (seq_1, seq_2, seq_3, seq_4, seq_5, seq_6)]
        return (pred_1, pred_2, *keys)
