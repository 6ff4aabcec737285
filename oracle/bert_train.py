"""Oracle: one fastai training step of the remix encoder's mask task.  TEST INFRASTRUCTURE (plain PyTorch fp32, CPU).

Restates what ``Learner.fit`` does per batch around ``MultiTransformer`` (oracle/bert.py) for ``{'msk': {'x', 'pos'}}``:

    model.train(); logits = head(encoder(x_masked, pos))                  # deep_music_remix.py:1874-1881, 1910-2104
    loss = CrossEntropyFlat(ignore_index=pad_idx)(logits, y_masked)       # MultiLoss (:2734-2741) with the msk task only
    loss.backward(); clip_grad_norm_; p.mul_(1 - wd*lr); Adam(betas=(0.9, 0.99)).step()

``MTTrainer`` adds no AR/TAR terms (it only sets ``mask_steps``, which the encoder does not use).  The ``ignore_index=pad_idx``
reading follows from ``mask_tfm`` writing ``pad_idx`` into ``y`` at every position it did not select.  The optimizer is
oracle/train.py's ``AdamTrueWD`` (same known deviation on clipping).
Parity status: unpinned (the reference stores no training artefacts); this file is the definition the CUDA path is tested against.
"""
import torch
import torch.nn.functional as F

from .train import FixedMask, unique_params


def install_dropout_masks(model):
    """Swap every dropout the mask task runs through for a FixedMask; returns site -> list of modules:
    'embed' [1], 'attn' [L], 'res1' [L], 'out' [1]  (mask shapes [b,T,d], [b,H,T,T], [b,T,d], [b,1,d])."""
    enc, head = model.encoder, model.head
    sites = {'embed': [], 'attn': [], 'res1': [], 'out': []}
    enc.embed.drop = FixedMask(); sites['embed'].append(enc.embed.drop)
    for layer in enc.layers:
        layer.mha1.drop_att = FixedMask(); sites['attn'].append(layer.mha1.drop_att)
        layer.mha1.drop_res = FixedMask(); sites['res1'].append(layer.mha1.drop_res)
    head.output_dp = FixedMask(); sites['out'].append(head.output_dp)
    return sites


def masked_ce(logits, y, pad_idx):
    "CrossEntropyFlat(ignore_index=pad_idx): mean of -log softmax(logits)[y] over the positions whose target is not pad_idx (NaN if none)."
    lg = logits.reshape(-1, logits.size(-1)).float()
    t = y.reshape(-1)
    keep = t != pad_idx
    nll = torch.logsumexp(lg, -1) - lg.gather(1, t.clamp_min(0)[:, None])[:, 0]
    return (nll * keep).sum() / keep.sum()


def train_step(model, x, pos, y, opt, lr, pad_idx, wd=0.01, clip=0.5, betas=None):
    "One reference step of the mask task (model in train() mode with FixedMask dropouts or p=0); returns {'ce', 'grad_norm'}."
    for p in unique_params(model):
        p.grad = None
    logits = model({'msk': {'x': x, 'pos': pos}})['msk']
    ce = masked_ce(logits, y, pad_idx)
    ce.backward()
    gn = opt.step(lr, wd=wd, clip=clip, betas=betas)
    return {'ce': ce.item(), 'grad_norm': gn}
