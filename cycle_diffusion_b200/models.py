"""The reference's model API kept verbatim in shape: what ``Trainer.prediction_step`` calls (trainer.py:786-789).

  TextUnsupervisedTranslation   ref model/text_unsupervised_translation.py:8-47
  UnsupervisedTranslation       ref model/unsupervised_translation.py:9-62
``args.gan`` is the parsed ``[gan]`` INI section (an iterable of (key, value) with a ``gan_type`` attribute, or a dict).
Extra keyword arguments (engine, state_dict, cond_stage, ...) are forwarded to the wrapper constructors.
"""
import torch
import torch.nn as nn

from .wrappers import get_gan_wrapper


def _gan_args(args):
    return args['gan'] if isinstance(args, dict) else args.gan


class TextUnsupervisedTranslation(nn.Module):

    def __init__(self, args, **wrapper_kwargs):
        super().__init__()
        self.gan_wrapper = get_gan_wrapper(_gan_args(args), **wrapper_kwargs)

    def forward(self, sample_id, original_image, encode_text, decode_text):
        self.gan_wrapper.eval()
        assert not self.training
        w = self.gan_wrapper
        if getattr(w, 'single_member', None) is not None and w.single_member():
            # one ensemble member: the reference's encode -> z -> generate (text_unsupervised_translation.py:33-36) as one lock-step loop
            img = w.cycle(original_image, encode_text, decode_text)
        else:
            z_ensemble = w.encode(image=original_image, encode_text=encode_text)
            img = w(z_ensemble=z_ensemble, original_img=original_image, encode_text=encode_text, decode_text=decode_text)
        losses = dict()
        weighted_loss = torch.zeros_like(sample_id).float()
        return (original_image, img), weighted_loss, losses

    @property
    def device(self):
        return self.gan_wrapper.device


class UnsupervisedTranslation(nn.Module):

    def __init__(self, args, source_kwargs=None, target_kwargs=None):
        super().__init__()
        self.source_gan_wrapper = get_gan_wrapper(_gan_args(args), **(source_kwargs or {}))
        self.target_gan_wrapper = get_gan_wrapper(_gan_args(args), target=True, **(target_kwargs or {}))
        assert self.source_gan_wrapper.resolution == self.target_gan_wrapper.resolution

    def forward(self, sample_id, class_label=None, original_image=None):
        self.source_gan_wrapper.eval()
        self.target_gan_wrapper.eval()
        assert not self.training
        if getattr(self.source_gan_wrapper, "enforce_class_input", False):
            assert getattr(self.target_gan_wrapper, "enforce_class_input", False)
            assert class_label is not None
            z = self.source_gan_wrapper.encode(image=original_image, class_label=class_label)
            img = self.target_gan_wrapper(z=z, class_label=class_label)
        else:
            assert class_label is None
            src, tgt = self.source_gan_wrapper, self.target_gan_wrapper
            if getattr(src, 'pair_cycle_applies', None) is not None and src.pair_cycle_applies(tgt):
                # matching schedules and shapes: the reference's encode -> z -> target (unsupervised_translation.py:48-49) as one
                # lock-step loop over both models, same result without the z tensor
                img = src.pair_cycle(tgt, original_image)
            else:
                z = src.encode(image=original_image)
                img = tgt(z=z)
        losses = dict()
        weighted_loss = torch.zeros_like(sample_id).float()
        return (original_image, img), weighted_loss, losses

    @property
    def device(self):
        return self.source_gan_wrapper.device


Model = TextUnsupervisedTranslation
