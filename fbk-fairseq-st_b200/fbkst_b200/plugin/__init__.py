"""fairseq ``--user-dir`` plugin: registers ``conv_transformer_b200`` and its four architectures.

    python train.py DATA --user-dir /path/to/fbk-fairseq-st_b200/fbkst_b200/plugin \\
        --arch conv_transformer_big2_b200 --task speech_translation_with_transcription \\
        --criterion ctc_multi_loss ... --no-attn-2d --distance-penalty log --ctc-compress-out

fairseq imports the user dir before parsing arguments (fairseq/options.py:119-122,
fairseq/utils.py:344-359).  The plugin first imports the reference's own
``examples.speech_recognition`` package (tasks, criterions, the reference model), then registers a
model whose ``build_model`` is the reference's (examples/speech_recognition/models/
conv_transformer.py:74-103) with the encoder swapped for the sm_100a one; decoder, task, criterion,
trainer and checkpoints are fairseq's.  Architectures reuse the reference's arch functions, so every
default (``:429-586``) is inherited.
"""
import os
import sys

import torch

_PKG_PARENT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _PKG_PARENT not in sys.path:
    sys.path.insert(0, _PKG_PARENT)

# compat.py is loaded by PATH: fairseq imports this directory as a top-level module (fairseq/utils.py:344-359),
# and importing it again as the package ``fbkst_b200.plugin`` would run the registrations twice
import importlib.util as _ilu  # noqa: E402
_spec = _ilu.spec_from_file_location("fbkst_b200_plugin_compat",
                                     os.path.join(os.path.dirname(os.path.abspath(__file__)), "compat.py"))
_compat = _ilu.module_from_spec(_spec)
_spec.loader.exec_module(_compat)
_compat.apply()  # (the numpy half is a no-op when the launcher already applied it)

from fairseq.models import FairseqEncoder, register_model, register_model_architecture  # noqa: E402
from fairseq.models.transformer import TransformerDecoder  # noqa: E402

import examples.speech_recognition  # noqa: E402,F401  (registers the reference task/criterion/model)
from examples.speech_recognition.models import conv_transformer as _ref  # noqa: E402

from fbkst_b200 import encoder as _enc  # noqa: E402
from fbkst_b200.cross_attention import swap_cross_attention  # noqa: E402

B200ConvolutionalTransformerEncoder = _enc.make_encoder_class(FairseqEncoder)
# hand fairseq's own NamedTuple types to downstream isinstance checks
_enc.EncoderOut = _ref.EncoderOut
_enc.CTCAwareEncoderOut = _ref.CTCAwareEncoderOut


@register_model("conv_transformer_b200")
class B200ConvolutionalTransformerModel(_ref.ConvolutionalTransformerModel):
    """Reference model class (args, state-dict upgrade hooks, freeze logic) with our encoder."""

    @classmethod
    def build_model(cls, args, task):
        _ref.base_architecture(args)
        if not hasattr(args, "max_source_positions"):
            args.max_source_positions = 100000
        if not hasattr(args, "max_target_positions"):
            args.max_target_positions = 100000
        src_dict, tgt_dict = task.source_dictionary, task.target_dictionary
        emb = _ref.Embedding(len(tgt_dict), args.decoder_embed_dim, tgt_dict.pad())
        if args.decoder_embed_path:
            from fairseq import utils
            utils.load_embedding(utils.parse_embedding(args.decoder_embed_path), tgt_dict, emb)
        encoder = B200ConvolutionalTransformerEncoder(
            args, src_dict if src_dict is not None else tgt_dict,
            audio_features=args.input_feat_per_channel)
        encoder.precision = getattr(args, "b200_precision", "bf16") or "bf16"
        decoder = TransformerDecoder(args, tgt_dict, emb)
        # SURVEY 8f N4: encoder-decoder attention on the device kernel (K/V once per utterance, beam
        # reorders move an index vector).  Same parameters / state_dict keys; inference only, so it
        # is opt-in: --b200-cross-attention (generate.py), never needed for train.py.
        if getattr(args, "b200_cross_attention", False):
            swap_cross_attention(decoder)
            encoder.lazy_beam_reorder = getattr(args, "b200_lazy_beam_reorder", False)
        return cls(encoder, decoder)

    @staticmethod
    def add_args(parser):
        _ref.ConvolutionalTransformerModel.add_args(parser)
        parser.add_argument("--b200-cross-attention", action="store_true",
                            help="run the decoder's encoder-decoder attention on the sm_100a kernel "
                                 "(inference: generate.py)")
        parser.add_argument("--b200-lazy-beam-reorder", action="store_true",
                            help="with --b200-cross-attention: never replicate the encoder output "
                                 "x beam (reorder_encoder_out returns tagged aliases)")
        parser.add_argument("--b200-precision", choices=["bf16", "fp32"], default="bf16",
                            help="encoder operand precision at inference: bf16 tensor-core operands (default) "
                                 "or fp32 on split-TF32 tensor cores (within 1e-3 of an fp32 reference; "
                                 "inference only)")


# ---------------------------------------------------------------------------------------------------
# SURVEY 8f N1: the CTC half of ``ctc_multi_loss`` on the device kernels.  Same class, flags, sample fields,
# logging keys and loss value as the reference criterion (criterions/ctc_multi_loss.py:107-194 +
# CTC_loss.py:101-175); what changes is where the arithmetic runs: the frame arg-max, log-sum-exp, alpha /
# beta recursions, the gradient w.r.t. the logits and the edit distance are CUDA kernels (fbkst_b200.criterion),
# the T x B x V log-softmax is never materialised and nothing is pulled to the host per utterance.
from fairseq import utils as _utils  # noqa: E402
from fairseq.criterions import register_criterion  # noqa: E402
from examples.speech_recognition.criterions import ctc_multi_loss as _cml  # noqa: E402
from fbkst_b200 import criterion as _crit  # noqa: E402


class B200CTCLoss(_cml.BaseCTCLoss):
    def forward(self, model, sample, reduce=True, log_probs=True):
        net_output = model(**sample["net_input"])  # FakeEncoderModel: the encoder's ctc_out + T x B padding mask
        logits = net_output["encoder_out"]
        if not torch.is_tensor(logits) or not logits.is_cuda:
            raise RuntimeError("ctc_multi_loss_b200: CUDA logits expected (there is no CPU fallback; use "
                               "--criterion ctc_multi_loss for the reference's CPU path)")
        if getattr(model, "output_batch_first", False):
            logits = logits.transpose(0, 1)
        targets, target_lengths = sample["target"], sample["target_lengths"]
        loss, totals, il = _crit.ctc_loss_train(logits, net_output["encoder_padding_mask"], targets,
                                                target_lengths, self.blank_idx)
        errors, total = (float(v) for v in totals.tolist())  # 16 bytes: the criterion's one host read
        if self.args.sentence_avg:
            sample_size = sample["target"].size(0)
        elif getattr(self.args, "use_source_side_sample_size", False):
            sample_size = int(il.sum().item())
        else:
            sample_size = sample["ntokens"]
        logging_output = {
            "loss": _utils.item(loss.data) if reduce else loss.data,
            "ntokens": sample["ntokens"],
            "nsentences": sample["target"].size(0),
            "sample_size": sample_size,
            "errors": errors,
            "total": total,
            "nframes": torch.sum(sample["net_input"]["src_lengths"]).item(),
        }
        return loss, sample_size, logging_output


@register_criterion("ctc_multi_loss_b200")
class B200CTCMultiLoss(_cml.CTCMultiLoss):
    """``--criterion ctc_multi_loss_b200``: the reference's CTCMultiLoss with its CTC term on the GPU kernels."""

    def __init__(self, args, task):
        super().__init__(args, task)
        self.ctc_criterion = B200CTCLoss(args, task)


for _name, _fn in (("conv_transformer_b200", _ref.base_architecture),
                   ("conv_transformer_big_b200", _ref.speechtransformer_big),
                   ("conv_transformer_big2_b200", _ref.speechtransformer_big2),
                   ("conv_transformer_giant_b200", _ref.speechtransformer_giant)):
    register_model_architecture("conv_transformer_b200", _name)(_fn)
