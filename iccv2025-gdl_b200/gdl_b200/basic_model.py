"""Drop-in for reference models/basic_model.py: `AVClassifier_DGL(args)` with attributes
fusion_module / audio_net / visual_net / modality / args, the reference's construction order
(fusion head first, then audio_net, then visual_net: same init RNG stream), the same error
messages, and `forward(audio, visual) -> (out, a_out, v_out)` (reference :65-86; note the return
order differs from the fusion module's (a, v, out)).  Only modality == 'full' is built — the
unimodal ablation branches (reference :88-122) are out of scope of the hot path.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .backbone import resnet18
from .fusion_modules import ConcatFusion_DGL, FiLM_DGL, GatedFusion_DGL, SumFusion_DGL

N_CLASSES = {'VGGSound': 309, 'KineticSound': 34, 'kinect400': 400, 'CREMAD': 6, 'AVE': 28}


class AVClassifier_DGL(nn.Module):
    def __init__(self, args):
        super().__init__()
        fusion = args.fusion_method
        if args.dataset not in N_CLASSES:
            raise NotImplementedError('Incorrect dataset name {}'.format(args.dataset))
        n_classes = N_CLASSES[args.dataset]
        if fusion == 'sum':
            self.fusion_module = SumFusion_DGL(output_dim=n_classes)
        elif fusion == 'concat':
            self.fusion_module = ConcatFusion_DGL(output_dim=n_classes)
        elif fusion == 'film':
            self.fusion_module = FiLM_DGL(output_dim=n_classes, x_film=True)
        elif fusion == 'gated':
            self.fusion_module = GatedFusion_DGL(output_dim=n_classes, x_gate=True)
        else:
            raise NotImplementedError('Incorrect fusion method: {}!'.format(fusion))
        if getattr(args, 'modality', 'full') != 'full':
            raise NotImplementedError("gdl_b200 builds the DGL hot path only: modality must be 'full' "
                                      "(got {})".format(args.modality))
        self.audio_net = resnet18(modality='audio', args=args)
        self.visual_net = resnet18(modality='visual', args=args)
        self.modality = args.modality if hasattr(args, 'modality') else 'full'
        self.args = args
        self.n_classes = n_classes

    def forward(self, audio, visual):
        if not self.training:
            # eval mode: the EvalStep valid() runs (folded BatchNorm, fused pooling + head), so the logits of
            # model(...) and of valid() come from one arithmetic; no autograd graph is recorded
            from .step import eval_forward
            return eval_forward(self, audio, visual)
        a = self.audio_net(audio)    # [B,512,h,w]
        v = self.visual_net(visual)  # [B*T,512,7,7]
        (_, C, H, W) = v.size()
        B = a.size()[0]
        v = v.view(B, -1, C, H, W).permute(0, 2, 1, 3, 4)
        a = torch.flatten(F.adaptive_avg_pool2d(a, 1), 1)
        v = torch.flatten(F.adaptive_avg_pool3d(v, 1), 1)
        a_out, v_out, out = self.fusion_module(a, v)
        return out, a_out, v_out


AVClassifier = AVClassifier_DGL  # north_star naming alias
