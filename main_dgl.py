#!/usr/bin/env python
"""CLI-compatible entry point for the reference's main_dgl.py (same flags, same defaults,
same prints / csv / checkpoint file names, same evaluation-mode checkpoint loading), running the B200-native DGL step.
Deviations: no TensorBoard branch; `--resume`, `--synthetic_len`, `--dp_replicas`, `--per_class` and `--ap` are
additions.

    python main_dgl.py --train --ckpt_path ckpt --dataset CREMAD --fusion_method concat \
        --fps 3 --alpha 4 --batch_size 64 --audio_path synthetic

Multi-GPU: launch with torchrun (one process per GPU); the reference's nn.DataParallel
(main_dgl.py:244) becomes per-process replicas + NCCL gradient all-reduce.  Real datasets need
the reference's dataset classes (librosa, image folders); `--audio_path synthetic` selects the
synthetic loader of gdl_b200/synthetic.py.
"""
import argparse
import csv
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.optim as optim  # noqa: E402
from torch.utils.data import DataLoader  # noqa: E402

from gdl_b200 import AVClassifier_DGL, setup_seed, weight_init  # noqa: E402
from gdl_b200.parallel import replicas_per_rank  # noqa: E402
from gdl_b200.synthetic import SyntheticAV  # noqa: E402
from gdl_b200.train import train_epoch, valid, valid_report  # noqa: E402


def get_arguments(argv=None):
    """Argument surface of reference main_dgl.py:24-65 (byte-compatible names and defaults)."""
    parser = argparse.ArgumentParser()
    parser.add_argument('--dataset', default='CREMAD', type=str, help='VGGSound, KineticSound, CREMAD, AVE')
    parser.add_argument('--modulation', default='OGM_GE', type=str, choices=['Normal', 'OGM', 'OGM_GE'])
    parser.add_argument('--fusion_method', default='concat', type=str, choices=['sum', 'concat', 'gated', 'film'])
    parser.add_argument('--fps', default=1, type=int)
    parser.add_argument('--use_video_frames', default=3, type=int)
    parser.add_argument('--num_frame', default=1, type=int, help='use how many frames for train')
    parser.add_argument('--audio_path', default='./train_test_data/CREMA-D/AudioWAV', type=str)
    parser.add_argument('--visual_path', default='./train_test_data/CREMA-D', type=str)
    parser.add_argument('--batch_size', default=64, type=int)
    parser.add_argument('--epochs', default=100, type=int)
    parser.add_argument('--optimizer', default='sgd', type=str)
    parser.add_argument('--learning_rate', default=0.001, type=float, help='initial learning rate')
    parser.add_argument('--lr_decay_step', default='[70]', type=str, help='where learning rate decays')
    parser.add_argument('--lr_decay_ratio', default=0.1, type=float, help='decay coefficient')
    parser.add_argument('--modulation_starts', default=0, type=int, help='where modulation begins')
    parser.add_argument('--modulation_ends', default=50, type=int, help='where modulation ends')
    parser.add_argument('--alpha', default=4.0, type=float, help='alpha in DGL')
    parser.add_argument('--ckpt_path', required=True, type=str, help='path to save trained models')
    parser.add_argument('--train', action='store_true', help='turn on train mode')
    parser.add_argument('--use_tensorboard', default=False, type=bool, help='whether to visualize')
    parser.add_argument('--tensorboard_path', type=str, help='path to save tensorboard logs')
    parser.add_argument('--random_seed', default=0, type=int)
    parser.add_argument('--gpu_ids', default='1', type=str, help='GPU ids')
    parser.add_argument('--modality', type=str, default='full')
    parser.add_argument('--backbone', type=str, default='resnet')
    parser.add_argument('--total_epoch', default=10, type=int)
    parser.add_argument('--drop', default=0, type=int)
    # additions (defaults preserve the reference behaviour)
    parser.add_argument('--synthetic_len', default=0, type=int, help='synthetic dataset length (0 = CREMA-D sizes)')
    parser.add_argument('--resume', default=None, type=str,
                        help='checkpoint written by this script or by the reference (main_dgl.py:396-412) to continue from')
    parser.add_argument('--dp_replicas', default=0, type=int,
                        help='data-parallel replicas R (0 = one per process): batch_size / R rows per BatchNorm batch, '
                             'R / processes of them run one after another on each GPU, like nn.DataParallel over R GPUs')
    parser.add_argument('--per_class', action='store_true',
                        help='evaluate with per-class accuracies of the fused, audio and visual heads: appended to '
                             '<ckpt_path>/<dataset>_<modality>_per_class.csv when training, printed in evaluation mode')
    parser.add_argument('--ap', action='store_true',
                        help='evaluate with per-class average precision, mAP and top-5 accuracy of the fused, audio and '
                             'visual heads: appended to <ckpt_path>/<dataset>_<modality>_ap.csv and printed as an mAP '
                             'line when training, printed with the per-class table in evaluation mode')
    return parser.parse_args(argv)


PER_CLASS_HEADER = ['epoch', 'head', 'class', 'support', 'correct', 'accuracy']
AP_HEADER = ['epoch', 'head', 'class', 'support', 'ap']


def _append_csv(path, header, rows):
    new = not os.path.exists(path)
    with open(path, 'a+', newline='') as f:
        w = csv.writer(f)
        if new:
            w.writerow(header)
        w.writerows(rows)


def ap_line(report):
    """The --ap summary line of an EvalReport of valid_report(ap=True)."""
    return 'mAP: {:.4f}, Audio mAP: {:.4f}, Visual mAP: {:.4f}, Top-{} Acc: {:.4f}'.format(
        report.map, report.map_a, report.map_v, report.k, report.top5)


def evaluate_epoch(args, model, device, loader, epoch, rank=0, reports=None):
    """The evaluation pass of a training epoch: valid() (acc, acc_a, acc_v), or with --per_class / --ap
    valid_report(), whose accuracies are the same; rank 0 then appends the epoch's per-class rows to
    <ckpt_path>/<dataset>_<modality>_per_class.csv (--per_class) and its AP rows to
    <ckpt_path>/<dataset>_<modality>_ap.csv (--ap), a header first when a file is new.  The report is appended to
    `reports` when given."""
    use_ap = getattr(args, 'ap', False)
    if not args.per_class and not use_ap:
        return valid(args, model, device, loader)
    report = valid_report(args, model, device, loader, ap=True) if use_ap else valid_report(args, model, device, loader)
    if rank == 0:
        stem = os.path.join(args.ckpt_path, args.dataset + '_' + args.modality)
        if args.per_class:
            _append_csv(stem + '_per_class.csv', PER_CLASS_HEADER, report.rows(epoch))
        if use_ap:
            _append_csv(stem + '_ap.csv', AP_HEADER, report.ap_rows(epoch))
    if reports is not None:
        reports.append(report)
    return report.acc, report.acc_a, report.acc_v


def main(argv=None):
    args = get_arguments(argv)
    args.p = [0, 0]
    print(args)
    setup_seed(args.random_seed)
    if args.backbone != 'resnet':
        raise EOFError  # reference main_dgl.py:236-240
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dp_replicas and args.train:
        replicas_per_rank(args.batch_size, args.dp_replicas, world)  # ValueError before any device or data work
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=device)
    rank = int(os.environ.get("RANK", "0"))
    model = AVClassifier_DGL(args)
    model.apply(weight_init)
    model.to(device)

    class _Module(nn.Module):  # keeps the reference's `module.` prefix (DataParallel names)
        def __init__(self, m):
            super().__init__()
            self.module = m

        def forward(self, *a):
            return self.module(*a)
    model = _Module(model)

    if args.optimizer == 'sgd':
        optimizer = optim.SGD(model.parameters(), lr=args.learning_rate, momentum=0.9, weight_decay=1e-4)
    elif args.optimizer == 'AdaGrad':  # reference main_dgl.py:251-256 (OGM-GE lineage arguments)
        optimizer = optim.Adagrad(model.parameters(), lr=args.learning_rate)
    elif args.optimizer == 'Adam':
        optimizer = optim.Adam(model.parameters(), lr=args.learning_rate, betas=(0.9, 0.999), eps=1e-08)
    else:
        raise ValueError('Incorrect optimizer: {}'.format(args.optimizer))  # reference main_dgl.py:259
    scheduler = optim.lr_scheduler.MultiStepLR(optimizer, eval(args.lr_decay_step), args.lr_decay_ratio)

    if args.audio_path not in ('synthetic', 'synthetic_exact', 'synthetic_device'):
        raise NotImplementedError("this environment ships no datasets: pass --audio_path synthetic (random tensors) "
                                  "or synthetic_exact (the reference's per-item random-draw order on seeded images), "
                                  "or plug the reference's dataset classes (same (spec, images, label) contract) in")
    n = args.synthetic_len or None
    if args.audio_path == 'synthetic_device':
        # the reference's draw order with the pixels left on the GPU: items carry crop boxes, the frames are
        # produced by gdl_crop_resize_normalize from a device-resident uint8 store (CREMA-D contract only)
        from gdl_b200.synthetic import SyntheticCramedDevice
        if args.dataset != 'CREMAD':
            raise NotImplementedError('synthetic_device implements the CREMA-D sample contract only')
        train_dataset = SyntheticCramedDevice(args, 'train', n or 512)
        test_dataset = SyntheticCramedDevice(args, 'test', (n and max(n // 8, args.batch_size)) or 64)
        train_dataset.attach_pipeline(device)
        test_dataset.attach_pipeline(device)
    elif args.audio_path == 'synthetic_exact':
        from gdl_b200.synthetic import SyntheticCramed, SyntheticKS
        cls = SyntheticCramed if args.dataset == 'CREMAD' else SyntheticKS
        train_dataset = cls(args, 'train', n or 6698)
        test_dataset = cls(args, 'test', (n and max(n // 8, args.batch_size)) or 744)
    else:
        train_dataset = SyntheticAV(args, 'train', n)
        test_dataset = SyntheticAV(args, 'test', n and max(n // 8, args.batch_size))
    per_rank = args.batch_size // world
    shard_sampler = None
    if world > 1:
        # the reference's DataLoader(shuffle=True) order, cut into global batches that are split contiguously in
        # DataParallel chunk order (main_dgl.py:244): rank r's BatchNorm sees the rows reference device r would
        from gdl_b200.parallel import ChunkShardBatchSampler
        shard_sampler = ChunkShardBatchSampler(torch.utils.data.RandomSampler(train_dataset), args.batch_size, rank, world)
        train_loader = DataLoader(train_dataset, batch_sampler=shard_sampler, num_workers=8, pin_memory=True)
    else:
        train_loader = DataLoader(train_dataset, batch_size=per_rank, shuffle=True, num_workers=8, pin_memory=True,
                                  drop_last=True)
    if world > 1:
        # the reference's test loader (batch_size = G, drop_last) whose batches DataParallel splits over the GPUs:
        # rank r evaluates contiguous chunk r of every global batch and valid() sums the counts over the ranks
        from gdl_b200.parallel import ChunkShardBatchSampler
        test_loader = DataLoader(test_dataset, batch_sampler=ChunkShardBatchSampler(
            torch.utils.data.SequentialSampler(test_dataset), args.batch_size, rank, world), num_workers=8,
            pin_memory=True)
    else:
        test_loader = DataLoader(test_dataset, batch_size=per_rank, shuffle=False, num_workers=8, pin_memory=True,
                                 drop_last=True)  # the reference drops the test tail too (main_dgl.py:287-288)

    start_epoch, best_acc = 0, 0.0
    if args.resume and args.train:
        # the reference saves {'saved_epoch', 'model' (module.-prefixed keys), 'optimizer', 'scheduler', ...} but has
        # no way to load it back; the optimizer state (momentum, Adam moments, Adagrad sums, step count) is adopted by
        # the fused update on the first batch
        ckpt = torch.load(args.resume, map_location=device)
        model.load_state_dict(ckpt['model'])
        optimizer.load_state_dict(ckpt['optimizer'])
        scheduler.load_state_dict(ckpt['scheduler'])
        start_epoch = int(ckpt['saved_epoch']) + 1
        best_acc = float(ckpt.get('acc', 0.0))  # a resumed run only overwrites "best" with something better
        print('Resumed from {} (epoch {}, acc {})'.format(args.resume, ckpt['saved_epoch'], ckpt.get('acc')))

    if args.train:
        os.makedirs(args.ckpt_path, exist_ok=True)
        log = os.path.join(args.ckpt_path, args.dataset + '_' + args.modality + '.csv')
        if rank == 0:
            with open(log, 'a+', newline='') as f:
                csv.writer(f).writerow([1000, 1000, 1000])  # run separator, main_dgl.py:292-295
        for epoch in range(start_epoch, args.epochs):
            print('Epoch: {}: '.format(epoch))
            args.epoch_now = epoch
            batch_loss, batch_loss_a, batch_loss_v, a_div, v_div, a_re, v_re = train_epoch(
                args, epoch, model, device, train_loader, optimizer, scheduler)
            if shard_sampler is not None:
                from gdl_b200.parallel import assert_same_order
                assert_same_order(shard_sampler.order_digest)
            reports = []
            acc, acc_a, acc_v = evaluate_epoch(args, model, device, test_loader, epoch, rank, reports)
            if rank == 0:
                with open(log, 'a+', newline='') as f:
                    csv.writer(f).writerow([acc, acc_a, acc_v])
            if acc > best_acc and epoch:
                best_acc = float(acc)
                # the reference's exact file name (main_dgl.py:358-367: no fusion field, no '_' before 'optimizer')
                name = 'best_model_of_dataset_{}_{}_alpha_{}' \
                       'optimizer_{}_modulate_starts_{}_ends_{}_' \
                       'epoch_{}_acc_{}.pth'.format(args.dataset, args.modulation, args.alpha, args.optimizer,
                                                    args.modulation_starts, args.modulation_ends, epoch, acc)
                if rank == 0:
                    torch.save({'saved_epoch': epoch, 'modulation': args.modulation, 'alpha': args.alpha,
                                'fusion': args.fusion_method, 'acc': acc, 'model': model.state_dict(),
                                'optimizer': optimizer.state_dict(), 'scheduler': scheduler.state_dict()},
                               os.path.join(args.ckpt_path, name))
                print('The best model has been saved at {}.'.format(os.path.join(args.ckpt_path, name)))
                print("Loss: {:.3f}, Acc: {:.3f}".format(batch_loss, acc))
            else:
                print("Loss: {:.3f}, Acc: {:.3f}, Best Acc: {:.3f}".format(batch_loss, acc, best_acc))
            print("Audio Acc: {:.3f}， Visual Acc: {:.3f} ".format(acc_a, acc_v))
            if args.ap:
                print(ap_line(reports[0]))
            print("Audio similar: {:.3f}， Visual similar: {:.3f} ".format(a_div, v_div))
            print("Audio regurize: {:.3f}， Visual regurize: {:.3f} ".format(a_re, v_re))
    else:
        # reference main_dgl.py:396-418: args.ckpt_path IS the checkpoint file in evaluation mode
        path = args.resume or args.ckpt_path
        if not os.path.isfile(path):
            raise FileNotFoundError("evaluation mode loads a trained model: --ckpt_path (or --resume) must name a "
                                    "checkpoint file written by --train, got {!r}".format(path))
        loaded_dict = torch.load(path, map_location=device)
        assert loaded_dict['modulation'] == args.modulation, \
            'inconsistency between modulation method of loaded model and args !'
        assert loaded_dict['fusion'] == args.fusion_method, \
            'inconsistency between fusion method of loaded model and args !'
        model.load_state_dict(loaded_dict['model'])
        print('Trained model loaded!')
        if args.ap:
            report = valid_report(args, model, device, test_loader, ap=True)
            acc, acc_a, acc_v = report.acc, report.acc_a, report.acc_v
        elif args.per_class:
            report = valid_report(args, model, device, test_loader)
            acc, acc_a, acc_v = report.acc, report.acc_a, report.acc_v
        else:
            acc, acc_a, acc_v = valid(args, model, device, test_loader)
        print('Accuracy: {}, accuracy_a: {}, accuracy_v: {}'.format(acc, acc_a, acc_v))
        if args.ap:
            print(ap_line(report))
        if args.per_class:
            print('Per-class accuracy ({} samples):'.format(report.total))
            print(report.table())
        if args.ap:
            print('Per-class average precision ({} samples):'.format(report.total))
            print(report.ap_table())


if __name__ == "__main__":
    main()
