"""
Command-line entry points -- mirror of PyLC's pylc.py / utils/argparse.py / preprocess.py / test.py /
train.py (reference pylc.py:19-40, utils/argparse.py:22-337, preprocess.py:21-91, test.py:23-115,
train.py:22-174), same sub-commands and flags for the tiled-segmentation path:

    python -m pylc_b200.pylc extract --ch 3 --img DIR --mask DIR [--schema S] [--output DIR]
    python -m pylc_b200.pylc profile --db FILE            (documented by the reference README but
                                                          not wired there: preprocess.py:77-91 recurses)
    python -m pylc_b200.pylc augment --db FILE            (sample-rate search + over-sampling of rare classes)
    python -m pylc_b200.pylc train   --db FILE [--batch_size N --n_epochs E --lr LR --weighted ...]
    python -m pylc_b200.pylc test    --model M --img I [--mask G] [--scale S] [--save_logits]
                                     [--aggregate_metrics] [--stitch reference|mean] [--save_confidence]
                                     [--multiscale S1 S2 ...]   (with --stitch mean) [--temperature T]
    python -m pylc_b200.pylc calibrate -l M -i I -m G [--scale S] [--batch_tiles N] [-o OUT] [--max_resident_gb G]
                                     (fits the mean stitch's softmax temperature; writes a calibrated model copy)

Launched under torchrun (WORLD_SIZE > 1), `extract`/`profile`/`test` shard images or tiles across
the GPUs and all-reduce only histograms / confusion matrices (pylc_b200.dist).  `merge` and `grayscale`
are stubs in the reference itself (preprocess.py:94-122: commented-out body / bare return) and are not provided.
"""
import argparse
import json
import math
import os
import sys

import cv2
import torch

from . import dist as pdist
from .config import Parameters, defaults


def _mkdirs():
    for d in (defaults.root, defaults.db_dir, defaults.save_dir, defaults.model_dir, defaults.output_dir):
        os.makedirs(d, exist_ok=True)


# ---- handlers ---------------------------------------------------------------------------------

def extract(args):
    """Tile extraction + profiling -> tile database (reference preprocess.py:21-51)."""
    from .utils.extract import Extractor
    from .utils import tools
    params = Parameters(args)
    rank, world, _ = pdist.init_from_env()
    extractor = Extractor(params)
    extractor.verbose = rank == 0
    extractor.load(args.img, args.mask)
    if world > 1:                                   # images are independent: shard them by index
        mine = pdist.shard_indices(len(extractor.files))
        extractor.files = [extractor.files[i] for i in mine]
        extractor.n_files = len(extractor.files)
    extractor.extract().coshuffle().profile(distributed=world > 1)
    dset = extractor.get_data()
    meta = dset.get_meta()
    if world > 1:
        meta.id = meta.id + '_rank%d' % rank        # one shard file per rank; metadata is global
    if getattr(args, 'output', None):
        meta.output_dir = tools.mk_path(args.output)
    path = dset.save()
    print('Extraction done: {} tiles -> {}'.format(dset.size, path))
    return path


def profile(args):
    """Profile an existing tile database (what reference preprocess.py:77-91 intends)."""
    from .db.dataset import MLPDataset
    from .utils.profile import get_profile, print_meta
    dset = MLPDataset(args.db)
    meta = get_profile(dset)
    print_meta(meta)
    return meta


def augment(args):
    """Over-sample the rare classes of a tile database (reference preprocess.py:54-74): sample-rate search on
    the device (pylc_sample_rate_grid), the reference's OpenCV warps on the host, profile of the result on the
    device, `_aug<id>` database written next to the others."""
    from .utils.augment import Augmentor
    from .utils.profile import print_meta
    print('\nStarting augmentation on database:\n\t{}'.format(args.db))
    augmentor = Augmentor().load(args.db)
    print_meta(augmentor.input_meta)
    augmentor.optimize()
    augmentor.oversample(device=True if getattr(args, 'device_warps', False) else None)
    aug_dset = augmentor.print_settings().get_data()
    print_meta(augmentor.output_meta)
    path = aug_dset.save()
    print('Augmentation done: {} tiles -> {}'.format(aug_dset.size, path))
    return path


def train(args):
    """Training loop (reference train.py:22-174): validate at epoch 0, then train + validate."""
    from .db.dataset import MLPDataset
    from .models.model import Model
    if getattr(args, 'weighted', None) is not None:      # the reference tests the option's truthiness
        args.weighted = bool(args.weighted)
    params = Parameters(args)
    rank, world, local = pdist.init_from_env()
    tr_dset = MLPDataset(db_path=args.db, partition=(0, 1 - defaults.partition))
    va_dset = MLPDataset(db_path=args.db, partition=(1 - defaults.partition, 1.))
    if rank == 0:
        tr_dset.print_meta(defaults.TRAIN)
        va_dset.print_meta(defaults.VALID)
    tr_loader, tr_batches = tr_dset.loader(batch_size=params.batch_size, n_workers=params.n_workers, drop_last=True)
    va_loader, va_batches = va_dset.loader(batch_size=params.batch_size, n_workers=params.n_workers, drop_last=True)
    model = Model().update_meta(tr_dset.get_meta())
    model.update_meta({k: getattr(args, k) for k in ('arch', 'backbone', 'weighted', 'ce_weight', 'dice_weight',
                                                     'focal_weight', 'lr', 'batch_size', 'n_epochs', 'report')
                       if getattr(args, k, None) is not None})
    model.meta.optim_type = getattr(args, 'optim', None) or model.meta.optim_type
    model.meta.sched_type = getattr(args, 'sched', None) or model.meta.sched_type
    pretrained = getattr(args, 'pretrained', None)
    model.meta.pretrained = (defaults.pretrained if pretrained is True else pretrained) or False
    model.resume_checkpoint = bool(getattr(args, 'resume', False))
    model.distributed = world > 1
    model.is_writer = rank == 0                      # one rank writes checkpoints / loss logs
    model.build()
    model.resume()
    if world > 1:                                    # stock DDP for the network gradients
        model.net = torch.nn.parallel.DistributedDataParallel(model.net, device_ids=[local] if torch.cuda.is_available() else None)
    model.net.train()
    if rank == 0:
        model.print_settings()
    for epoch in range(model.epoch, params.n_epochs - model.epoch):
        model.loss.lr += [(model.iter, model.get_lr())]
        if rank == 0:
            print('\nEpoch {} / {}   lr {}'.format(epoch + 1, params.n_epochs, model.get_lr()))
        if epoch == 0:
            _validate(model, va_loader, va_batches, rank, world)
        model.net.train()
        for i, (x, y) in enumerate(tr_loader):
            if i >= rank_steps(tr_batches, world) * world:
                break
            if i % world == rank:                    # batches round-robin across ranks
                model.train(x, y)
        _validate(model, va_loader, va_batches, rank, world)
        if model.sched is not None:
            model.sched.step()
        model.epoch += 1
    return model


def rank_steps(n_batches, world):
    """Steps every rank takes over `n_batches` batches dealt round-robin.  Each step issues collectives
    (DDP's gradient all-reduce, the loss-partials all-reduce of MultiLoss(distributed=True)), so all
    ranks must take the SAME number: the trailing n_batches mod world batches are dropped (the loaders
    already drop the trailing partial batch, drop_last=True)."""
    return n_batches // world


def _validate(model, loader, n_batches, rank, world):
    model.net.eval()
    for i, (x, y) in enumerate(loader):
        if i >= rank_steps(n_batches, world) * world:
            break
        if i % world == rank:
            model.eval(x, y)
    model.log()
    if rank == 0:
        model.save()
    model.net.train()


def test(args):
    """Tiled inference (+ evaluation when masks are given) (reference test.py:23-115)."""
    from .models.model import Model
    from .pipeline import TiledSegmenter
    from .utils import tools
    from .utils.evaluate import Evaluator
    from .utils.extract import Extractor
    from .pipeline import check_scales
    multiscale = getattr(args, 'multiscale', None)
    stitch = getattr(args, 'stitch', 'reference')
    temperature = getattr(args, 'temperature', None)
    if temperature is not None and not (math.isfinite(temperature) and temperature > 0):
        print('--temperature must be finite and > 0, got %r.' % temperature, file=sys.stderr)
        sys.exit(2)
    if temperature is not None and stitch != 'mean':
        print("--temperature scales the mean stitch's probabilities: add --stitch mean.", file=sys.stderr)
        sys.exit(2)
    if multiscale and stitch != 'mean':
        print('--multiscale averages the probabilities of the mean stitch: add --stitch mean.', file=sys.stderr)
        sys.exit(2)
    try:
        multiscale = check_scales(multiscale) if multiscale else None
    except ValueError as exc:
        print('--multiscale: %s' % exc, file=sys.stderr)
        sys.exit(2)
    params = Parameters(args)
    rank, world, _ = pdist.init_from_env()
    model = Model().load(args.model)
    if rank == 0:
        model.print_settings()
    model.net.eval()
    stored = (model.calibration or {}).get('temperature')
    if temperature is None:              # a calibrated model file applies its temperature to the mean stitch
        temperature = float(stored) if stored is not None and stitch == 'mean' else 1.0
        if stored is not None and stitch != 'mean' and rank == 0:
            print('The model is calibrated (temperature %g); the temperature is not applied with --stitch reference.'
                  % stored)
    files = tools.collate(args.img, args.mask)
    mine = pdist.shard_indices(len(files))
    extractor = Extractor(model.meta)
    extractor.verbose = False
    evaluator = Evaluator(model.meta)
    evaluator.aggregate_inject = 0 in mine           # the concatenated vectors carry ONE injection
    save_confidence = bool(getattr(args, 'save_confidence', False))
    seg = TiledSegmenter(model, batch_tiles=getattr(args, 'batch_tiles', 32), keep_masks=True,
                         stitch=stitch, confidence=save_confidence, scales=multiscale, temperature=temperature)

    def save_metrics():
        if seg.scales is not None:                    # a multi-scale run records its scales with the scores
            evaluator.metrics.results['multiscale'] = list(seg.scales)
        if seg.temperature != 1.0:
            evaluator.metrics.results['temperature'] = seg.temperature
        evaluator.save_metrics()

    def decode(i):
        fpair = files[i]
        img_file, mask_file = (fpair['img'], fpair['mask']) if isinstance(fpair, dict) else (fpair, None)
        gt = None
        if mask_file:                                 # what Evaluator.load decodes (reference evaluate.py:87-91)
            gt = tools.get_image(mask_file, ch=3, scale=params.scale, interpolate=cv2.INTER_NEAREST)[0]
        return (i, img_file, mask_file, gt) + tuple(tools.get_image(img_file, model.meta.ch, scale=params.scale))

    # the next files (image + ground truth) decode on host threads while the current image is on the GPU
    for i, img_file, mask_file, gt, img, w_full, h_full, w_scaled, h_scaled in \
            tools.ordered_prefetch(decode, mine, depth=3):
        f = seg.stage(img, None, index=i)
        torch.cuda.current_stream().wait_event(f.ready)
        res = seg.segment_fitted(f, inject=0)         # stitch + argmax + colourise + resample on the GPU
        meta = extractor.meta
        meta.stride = seg.S
        meta.extract = {'fid': os.path.basename(img_file.replace('.', '_')) + '_scale_' + str(params.scale),
                        'n': (f.h // seg.S - 1) * (f.w // seg.S - 1), 'w_full': w_full, 'h_full': h_full,
                        'w_scaled': w_scaled, 'h_scaled': h_scaled, 'w_fitted': f.w, 'h_fitted': f.h, 'offset': 0}
        evaluator.load(res, meta, mask_true_path=mask_file, scale=params.scale, mask_true=gt).save_image()
        if save_confidence:
            evaluator.save_confidence()
        if mask_file and not params.aggregate_metrics:
            print("\nStarting evaluation ... ")
            evaluator.evaluate()
            save_metrics()
        if getattr(args, 'save_logits', False):
            print('--save_logits: logits stay on the device in this implementation; saving the label map instead.')
            evaluator.save_logits([res["labels"].cpu()])
        evaluator.reset()
    if getattr(args, 'aggregate_metrics', False):
        evaluator.evaluate(aggregate=True, distributed=world > 1)
        if rank == 0:
            save_metrics()
    return evaluator


def calibrate(args):
    """Fit the softmax temperature of the mean stitch on labelled images (utils/calibrate.py) and write a copy of the
    model file with a "calibration" entry, plus <output>/<id>/metrics/calibration_fit.json."""
    from .models.model import Model
    from .pipeline import TiledSegmenter
    from .utils import tools
    from .utils.calibrate import ResidentBudgetError, TemperatureFit, write_calibrated_copy
    if int(os.environ.get('WORLD_SIZE', '1')) > 1:
        print('pylc calibrate runs on one GPU: launch it without torchrun.', file=sys.stderr)
        sys.exit(2)
    stem, _ = os.path.splitext(args.model)
    out_file = args.output or stem + '_calibrated.pth'
    if os.path.abspath(out_file) == os.path.abspath(args.model):
        print('pylc calibrate writes a copy: the output %s is the input model.' % out_file, file=sys.stderr)
        sys.exit(2)
    params = Parameters(args)
    model = Model().load(args.model)
    model.net.eval()
    free = torch.cuda.mem_get_info()[0]
    budget = args.max_resident_gb * 1e9 if args.max_resident_gb is not None else free / 2
    seg = TiledSegmenter(model, batch_tiles=args.batch_tiles, stitch='mean')
    fit = TemperatureFit(seg, budget)
    files = tools.collate(args.img, args.mask)
    for fpair in files:
        img_file, mask_file = (fpair['img'], fpair['mask']) if isinstance(fpair, dict) else (fpair, None)
        if not mask_file:
            print('pylc calibrate needs a mask for every image; none for %s.' % img_file, file=sys.stderr)
            sys.exit(2)
        img = tools.get_image(img_file, model.meta.ch, scale=params.scale)[0]
        gt = tools.get_image(mask_file, ch=3, scale=params.scale, interpolate=cv2.INTER_NEAREST)[0]
        try:
            fit.add(img, gt)
        except ResidentBudgetError as exc:
            print('pylc calibrate: %s' % exc, file=sys.stderr)
            sys.exit(2)
    before = fit.report(1.0)
    res = fit.fit()
    after = fit.report(res['temperature'])
    if res['at_bound']:
        print('Warning: the best temperature %g lies at the end of the searched range [0.05, 20]; the minimum may lie '
              'outside it.' % res['temperature'])
    calibration = {'temperature': res['temperature'], 'n_images': len(fit.retained), 'n_px': fit.n_px,
                   'nll_before': before['nll'], 'nll_after': after['nll']}
    write_calibrated_copy(args.model, out_file, calibration)
    metrics_dir = tools.mk_path(os.path.join(defaults.output_dir, str(model.meta.id), 'metrics'))
    fit_file = os.path.join(metrics_dir, 'calibration_fit.json')
    with open(fit_file, 'w') as fp:
        json.dump({'temperature': res['temperature'], 'at_bound': res['at_bound'],
                   'evaluations': [[t, v] for t, v in res['evals']], 'before': before, 'after': after}, fp, indent=4)
    print('Temperature %.6g: NLL %.6g -> %.6g, ECE %.4g -> %.4g, accuracy %.4f -> %.4f' % (
        res['temperature'], before['nll'], after['nll'], before['ece'], after['ece'], before['accuracy'],
        after['accuracy']))
    print('Calibrated model saved to:\n\t%s\nFit report:\n\t%s' % (out_file, fit_file))
    return calibration


# ---- parser -----------------------------------------------------------------------------------

def get_parser():
    parser = argparse.ArgumentParser(prog='pylc', description='PyLC tiled-segmentation path on B200 (pylc_b200).')
    sub = parser.add_subparsers(title='actions', dest='action')
    sub.required = True

    def common(p):
        p.add_argument('--schema', type=str, default=defaults.schema, help='Categorization schema (JSON file).')

    p = sub.add_parser('extract', help='Extract tiles from images/masks and profile them.')
    common(p)
    p.set_defaults(func=extract)
    p.add_argument('-i', '--img', type=str, default='./data/raw/images/', required=True, help='Path to images directory or file.')
    p.add_argument('-m', '--mask', type=str, default=None, help='Path to masks directory or file (optional, as in the reference).')
    p.add_argument('--ch', type=int, default=3, required=True, choices=defaults.ch_options, help='Number of image channels.')
    p.add_argument('--batch_size', type=int, default=defaults.batch_size)
    p.add_argument('-o', '--output', type=str, default=None, help='Database output directory.')

    p = sub.add_parser('profile', help='Profile an extraction database.')
    common(p)
    p.set_defaults(func=profile)
    p.add_argument('--db', type=str, required=True, help='Path to database file.')

    p = sub.add_parser('augment', help='Data augmentation for database.')
    common(p)
    p.set_defaults(func=augment)
    p.add_argument('--db', type=str, required=True, help='Path to database file.')
    p.add_argument('--device_warps', action='store_true',
                   help='Make the over-sampled copies with pylc_augment_tiles_u8 (same bytes as the OpenCV calls).')

    p = sub.add_parser('train', help='Train model on an extraction database.')
    common(p)
    p.set_defaults(func=train)
    p.add_argument('--db', type=str, required=True)
    p.add_argument('--arch', type=str, default=defaults.arch, choices=defaults.arch_options)
    p.add_argument('--backbone', type=str, default=defaults.backbone, choices=defaults.backbone_options)
    # the reference's --weighted takes a value (any non-empty string enables it); the bare flag is accepted too
    p.add_argument('--weighted', nargs='?', const=True, default=None, help='Weight cross-entropy by class (profile weights).')
    p.add_argument('--ce_weight', type=float, default=defaults.ce_weight)
    p.add_argument('--dice_weight', type=float, default=defaults.dice_weight)
    p.add_argument('--focal_weight', type=float, default=defaults.focal_weight)
    p.add_argument('--optim', type=str, default=defaults.optim_type, choices=defaults.optim_options)
    p.add_argument('--sched', type=str, default=defaults.sched_type, choices=defaults.sched_options)
    p.add_argument('--lr', type=float, default=defaults.lr)
    p.add_argument('--batch_size', type=int, default=defaults.batch_size)
    p.add_argument('--n_epochs', type=int, default=defaults.n_epochs)
    # reference: a bare flag that loads defaults.pretrained; a path may follow here
    p.add_argument('--pretrained', nargs='?', const=True, default=None, help='Use pre-trained ResNet-101 weights (optionally: path).')
    # U-Net-only options of the reference parser: accepted for command-line compatibility, unused by DeepLabv3+
    p.add_argument('--normalize', type=str, default=defaults.norm_type, choices=defaults.norm_options)
    p.add_argument('--activation', type=str, default=defaults.activ_type, choices=defaults.activ_options)
    p.add_argument('--up_mode', type=str, default=defaults.up_mode, choices=defaults.up_mode_options)
    p.add_argument('--n_workers', type=int, default=defaults.n_workers)
    p.add_argument('--report', type=int, default=defaults.report)
    p.add_argument('--resume', action='store_true')
    p.add_argument('--clip', type=float, default=defaults.clip)

    p = sub.add_parser('test', help='Segment images with a trained model; evaluate against masks.')
    common(p)
    p.set_defaults(func=test)
    p.add_argument('-l', '--model', type=str, required=True, help='Path to trained PyLC model.')
    p.add_argument('-i', '--img', type=str, default='./data/raw/images/', help='Path to images directory or file.')
    p.add_argument('-m', '--mask', type=str, default=None)
    p.add_argument('--scale', type=float, default=defaults.scale)
    p.add_argument('--save_logits', action='store_true')
    p.add_argument('--aggregate_metrics', action='store_true')
    p.add_argument('--batch_tiles', type=int, default=32)
    # extensions: per-pixel probabilities (the mean of the covering tiles' softmaxes) and calibration
    p.add_argument('--stitch', type=str, default='reference', choices=['reference', 'mean'],
                   help="Labels from the reference's merge ('reference', default) or from the mean of the covering "
                        "tiles' softmaxes ('mean').")
    p.add_argument('--save_confidence', action='store_true',
                   help='Write full-resolution confidence PNGs (255 = 1.0); with masks, add calibration (ECE) to the metrics.')
    p.add_argument('--multiscale', type=float, nargs='+', default=None, metavar='S',
                   help='Average the class probabilities over these image scales (relative to the --scale image, at '
                        'most 8, no duplicates); needs --stitch mean.')
    p.add_argument('--temperature', type=float, default=None,
                   help="Softmax temperature of the mean stitch (default: the model file's fitted temperature, else "
                        "1; 1 turns a fitted temperature off); needs --stitch mean.")

    p = sub.add_parser('calibrate', help="Fit the mean stitch's softmax temperature on labelled images.")
    common(p)
    p.set_defaults(func=calibrate)
    p.add_argument('-l', '--model', type=str, required=True, help='Path to trained PyLC model.')
    p.add_argument('-i', '--img', type=str, required=True, help='Path to images directory or file.')
    p.add_argument('-m', '--mask', type=str, required=True, help='Path to masks directory or file.')
    p.add_argument('--scale', type=float, default=defaults.scale)
    p.add_argument('--batch_tiles', type=int, default=32)
    p.add_argument('-o', '--output', type=str, default=None,
                   help='Calibrated model file to write (default: <model stem>_calibrated.pth next to the model).')
    p.add_argument('--max_resident_gb', type=float, default=None,
                   help="Device memory for the retained network outputs (default: half the device's free memory).")
    return parser


def main(argv=None):
    args, unknown = get_parser().parse_known_args(argv)
    if unknown:
        print("\n'{}' is not a valid option. See usage:".format(unknown[0]))
        get_parser().print_usage()
        return 1
    _mkdirs()
    args.func(args)
    if pdist.is_initialized():
        torch.distributed.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
