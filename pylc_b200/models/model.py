"""
Model wrapper -- host-side mirror of PyLC's models/model.py, models/modules/checkpoint.py and the
RunningLoss log (reference model.py:29-492, checkpoint.py:17-66, loss.py:218-327).

Same interface: Model().load(path) / .build() / .resume() / .train(x, y) / .eval(x, y) -> [y_hat] /
.test(x) -> [y_hat] / .save() / .log(); attributes .net .meta .loss .iter .epoch .crit.  Same model
file format: torch.save({"model": state_dict, "optim": ..., "meta": Parameters}).

Only DeepLabv3+/ResNet-101 can be built -- it is the only architecture the reference can run
(SURVEY.md M3).  The network is stock PyTorch (cuDNN tensor-core convolutions); what changes is
around it: the multi-loss is the fused kernel pair (modules/loss.py), its three component values
are read with one D2H copy instead of three .item() syncs (model.py:319), and `test_tiles()`
consumes network-ready f32 tiles produced on the device by pylc_tile_gather_norm_f32 (which fuses
normalize_image and the grayscale x3 replicate, model.py:372-377,416-445).
"""
import os
import random

import numpy as np
import torch
import torch.nn as nn

from ..config import Parameters, defaults
from ..utils.tools import get_fname, mk_path
from .deeplab import DeepLab
from .modules.loss import MultiLoss


def strip_module_prefix(state_dict):
    """State dict saved from a DistributedDataParallel / DataParallel wrapper -> bare network keys."""
    if state_dict and all(k.startswith('module.') for k in state_dict):
        return type(state_dict)((k[len('module.'):], v) for k, v in state_dict.items())
    return state_dict


class Checkpoint:
    """Training checkpoint + best-model files under <save_dir>/<id>/ (reference checkpoint.py:17-66)."""

    def __init__(self, model_id, save_dir=None):
        save_dir = save_dir or defaults.save_dir
        self.model_dir = mk_path(os.path.join(save_dir, model_id))
        self.checkpoint_file = os.path.join(self.model_dir, 'checkpoint.pth')
        self.model_file = os.path.join(self.model_dir, model_id + '.pth')

    def load(self):
        if os.path.exists(self.checkpoint_file):
            print('\nCheckpoint found at:\n\t{}\n\tResuming!'.format(self.checkpoint_file))
            return torch.load(self.checkpoint_file, weights_only=False)
        print('\nCheckpoint does not exist. Starting new.')

    def reset(self):
        if os.path.exists(self.checkpoint_file):
            os.remove(self.checkpoint_file)

    def save(self, model, is_best=False):
        # a DistributedDataParallel wrapper prefixes every key with "module."; the model file holds the
        # bare network's keys (what Model.load, resume and the reference read back)
        net = getattr(model.net, 'module', model.net)
        state = {"model": net.state_dict(), "optim": model.optim.state_dict(), "meta": model.meta}
        torch.save(dict(state, epoch=model.epoch, iter=model.iter), self.checkpoint_file)
        if is_best:
            torch.save(state, self.model_file)


class RunningLoss(object):
    """Interval loss log: (iter, ce, dice, focal) rows for train / valid, best Dice, lr trace
    (reference loss.py:218-327).  `intv` rows may hold device tensors; they are only read at log()."""

    def __init__(self, model_id, save_dir=None, resume=False):
        self.train, self.valid, self.test = [], [], []
        self.intv = []
        self.avg_ce, self.avg_dice, self.best_dice, self.avg_fl = 0., 1., 1., 0.
        self.is_best = False
        self.lr = []
        self.resume = resume
        self.model_dir = os.path.join(save_dir or defaults.save_dir, model_id)
        self.log_file = os.path.join(mk_path(self.model_dir), 'losses.pth')
        self.load()

    def load(self):
        if os.path.exists(self.log_file):
            if self.resume:
                res = torch.load(self.log_file, weights_only=False)
                self.train, self.valid, self.test = res['train'], res['valid'], res['test']
                self.best_dice = res['best_dice']
            else:
                os.remove(self.log_file)

    def log(self, iteration, training):
        if not self.intv:
            return
        rows = torch.stack([torch.as_tensor(r, dtype=torch.float32).flatten()[-3:].cpu() if not torch.is_tensor(r)
                            else r.detach().float().flatten()[-3:].cpu() for r in self.intv])
        self.avg_ce, self.avg_dice, self.avg_fl = [float(v) for v in rows.mean(dim=0)]
        self.intv = []
        row = (iteration, self.avg_ce, self.avg_dice, self.avg_fl)
        if training:
            self.train += [row]
        else:
            self.valid += [row]
            self.is_best = self.avg_dice < self.best_dice
            if self.is_best:
                self.best_dice = self.avg_dice

    def save(self):
        torch.save({"train": self.train, "valid": self.valid, "test": self.test, "best_dice": self.best_dice,
                    "lr": self.lr}, self.log_file)

    def print_status(self, mode):
        mode = 'Training' if mode == defaults.TRAIN else 'Validation'
        hline = '_' * 40
        print('\nLoss Update\n' + hline)
        print('{:30s} {}'.format('Mode', mode))
        print('{:30s} {:4f}'.format('CE Average', self.avg_ce))
        print('{:30s} {:4f}'.format('Focal Average', self.avg_fl))
        print('{:30s} {:4f}'.format('Dice Average', self.avg_dice))
        print('{:30s} {:4f}'.format('Best Dice Average', self.best_dice))
        print(hline + '\n')


class Model:
    def __init__(self):
        self.meta = defaults
        # one process per GPU: the process's current CUDA device (dist.init_from_env selects LOCAL_RANK's),
        # not the import-time default "cuda:0" of config.py
        self.device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() \
            else torch.device(self.meta.device)
        self.net = None
        self.model_path = None
        self.calibration = None     # the model file's "calibration" entry (pylc calibrate), None when it has none
        self.iter = 0
        self.crit = None
        self.loss = None
        self.epoch = 0
        self.optim = None
        self.sched = None
        self.crop_target = False
        self.checkpoint = None
        self.resume_checkpoint = False
        self.distributed = False
        self.is_writer = True       # data parallel: only rank 0 writes checkpoint / loss-log files
        self.track = True           # False: no checkpoint / loss-log files (benchmarks, tests)
        self.normalizers = {'batch': nn.BatchNorm2d, 'instance': nn.InstanceNorm2d,
                            'layer': nn.LayerNorm, 'syncbatch': nn.SyncBatchNorm}

    # ---- construction -------------------------------------------------------------------------
    def load(self, model_path):
        """Load a PyLC model file for evaluation (reference model.py:78-121)."""
        if not model_path:
            print("\nModel path is empty. Use '--model' option to specify path.")
            exit(1)
        print('\nLoading model:\n\t{}'.format(model_path))
        if not os.path.exists(model_path):
            print('Model file does not exist.')
            exit()
        self.model_path = model_path
        try:
            model_data = _load_model_file(model_path, self.device)
        except Exception as err:
            print('An error occurred loading model:\n\t{}.'.format(model_path))
            print(err)
            exit()
        assert 'meta' in model_data, '\nLoaded model missing metadata attribute.'
        self.meta.update(model_data["meta"] if isinstance(model_data["meta"], dict) else vars(model_data["meta"]))
        self.meta.pretrained = False
        self.calibration = model_data.get("calibration")
        self.build()
        self.net.load_state_dict(strip_module_prefix(model_data["model"]))
        return self

    def build(self):
        """Build network, criterion, optimiser, scheduler from metadata (reference model.py:123-220)."""
        self.gen_id()
        if self.meta.arch != 'deeplab' or self.meta.backbone != 'resnet':
            # unet / resunet cannot be constructed or run in the reference either (SURVEY.md M3)
            print('Model {} ({}) not available.'.format(self.meta.arch, self.meta.backbone))
            exit(1)
        self.net = DeepLab(n_classes=self.meta.n_classes, normalizer=self.normalizers[self.meta.norm_type],
                           in_channels=self.meta.ch)
        if self.meta.pretrained and isinstance(self.meta.pretrained, str) and os.path.isfile(self.meta.pretrained):
            wanted = self.net.backbone.state_dict()
            found = torch.load(self.meta.pretrained, map_location='cpu')
            wanted.update({k: v for k, v in found.items() if k in wanted})
            self.net.backbone.load_state_dict(wanted)
        self.net = self.net.to(self.device)
        self.crit = MultiLoss(
            loss_weights={'weighted': self.meta.weighted, 'weights': self.meta.weights, 'ce': self.meta.ce_weight,
                          'dice': self.meta.dice_weight, 'focal': self.meta.focal_weight},
            schema={'n_classes': self.meta.n_classes, 'class_codes': self.meta.class_codes,
                    'class_labels': self.meta.class_labels},
            distributed=self.distributed, ddp_average=self.distributed)
        # no host sync per training step: a target outside [0, n_classes) turns the step's loss values into
        # NaN on the device, and log() -- the first place they are read -- raises
        self.crit.validate_targets = False
        if self.track:
            self.checkpoint = Checkpoint(self.meta.id, self.meta.save_dir)      # every rank may resume from it
        if self.track and self.is_writer:
            self.loss = RunningLoss(self.meta.id, save_dir=self.meta.save_dir, resume=self.meta.resume_checkpoint)
        else:
            self.loss = _NullLoss()
        self.optim = self.init_optim()
        self.sched = self.init_sched()
        return self

    def resume(self):
        if self.resume_checkpoint:
            data = self.checkpoint.load()
            if data is not None:
                self.epoch, self.iter, self.meta = data['epoch'], data['iter'], data["meta"]
                self.net.load_state_dict(strip_module_prefix(data["model"]))
                self.optim.load_state_dict(data["optim"])
        elif self.checkpoint is not None and self.is_writer:
            self.checkpoint.reset()

    def init_optim(self):
        if self.meta.optim_type == 'adam':
            return torch.optim.AdamW(self.net.parameters(), lr=self.meta.lr, weight_decay=self.meta.weight_decay)
        if self.meta.optim_type == 'sgd':
            return torch.optim.SGD(self.net.parameters(), lr=self.meta.lr, momentum=self.meta.momentum)
        print('Optimizer is not defined.')
        exit()

    def init_sched(self):
        if self.meta.sched_type == 'step_lr':
            return torch.optim.lr_scheduler.StepLR(self.optim, step_size=1, gamma=self.meta.gamma)
        if self.meta.sched_type == 'cyclic_lr':
            return torch.optim.lr_scheduler.CyclicLR(self.optim, self.meta.lr_min, self.meta.lr_max, step_size_up=2000)
        if self.meta.sched_type == 'anneal':
            return None
        print('Optimizer scheduler is not defined.')
        exit()

    # ---- steps --------------------------------------------------------------------------------
    def _prepare(self, x, default=False):
        x = self.normalize_image(x, default=default).to(self.device, non_blocking=True)
        if self.meta.ch == 1 and self.meta.arch == 'deeplab':
            x = torch.cat((x, x, x), 1)
        return x

    def train(self, x, y):
        """One optimisation step (reference model.py:282-336)."""
        if bool(random.randint(0, 1)):
            x = torch.flip(x, [3])
            y = torch.flip(y, [2])
        x = self._prepare(x)
        y = y.to(self.device, non_blocking=True)
        y_hat = self.net.forward(x)
        loss = self.crit.forward(y_hat, y)
        self.loss.intv += [self.crit.last]        # device tensor (loss, ce, dice, focal); no sync here
        self.optim.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.net.parameters(), 0.5)
        self.optim.step()
        if self.iter % self.meta.report == 0:
            self.log()
        self.loss.lr += [(self.iter, self.get_lr())]
        self.iter += 1
        return loss

    def eval(self, x, y):
        """Validation step (reference model.py:338-365): forward + the three loss components."""
        self.net.eval()
        x = self._prepare(x)
        y = y.to(self.device, non_blocking=True)
        with torch.no_grad():
            y_hat = self.net.forward(x)
            ce, dice, focal = self.crit.components(y_hat, y)
            self.loss.intv += [torch.stack((ce, dice, focal))]
        return [y_hat]

    def test(self, x):
        """Forward pass on a batch of u8/f32 tiles [B,ch,T,T] (reference model.py:367-382)."""
        x = self._prepare(x, default=self.meta.normalize_default)
        with torch.no_grad():
            return [self.net.forward(x)]

    def test_tiles(self, tiles_f32):
        """Forward pass on network-ready tiles [B,3,T,T] f32 already normalised on the device."""
        with torch.no_grad():
            return [self.net.forward(tiles_f32)]

    def norm_params(self, default=None):
        """(mean[3], std[3], post_div, out_ch) that make pylc_tile_gather_norm_f32 reproduce
        normalize_image + the x3 replicate for this model (reference model.py:416-445)."""
        default = self.meta.normalize_default if default is None else default
        if self.meta.ch == 1:
            if default:
                return [defaults.px_grayscale_mean] * 3, [defaults.px_grayscale_std] * 3, 1.0, 3
            mean = float(np.mean(self.meta.px_mean))
            std = float(np.mean(self.meta.px_std))
            return [mean] * 3, [std] * 3, 255.0, 3
        if default:
            return list(defaults.px_rgb_mean), list(defaults.px_rgb_std), 255.0, 3
        return list(self.meta.px_mean), list(self.meta.px_std), 255.0, 3

    def normalize_image(self, img, default=False):
        """((x - mean) / std) / 255 with the profiled or default statistics (model.py:416-445)."""
        img = torch.as_tensor(img).float()
        mean, std, post_div, _ = self.norm_params(default)
        n = img.shape[1]
        m = torch.tensor(mean[:n], dtype=torch.float32, device=img.device)[None, :, None, None]
        s = torch.tensor(std[:n], dtype=torch.float32, device=img.device)[None, :, None, None]
        return ((img - m) / s) / post_div

    # ---- bookkeeping --------------------------------------------------------------------------
    def log(self):
        self.loss.log(self.iter, self.net.training)
        if self.loss.avg_ce != self.loss.avg_ce:
            raise FloatingPointError("loss is NaN: a target outside [0, n_classes) (the reference's CrossEntropyLoss "
                                     "raises on it) or non-finite logits")
        self.loss.save()

    def save(self):
        if self.checkpoint is not None and self.is_writer:
            self.checkpoint.save(self, is_best=self.loss.is_best)
        self.loss.save()

    def get_lr(self):
        for group in self.optim.param_groups:
            return group['lr']

    def get_meta(self):
        return self.meta

    def update_meta(self, params):
        self.meta.update(params)
        return self

    def gen_id(self):
        if self.model_path is None:
            self.meta.id = 'pylc_' + self.meta.arch + '_ch' + str(self.meta.ch) + '_' + self.meta.schema_name
        else:
            self.meta.id = get_fname(self.model_path)

    def print_settings(self):
        hline = '_' * 40
        print("\nModel Configuration")
        print(hline)
        print('{:30s} {}'.format('ID', self.meta.id))
        if self.model_path is not None:
            print('{:30s} {}'.format('Model File', os.path.basename(self.model_path)))
        print('{:30s} {}'.format('Architecture', self.meta.arch))
        print('   - {:25s} {}'.format('Backbone', self.meta.backbone))
        print('{:30s} {}'.format('Input channels', self.meta.ch))
        print('{:30s} {}'.format('Output channels', self.meta.n_classes))
        print('{:30s} {}{}'.format('Px mean', self.meta.px_mean, '*' if self.meta.normalize_default else ''))
        print('{:30s} {}{}'.format('Px std-dev', self.meta.px_std, '*' if self.meta.normalize_default else ''))
        print('{:30s} {}'.format('Batch size', self.meta.batch_size))
        print('{:30s} {}'.format('Optimizer', self.meta.optim_type))
        print('{:30s} {}'.format('Scheduler', self.meta.sched_type))
        print('{:30s} {}'.format('Learning rate (default)', self.meta.lr))
        print()
        self.crit.print_settings()


class _NullLoss(object):
    """Loss log that keeps nothing on disk (track=False)."""
    is_best = False
    avg_ce = 0.

    def __init__(self):
        self.intv, self.lr = [], []

    def log(self, *a, **k):
        self.intv = []

    def save(self):
        pass


def _load_model_file(path, device):
    """torch.load of a PyLC model file.  `meta` is a pickled config.Parameters of whichever
    package wrote the file; files written by the reference resolve `config.Parameters` to ours."""
    import pickle
    import sys
    import types

    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            if module == 'config' and name in ('Parameters', 'Schema'):
                from .. import config as cfg
                return getattr(cfg, name)
            return super().find_class(module, name)

    shim = types.ModuleType('_pylc_pickle')
    shim.Unpickler = _Unpickler
    shim.load = lambda f, **kw: _Unpickler(f, **kw).load()
    shim.__name__ = 'pickle'
    for attr in ('loads', 'dumps', 'dump', 'Pickler', 'HIGHEST_PROTOCOL', 'DEFAULT_PROTOCOL', 'PickleError',
                 'UnpicklingError', 'PicklingError'):
        setattr(shim, attr, getattr(pickle, attr))
    return torch.load(path, map_location=device, weights_only=False, pickle_module=shim)
