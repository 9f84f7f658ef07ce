"""Thin mirror of the reference's training / scoring base class.

Keeps the public surface of
/root/reference/point_vs/models/point_neural_network_base.py
(constructor signature :49-54, `train_model` :136, `val` :208, `get_loss`
:362, `backprop` :417, `save` :501, `load_weights` :528, `param_count`,
`set_task` :572, prediction-file line formats :289-319, checkpoint dict keys
:509-516) so `load_model` / `inference` and existing checkpoints work against
the CUDA models.  wandb / rich progress reporting is not part of the hot path
and is left out; per-batch host syncs are limited to what the file formats
need.
"""
import math
import time
from collections import OrderedDict
from pathlib import Path

import numpy as np
import torch
import yaml
from torch import nn

from . import _cabi

DEVICE = torch.device('cuda' if torch.cuda.is_available() else 'cpu')


def check_trainable_width(k):
    """The backward kernels cover hidden widths up to _cabi.MAX_K; wider
    models (up to _cabi.MAX_K_TC_FWD) can be scored but not trained."""
    if k is not None and int(k) > _cabi.MAX_K:
        raise NotImplementedError(
            f'hidden width {k}: training supports --channels up to '
            f'{_cabi.MAX_K}; models up to {_cabi.MAX_K_TC_FWD} channels can '
            'only be scored, in a tensor-core math mode')


def find_latest_checkpoint(root, model_task=None):
    """Most recently created checkpoint under root/checkpoints, as the
    reference picks it (utils.py:33-45: glob `<model_task>*.pt`, newest by
    st_ctime).  In a multitask pose -> affinity run that is the affinity
    checkpoint written last, not the file with the largest epoch number."""
    if model_task is not None and model_task not in ('pose', 'affinity'):
        raise RuntimeError(
            'model_task must be either pose or affinity if specified.')
    root = Path(root).expanduser()
    ckpt_dir = root / 'checkpoints' if (root / 'checkpoints').is_dir() else root
    found = list(ckpt_dir.glob((model_task or '') + '*.pt'))
    if not found:
        raise FileNotFoundError(f'No checkpoints found in {root}.')
    # ties (same ctime tick) go to the later file name, deterministically
    return max(found, key=lambda f: (f.stat().st_ctime_ns, f.name))


def top_n(predictions_file, n=1):
    """Fraction of receptors whose n best-scored poses contain an active
    (analysis/top_n.py:41-49 of the reference: predictions grouped by the
    receptor column, sorted by y_pred descending)."""
    scores = {}
    with open(Path(predictions_file).expanduser(), encoding='utf-8') as f:
        for line in f:
            parts = line.split()
            if len(parts) < 5:
                continue
            scores.setdefault(parts[3], []).append(
                (float(parts[2]), int(float(parts[0]))))
    if not scores:
        return 0.0
    hits = 0
    for vals in scores.values():
        vals.sort(key=lambda v: v[0], reverse=True)
        hits += 1 if sum(v[1] for v in vals[:n]) else 0
    return hits / len(scores)


def get_regression_pearson(predictions_file):
    """(r, p) of y_true vs y_pred in a predictions file (utils.py:189-198)."""
    from scipy.stats import pearsonr
    true, pred = [], []
    with open(Path(predictions_file).expanduser(), encoding='utf-8') as f:
        for line in f:
            parts = line.split()
            if len(parts) >= 5:
                true.append(float(parts[0]))
                pred.append(float(parts[2]))
    return pearsonr(true, pred)


class PointNeuralNetworkBase(nn.Module):
    """Optimiser, losses, train/val loops, checkpoint I/O."""

    def __init__(self, save_path, learning_rate, weight_decay=None,
                 wandb_project=None, wandb_run=None, silent=False,
                 use_1cycle=False, warm_restarts=False,
                 only_save_best_models=False, optimiser='adam',
                 regression_loss='mse', **model_kwargs):
        super().__init__()
        self.set_task(model_kwargs.get('model_task', 'classification'))
        self.include_strain_info = False
        self.batch = 0
        self.p_epoch = self.a_epoch = 0
        self.save_path = Path(save_path).expanduser()
        self.only_save_best_models = only_save_best_models
        if not silent:
            self.save_path.mkdir(parents=True, exist_ok=True)
        self.predictions_file = Path(self.save_path, 'predictions.txt')
        self.lr = learning_rate
        self.weight_decay = weight_decay
        self.bce = nn.BCEWithLogitsLoss()
        self.regression_loss = nn.MSELoss() if regression_loss == 'mse' \
            else nn.HuberLoss()
        self.wandb_project, self.wandb_run = wandb_project, wandb_run
        self.n_layers = model_kwargs.get('num_layers', 12)
        self.feats_linear_layers = None
        self.layers = self.build_net(**model_kwargs)
        wd = 0 if weight_decay is None else weight_decay
        if optimiser == 'adam':
            self.optimiser = torch.optim.Adam(
                self.parameters(), lr=self.lr, weight_decay=wd)
        elif optimiser == 'sgd':
            self.optimiser = torch.optim.SGD(
                self.parameters(), lr=self.lr, momentum=0.9, weight_decay=wd,
                nesterov=True)
        else:
            raise NotImplementedError(f'{optimiser} not recognised optimiser.')
        assert not (use_1cycle and warm_restarts), \
            '1cycle and warm restarts are mutually exclusive'
        self.use_1cycle, self.warm_restarts = use_1cycle, warm_restarts
        self.scheduler = None
        self.global_iter = self.val_iter = 0
        self.decoy_mean_pred = self.active_mean_pred = 0.5
        self.log_interval = 10
        self.test_metric = 0
        if not silent:
            with open(self.save_path / 'model_kwargs.yaml', 'w',
                      encoding='utf-8') as f:
                yaml.dump({k: v for k, v in model_kwargs.items()
                           if not isinstance(v, nn.Module)}, f)
        self.to(DEVICE)

    # -- to be provided by the model classes ---------------------------------
    def build_net(self, **model_kwargs):
        raise NotImplementedError

    def unpack_input_data_and_predict(self, input_data):
        raise NotImplementedError

    # -- task ------------------------------------------------------------------
    def set_task(self, task):
        if task not in ('classification', 'regression', 'multi_regression'):
            raise ValueError('Argument for set_task must be one of '
                             'classification, regression or multi_regression')
        self.model_task = task
        regress = 'regression' in task
        self.model_task_for_fnames = 'affinity' if regress else 'pose'
        self.model_task_string = 'Mean squared error' if regress \
            else 'Binary crossentropy'

    @property
    def param_count(self):
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    # -- loss / step -------------------------------------------------------------
    def get_loss(self, y_true, y_pred):
        y_true = y_true.to(y_pred.device)
        if self.model_task == 'classification':
            return self.bce(y_pred, y_true)
        if self.model_task == 'regression':
            return self.regression_loss(y_pred, y_true)
        # multi_regression: unlabeled targets are -1; one of three is real
        y_pred = torch.where(y_true == -1, torch.full_like(y_pred, -1), y_pred)
        return 3 * self.regression_loss(y_pred, y_true)

    def sync_gradients(self):
        """Hook for data-parallel training (pointvs_b200.parallel)."""

    _grad_arena = None

    def _arena_for_step(self, loss):
        """The flat gradient arena (parallel.GradArena) the backward kernels
        write into: one memset per step instead of a zero-filled tensor per
        layer, and no pack / unpack copies around the data-parallel
        all-reduce.  CUDA models only."""
        if not loss.is_cuda:
            return None
        if not getattr(self, '_fused_optimiser', False):
            # torch.optim.Adam with fused=True is the same update in ONE kernel
            # instead of ~20 foreach launches (1.1 ms -> 0.1 ms per step on the
            # 8 x 64 model); the flag lives in the param groups, which were
            # created while the parameters were still on the CPU
            self._fused_optimiser = True
            if isinstance(self.optimiser, torch.optim.Adam):
                for group in self.optimiser.param_groups:
                    group['fused'], group['foreach'] = True, False
        arena = self._grad_arena
        if arena is None or not arena.matches(self):
            from .parallel import GradArena
            arena = GradArena(self)
            self._grad_arena = arena
        return arena

    def backprop(self, y_true, y_pred, sync=True):
        """loss -> backward -> (all-reduce) -> clip -> optimiser step
        (point_neural_network_base.py:417-429).  sync=True returns the loss as
        a float and raises on NaN at once, as the reference does; sync=False
        returns the loss as a device tensor and leaves the NaN check to the
        caller, so the host can run ahead of the device (N1)."""
        self._check_trainable()
        loss = self.get_loss(y_true, y_pred)
        arena = self._arena_for_step(loss)
        # from now on the forward passes of this model may take the lean
        # training path (egnn._EGNNStackLeanFn): its parameter gradients reach
        # `p.grad` through the arena below instead of through autograd
        self._lean_training = arena is not None
        if arena is None:
            self.optimiser.zero_grad()
            loss.backward()
        else:
            # gradients live in one flat arena that the backward kernels write
            # directly: zeroing it replaces optimiser.zero_grad(), and p.grad
            # stays attached to its slot from step to step
            from . import backward as _bw
            arena.begin_step()
            with _bw.use_arena(arena):
                loss.backward()
            arena.attach_grads()
        self.sync_gradients()
        if arena is None:
            torch.nn.utils.clip_grad_value_(self.parameters(), 1.0)
        else:
            # clip_grad_value_(parameters, 1.0) as one clamp over the arena
            rest = arena.clamp_(1.0)
            if rest:
                torch.nn.utils.clip_grad_value_(rest, 1.0)
        self.optimiser.step()
        if not sync:
            return loss.detach()
        loss_ = float(loss.detach())
        if math.isnan(loss_):
            raise FloatingPointError('We have hit a NaN loss value.')
        return loss_

    @staticmethod
    def _drain_losses(pending, losses, overflow=None):
        """One device->host transfer for the losses of the last few steps (and
        for the edge-capacity overflow flags of their graphs, if the loader
        builds capacity-bounded graphs)."""
        if pending:
            vals = torch.stack(pending).cpu().tolist()
            pending.clear()
            if any(math.isnan(v) for v in vals):
                raise FloatingPointError('We have hit a NaN loss value.')
            losses.extend(vals)
        if overflow:
            dropped = int(torch.stack(overflow).sum().item())
            overflow.clear()
            if dropped:
                raise RuntimeError(
                    'edge capacity exceeded while training: a batch had more '
                    'edges than its capacity-bounded edge list holds; build '
                    'the loader with edge_capacity=None (exact edge lists) '
                    'or a larger bound')

    def training_setup(self, data_loader, epochs, model_task=None):
        if self.use_1cycle:
            self.scheduler = torch.optim.lr_scheduler.OneCycleLR(
                self.optimiser, max_lr=self.lr,
                steps_per_epoch=epochs * len(data_loader), epochs=1)
        elif self.warm_restarts:
            self.scheduler = \
                torch.optim.lr_scheduler.CosineAnnealingWarmRestarts(
                    self.optimiser, T_0=len(data_loader), T_mult=1, eta_min=0)
        if model_task is not None:
            self.set_task(model_task)
        init_epoch = self.a_epoch if 'regression' in self.model_task \
            else self.p_epoch
        return init_epoch, time.time()

    def _check_trainable(self):
        if '_width_checked' not in self.__dict__:     # once per model
            check_trainable_width(max(
                (m.hidden_nf for m in self.modules() if hasattr(m, 'hidden_nf')),
                default=None))
            self.__dict__['_width_checked'] = True

    def train_model(self, data_loader, epochs=1, epoch_end_validation_set=None,
                    top1_on_end=False):
        self._check_trainable()
        init_epoch, _ = self.training_setup(data_loader, epochs)
        losses, pending, overflow = [], [], []
        for _ in range(init_epoch, epochs):
            self.train()
            for self.batch, graph in enumerate(data_loader):
                y_pred, y_true, _, _ = self.unpack_input_data_and_predict(graph)
                pending.append(self.backprop(y_true, y_pred, sync=False))
                csr = getattr(graph, 'pvs_csr', None)
                if csr is not None and not csr.exact_edge_count:
                    overflow.append(csr._overflow)
                # losses (and the NaN / overflow checks) come back once per
                # log interval, not once per step
                if len(pending) >= self.log_interval:
                    self._drain_losses(pending, losses, overflow)
                if self.scheduler is not None:
                    self.scheduler.step()
                self.global_iter += 1
            self._drain_losses(pending, losses, overflow)
            self.eval()
            self.on_epoch_end(epoch_end_validation_set, epochs, top1_on_end)
        return losses

    def on_epoch_end(self, epoch_end_validation_set, epochs, top1_on_end):
        if 'regression' in self.model_task:
            self.a_epoch += 1
            epoch = self.a_epoch
        else:
            self.p_epoch += 1
            epoch = self.p_epoch
        if not self.only_save_best_models:
            self.save()
        if epoch_end_validation_set is not None and epoch < epochs:
            best = self.val(
                epoch_end_validation_set, predictions_file=Path(
                    self.predictions_file.parent,
                    f'predictions_epoch_{epoch}.txt'),
                top1_on_end=top1_on_end)
            if self.only_save_best_models and best:
                self.save()

    # -- scoring -------------------------------------------------------------------
    def val(self, data_loader, predictions_file=None, top1_on_end=False,
            rich_ctx=None):
        """Score a loader and write the reference's predictions file."""
        if predictions_file is None:
            predictions_file = self.predictions_file
        predictions_file = Path(predictions_file)
        predictions_file = (predictions_file.parent / (
            f'{self.model_task_for_fnames}_' + predictions_file.name)
                            ).expanduser()
        if predictions_file.is_file():
            predictions_file.unlink()
        self.eval()
        self.val_iter = 0
        n_batches = len(data_loader)
        pending = []      # (y_pred device tensor, y_true, ligands, receptors)
        with torch.no_grad():
            for self.batch, graph in enumerate(data_loader):
                self.val_iter += 1
                y_pred, y_true, ligands, receptors = \
                    self.unpack_input_data_and_predict(graph)
                if self.model_task == 'classification':
                    y_pred = torch.sigmoid(y_pred)
                pending.append((y_pred, y_true, ligands, receptors))
                # one device->host transfer per log interval, not per batch
                if not (self.batch + 1) % self.log_interval or \
                        self.batch == n_batches - 1:
                    text = ''.join(self._format_predictions(*p)
                                   for p in pending)
                    pending = []
                    with open(predictions_file, 'a', encoding='utf-8') as f:
                        f.write(text)
        if top1_on_end:
            # best-model tracking (point_neural_network_base.py:330-360): top-1
            # for pose classification, Pearson r (p < 0.05) for regression
            if self.model_task == 'classification':
                metric = top_n(predictions_file)
                best = metric > self.test_metric
            else:
                metric, p_value = get_regression_pearson(predictions_file)
                best = p_value < 0.05 and metric > self.test_metric
            if best:
                self.test_metric = metric
            if self.only_save_best_models and not best:
                return False
        return True

    def _format_predictions(self, y_pred, y_true, ligands, receptors):
        n = len(receptors)
        if self.model_task == 'multi_regression':
            pred = y_pred.detach().cpu().numpy().reshape((-1, 3))
            first = y_true[0][0] if isinstance(y_true, (tuple, list)) \
                else (None if y_true is None else y_true[0])
            if first is None:
                return '\n'.join(
                    '{0:.3f} {1:.3f} {2:.3f} | {3} {4}'.format(
                        *pred[i], receptors[i], ligands[i])
                    for i in range(n)) + '\n'
            true = torch.as_tensor(y_true).cpu().numpy().reshape((-1, 3))
            names = np.array([['pki', 'pkd', 'ic50']] * n)
            sel = np.where(true > -0.5)
            metrics, pred, true = list(names[sel]), pred[sel], true[sel]
            return '\n'.join(
                '{0:.3f} | {1:.3f} {2} {3} | {4}'.format(
                    float(true[i]), pred[i], receptors[i], ligands[i],
                    metrics[i]) for i in range(n)) + '\n'
        pred = y_pred.detach().cpu().numpy().reshape((-1,))
        num_type = int if self.model_task == 'classification' else float
        if y_true is None:
            return '\n'.join('{0:.3f} | {1} {2}'.format(
                pred[i], receptors[i], ligands[i]) for i in range(n)) + '\n'
        true = torch.as_tensor(y_true).cpu().numpy().reshape((-1,))
        return '\n'.join('{0:.3f} | {1:.3f} {2} {3}'.format(
            num_type(true[i]), pred[i], receptors[i], ligands[i])
            for i in range(n)) + '\n'

    # -- checkpoints -------------------------------------------------------------
    def save(self, save_path=None):
        epoch = self.a_epoch if 'regression' in self.model_task \
            else self.p_epoch
        if save_path is None:
            save_path = self.save_path / 'checkpoints' / \
                f'{self.model_task_for_fnames}_ckpt_epoch_{epoch}.pt'
        Path(save_path).parent.mkdir(parents=True, exist_ok=True)
        torch.save({
            'learning_rate': self.lr,
            'weight_decay': self.weight_decay,
            'p_epoch': self.p_epoch,
            'a_epoch': self.a_epoch,
            'model_state_dict': self.state_dict(),
            'optimiser_state_dict': self.optimiser.state_dict(),
        }, save_path)

    @staticmethod
    def _transform_names(d):
        """Key renames of old reference checkpoints (:520-526)."""
        import re
        return OrderedDict(
            (re.sub(r'(?<![A-Za-z_])att_mlp\.2\.', 'att_mlp.0.',
                    k.replace('edge_attention_mlp', 'att_mlp')
                     .replace('node_attention_mlp', 'node_att_mlp')), v)
            for k, v in d.items())

    def load_weights(self, checkpoint_file, silent=False):
        checkpoint_file = Path(checkpoint_file).expanduser()
        if checkpoint_file.is_dir():
            checkpoint_file = find_latest_checkpoint(checkpoint_file)
        checkpoint = torch.load(str(checkpoint_file), map_location=DEVICE,
                                weights_only=False)
        state = checkpoint['model_state_dict']
        kwargs_file = checkpoint_file.parents[1] / 'model_kwargs.yaml'
        saved_task = 'classification'
        if kwargs_file.is_file():
            with open(kwargs_file, encoding='utf-8') as f:
                saved_task = (yaml.safe_load(f) or {}).get(
                    'model_task', 'classification')
        if self.model_task == saved_task:
            try:
                self.load_state_dict(state)
            except RuntimeError as exc:
                # old reference checkpoints use other key names (:520-526);
                # a genuine shape mismatch must surface as it is
                msg = str(exc)
                if 'Missing key' not in msg and 'Unexpected key' not in msg:
                    raise
                self.load_state_dict(self._transform_names(state))
            try:
                self.optimiser.load_state_dict(
                    checkpoint['optimiser_state_dict'])
            except (ValueError, KeyError) as exc:
                import warnings
                warnings.warn(
                    f'optimiser state of {checkpoint_file} not restored '
                    f'({exc!r}): training resumes with fresh optimiser moments')
            self.p_epoch = checkpoint.get('p_epoch', checkpoint.get('epoch', 0))
            self.a_epoch = checkpoint.get('a_epoch', 0)
        else:
            own_state = self.state_dict()
            for name, param in state.items():
                own_state[name].copy_(param)
