"""Training entry point, mirror of /root/reference/point_vs.py (:35-420) for the
models on the B200 path.

    python -m pointvs_b200.train <egnn|multitask> <save_path> \
        --train_data_root_pose <root> --train_types_pose <types> -ep 1 \
        [--train_data_root_affinity <root> --train_types_affinity <types> -ea 1] \
        --layers 3 -k 32 --egnn_attention ... [--math fp32|bf16x3|fp16x2|bf16]

Same flags, same defaults, same `cmd_args.yaml` / `model_kwargs.yaml` /
`checkpoints/*.pt` / `*_predictions.txt` outputs (the flag -> kwarg map is
point_vs.py:189-221), so a run directory written here loads in the reference
and the other way round.  The loop is the reference's: pose epochs, pose
validation, affinity epochs, affinity validation.  Flags of features outside
this path (`lucid`, `--synth_pharm`, `--double`, wandb) are refused or ignored
as noted in `parse_args`.
"""
import argparse
import os
import socket
from pathlib import Path

import torch
import yaml

from .base import check_trainable_width
from .data import get_data_loader
from .egnn import MultitaskSatorrasEGNN, SartorrasEGNN


def parse_args(argv=None):
    """The reference's argument list (point_vs/parse_args.py), flag for flag."""
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('model', type=str, help='egnn or multitask')
    p.add_argument('save_path', type=str)
    p.add_argument('--train_data_root_pose', type=str)
    p.add_argument('--train_data_root_affinity', '--tdra', type=str)
    p.add_argument('--test_data_root_pose', type=str)
    p.add_argument('--test_data_root_affinity', type=str)
    p.add_argument('--logging_level', type=str, default='info')
    p.add_argument('--load_weights', '-l', type=str)
    p.add_argument('--translated_actives', type=str)
    p.add_argument('--batch_size', '-b', type=int, default=32)
    p.add_argument('--epochs_pose', '-ep', type=int, default=0)
    p.add_argument('--epochs_affinity', '-ea', type=int, default=0)
    p.add_argument('--channels', '-k', type=int, default=32)
    p.add_argument('--learning_rate', '-lr', type=float, default=0.002)
    p.add_argument('--weight_decay', '-w', type=float, default=1e-4)
    p.add_argument('--wandb_project', type=str)
    p.add_argument('--wandb_run', type=str)
    p.add_argument('--layers', type=int, default=6)
    p.add_argument('--radius', type=int, default=10)
    p.add_argument('--load_args', type=str)
    p.add_argument('--double', action='store_true')
    p.add_argument('--activation', type=str, default='relu')
    p.add_argument('--dropout', type=float, default=0.0)
    p.add_argument('--use_1cycle', action='store_true')
    p.add_argument('--warm_restarts', action='store_true')
    p.add_argument('--fourier_features', type=int, default=0)
    p.add_argument('--norm_coords', action='store_true')
    p.add_argument('--norm_feats', action='store_true')
    p.add_argument('--use_atomic_numbers', action='store_true')
    p.add_argument('--compact', action='store_true')
    p.add_argument('--thin_mlps', action='store_true')
    p.add_argument('--hydrogens', action='store_true')
    p.add_argument('--augmented_actives', type=int, default=0)
    p.add_argument('--min_aug_angle', type=float, default=30)
    p.add_argument('--max_active_rmsd', type=float)
    p.add_argument('--min_inactive_rmsd', type=float)
    p.add_argument('--val_on_epoch_end', '-v', action='store_true')
    p.add_argument('--synth_pharm', '-p', action='store_true')
    p.add_argument('--input_suffix', '-s', type=str, default='parquet')
    p.add_argument('--train_types_pose', type=str)
    p.add_argument('--train_types_affinity', type=str)
    p.add_argument('--test_types_pose', type=str)
    p.add_argument('--test_types_affinity', type=str)
    p.add_argument('--egnn_attention', action='store_true')
    p.add_argument('--egnn_tanh', action='store_true')
    p.add_argument('--egnn_normalise', action='store_true')
    p.add_argument('--egnn_residual', action='store_true')
    p.add_argument('--edge_radius', type=float, default=4.0)
    p.add_argument('--end_flag', action='store_true')
    p.add_argument('--wandb_dir', type=str)
    p.add_argument('--estimate_bonds', action='store_true')
    p.add_argument('--prune', action='store_true')
    p.add_argument('--top1', action='store_true')
    p.add_argument('--graphnorm', action='store_true')
    p.add_argument('--multi_fc', action='store_true')
    p.add_argument('--lucid_node_final_act', action='store_true')
    p.add_argument('--p_remove_entity', type=float, default=0)
    p.add_argument('--static_coords', action='store_true')
    p.add_argument('--permutation_invariance', action='store_true')
    p.add_argument('--node_attention', action='store_true')
    p.add_argument('--attention_activation_function', type=str,
                   default='sigmoid')
    p.add_argument('--only_save_best_models', action='store_true')
    p.add_argument('--egnn_edge_residual', action='store_true')
    p.add_argument('--gated_residual', action='store_true')
    p.add_argument('--rezero', action='store_true')
    p.add_argument('--extended_atom_types', action='store_true')
    p.add_argument('--max_inactive_rmsd', type=float)
    p.add_argument('--model_task', type=str, default='classification')
    p.add_argument('--synthpharm', action='store_true')
    p.add_argument('--p_noise', type=float, default=-1)
    p.add_argument('--include_strain_info', action='store_true')
    p.add_argument('--final_softplus', action='store_true')
    p.add_argument('--optimiser', '-o', type=str, default='adam')
    p.add_argument('--multi_target_affinity', action='store_true')
    p.add_argument('--regression_loss', type=str, default='mse')
    p.add_argument('--softmax_attention', action='store_true')
    # additions of this implementation
    p.add_argument('--math', default='bf16x3',
                   choices=['fp32', 'bf16x3', 'fp16x2', 'bf16'],
                   help='arithmetic of the dense contractions (forward and '
                        'the recompute inside the backward)')
    p.add_argument('--workers', type=int, default=4,
                   help='loader workers reading the parquets')
    p.add_argument('--worker_processes', action='store_true',
                   help='loader workers are spawned processes')
    p.add_argument('--host_crop', action='store_true',
                   help='crop / type the complexes on the host, not on the '
                        'device (K0)')
    return p.parse_args(argv)


def main(argv=None):
    args = parse_args(argv)
    # the --load_args overlay comes first (point_vs.py:54-58), so that values
    # it sets (double, synthpharm, model ...) meet the same checks as flags
    if args.load_args is not None:
        with open(Path(args.load_args).expanduser(), encoding='utf-8') as f:
            for key, value in (yaml.safe_load(f) or {}).items():
                if hasattr(args, key):
                    setattr(args, key, value)
    if args.model not in ('egnn', 'multitask'):
        raise NotImplementedError(
            f"model '{args.model}' is outside the B200 hot path "
            "(supported: egnn, multitask)")
    if args.model_task == 'both' and args.model != 'multitask':
        raise RuntimeError(
            'Sequential pose -> affinity training is only compatable with the '
            'multitask architecture')
    if args.double:
        raise NotImplementedError('--double: the CUDA path computes in fp32')
    if args.synth_pharm or args.synthpharm:
        raise NotImplementedError('synthpharm datasets are outside this path')
    check_trainable_width(args.channels)
    if args.wandb_project is None:
        save_path = Path(args.save_path).expanduser()
    elif args.wandb_run is None:
        raise SystemExit(
            'wandb_run must be specified if wandb_project is specified.')
    else:
        save_path = Path(args.save_path, args.wandb_project,
                         args.wandb_run).expanduser()
    save_path.mkdir(parents=True, exist_ok=True)

    args.hostname = socket.gethostname()
    args.slurm_jobid = os.getenv('SLURM_JOBID')
    with open(save_path / 'cmd_args.yaml', 'w', encoding='utf-8') as f:
        yaml.dump(vars(args), f)

    model_class = SartorrasEGNN if args.model == 'egnn' \
        else MultitaskSatorrasEGNN
    regression_task = 'multi_regression' if (
        args.multi_target_affinity or args.model_task == 'multi_regression') \
        else 'regression'

    dl_kwargs = dict(
        batch_size=args.batch_size, compact=args.compact, radius=args.radius,
        use_atomic_numbers=args.use_atomic_numbers, rot=False,
        polar_hydrogens=args.hydrogens, fname_suffix=args.input_suffix,
        edge_radius=args.edge_radius, estimate_bonds=args.estimate_bonds,
        prune=args.prune, extended_atom_types=args.extended_atom_types,
        include_strain_info=args.include_strain_info,
        num_workers=args.workers, worker_processes=args.worker_processes,
        device_crop=not args.host_crop)
    train_kwargs = dict(
        augmented_actives=args.augmented_actives,
        min_aug_angle=args.min_aug_angle,
        max_active_rms_distance=args.max_active_rmsd,
        min_inactive_rms_distance=args.min_inactive_rmsd,
        max_inactive_rms_distance=args.max_inactive_rmsd, mode='train',
        p_noise=args.p_noise, p_remove_entity=args.p_remove_entity)

    train_dl_pose = train_dl_affinity = None
    if args.model_task != 'regression':
        train_dl_pose = get_data_loader(
            args.train_data_root_pose, types_fname=args.train_types_pose,
            model_task='classification', **train_kwargs, **dl_kwargs)
    if args.model_task in ('both', 'regression'):
        train_dl_affinity = get_data_loader(
            args.train_data_root_affinity,
            types_fname=args.train_types_affinity, model_task=regression_task,
            **train_kwargs, **dl_kwargs)
    dim_input = (train_dl_pose or train_dl_affinity).dataset.feature_dim

    test_dl_pose = test_dl_affinity = None
    if 'regression' not in args.model_task and \
            args.test_data_root_pose is not None:
        test_dl_pose = get_data_loader(
            args.test_data_root_pose, types_fname=args.test_types_pose,
            mode='val', model_task='classification', **dl_kwargs)
    if args.model_task != 'classification' and \
            args.test_data_root_affinity is not None:
        test_dl_affinity = get_data_loader(
            args.test_data_root_affinity, types_fname=args.test_types_affinity,
            mode='val', model_task=regression_task, **dl_kwargs)

    # point_vs.py:189-221
    model_kwargs = {
        'act': args.activation, 'bn': True, 'cache': False, 'ds_frac': 1.0,
        'k': args.channels, 'num_layers': args.layers,
        'dropout': args.dropout, 'dim_input': dim_input,
        'dim_output': 3 if regression_task == 'multi_regression' else 1,
        'norm_coords': args.norm_coords, 'norm_feats': args.norm_feats,
        'thin_mlps': args.thin_mlps, 'edge_attention': args.egnn_attention,
        'attention': args.egnn_attention, 'tanh': args.egnn_tanh,
        'normalize': args.egnn_normalise, 'residual': args.egnn_residual,
        'edge_residual': args.egnn_edge_residual,
        'graphnorm': args.graphnorm, 'multi_fc': args.multi_fc,
        'update_coords': not args.static_coords,
        'node_final_act': args.lucid_node_final_act,
        'permutation_invariance': args.permutation_invariance,
        'attention_activation_fn': args.attention_activation_function,
        'node_attention': args.node_attention,
        'gated_residual': args.gated_residual, 'rezero': args.rezero,
        'model_task': args.model_task,
        'include_strain_info': args.include_strain_info,
        'final_softplus': args.final_softplus,
        'softmax_attention': args.softmax_attention,
    }
    if args.model_task == 'both':
        model_kwargs['model_task'] = 'classification'

    model = model_class(
        save_path, args.learning_rate, args.weight_decay,
        wandb_project=args.wandb_project, use_1cycle=args.use_1cycle,
        warm_restarts=args.warm_restarts,
        only_save_best_models=args.only_save_best_models,
        regression_loss=args.regression_loss, optimiser=args.optimiser,
        **model_kwargs)
    model.set_math(args.math)
    if not torch.cuda.is_available():
        from ._cabi import PvsError
        raise PvsError('training needs a CUDA device (no CPU fallback)')
    if args.load_weights is not None:
        model.load_weights(args.load_weights)

    if args.epochs_pose and train_dl_pose is not None:
        model.set_task('classification')
        model.train_model(
            train_dl_pose, epochs=args.epochs_pose, top1_on_end=args.top1,
            epoch_end_validation_set=test_dl_pose
            if args.val_on_epoch_end else None)
    if test_dl_pose is not None:
        model.set_task('classification')
        model.val(test_dl_pose, top1_on_end=args.top1)
    if args.epochs_affinity and train_dl_affinity is not None:
        model.set_task(regression_task)
        model.train_model(
            train_dl_affinity, epochs=args.epochs_affinity,
            top1_on_end=args.top1,
            epoch_end_validation_set=test_dl_affinity
            if args.val_on_epoch_end else None)
    if test_dl_affinity is not None:
        model.set_task(regression_task)
        model.val(test_dl_affinity, top1_on_end=args.top1)

    if args.end_flag:
        with open(save_path / '_FINISHED', 'w', encoding='utf-8') as f:
            f.write('')
    return model


if __name__ == '__main__':
    main()
