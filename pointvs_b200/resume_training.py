"""Resume training of a run directory, mirror of
/root/reference/point_vs/resume_training.py (:14-221).

    python -m pointvs_b200.resume_training <base_path> [-ep N] [-ea N]

Reads `cmd_args.yaml` / `model_kwargs.yaml` and the latest checkpoint through
`load_model(base_path, init_path=True)`, rebuilds the data loaders from the
recorded flags (both the current `*_pose` / `*_affinity` layout and the older
single `epochs` / `train_data_root` layout) and runs the remaining epochs:
`train_model` starts at the epoch stored in the checkpoint.
"""
import argparse
from pathlib import Path

from .base import check_trainable_width
from .data import get_data_loader
from .load_model import load_model


def _loaders(cmd, root_train, types_train, root_test, types_test, task):
    if root_train is None:
        return None, None
    common = dict(
        batch_size=cmd['batch_size'], compact=cmd['compact'],
        radius=cmd['radius'], use_atomic_numbers=cmd['use_atomic_numbers'],
        rot=False, polar_hydrogens=cmd['hydrogens'],
        fname_suffix=cmd['input_suffix'], edge_radius=cmd['edge_radius'],
        estimate_bonds=cmd.get('estimate_bonds', False),
        prune=cmd.get('prune', False),
        extended_atom_types=cmd.get('extended_atom_types', False),
        include_strain_info=cmd.get('include_strain_info', False),
        model_task=task, num_workers=cmd.get('workers', 4),
        worker_processes=cmd.get('worker_processes', False),
        device_crop=not cmd.get('host_crop', False))
    train_dl = get_data_loader(
        root_train, types_fname=types_train, mode='train',
        augmented_actives=cmd['augmented_actives'],
        min_aug_angle=cmd['min_aug_angle'],
        max_active_rms_distance=cmd['max_active_rmsd'],
        min_inactive_rms_distance=cmd['min_inactive_rmsd'],
        max_inactive_rms_distance=cmd.get('max_inactive_rmsd', None),
        p_remove_entity=cmd.get('p_remove_entity', 0),
        p_noise=cmd.get('p_noise', 0), **common)
    test_dl = None
    if root_test is not None:
        test_dl = get_data_loader(root_test, types_fname=types_test,
                                  mode='val', **common)
    return train_dl, test_dl


def main(argv=None):
    parser = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    parser.add_argument('base_path', type=str)
    parser.add_argument('--epochs_pose', '-ep', type=int, default=-1)
    parser.add_argument('--epochs_affinity', '-ea', type=int, default=-1)
    args = parser.parse_args(argv)
    base_path = Path(args.base_path).expanduser().resolve()
    _, _, _, cmd = load_model(base_path, fetch_args_only=True)
    check_trainable_width(cmd.get('channels', 0))
    _, model, _, cmd = load_model(base_path, init_path=True)
    ea, ep = args.epochs_affinity, args.epochs_pose

    pose = dict(root_train=None, types_train=None, root_test=None,
                types_test=None)
    affinity = dict(pose)
    if cmd.get('epochs', False):           # runs recorded before the split
        regression_task = 'multi_regression' if cmd.get(
            'model_task', 'regression') == 'multi_regression' else 'regression'
        slot = pose if cmd.get('model_task', 'classification') == \
            'classification' else affinity
        slot.update(root_train=cmd['train_data_root'],
                    types_train=cmd['train_types'],
                    root_test=cmd['test_data_root'],
                    types_test=cmd['test_types'])
        epochs_classi = (cmd['epochs'] if ep == -1 else ep) \
            if slot is pose else 0
        epochs_affini = (cmd['epochs'] if ea == -1 else ea) \
            if slot is affinity else 0
    else:
        regression_task = 'multi_regression' \
            if cmd['multi_target_affinity'] else 'regression'
        epochs_affini = cmd['epochs_affinity'] if ea == -1 else ea
        epochs_classi = cmd['epochs_pose'] if ep == -1 else ep
        affinity.update(root_train=cmd['train_data_root_affinity'],
                        types_train=cmd['train_types_affinity'],
                        root_test=cmd['test_data_root_affinity'],
                        types_test=cmd['test_types_affinity'])
        pose.update(root_train=cmd['train_data_root_pose'],
                    types_train=cmd['train_types_pose'],
                    root_test=cmd['test_data_root_pose'],
                    types_test=cmd['test_types_pose'])

    pose_train_dl, pose_test_dl = _loaders(cmd, task='classification', **pose)
    aff_train_dl, aff_test_dl = _loaders(cmd, task=regression_task, **affinity)
    model.set_math(cmd.get('math', 'fp32'))
    val_on_epoch_end = cmd.get('val_on_epoch_end', False)
    top1 = cmd.get('top1', False)
    if pose_train_dl is not None:
        model.train()
        model.set_task('classification')
        model.train_model(
            pose_train_dl, epochs=epochs_classi, top1_on_end=top1,
            epoch_end_validation_set=pose_test_dl if val_on_epoch_end else None)
    if pose_test_dl is not None:
        model.eval()
        model.set_task('classification')
        model.val(pose_test_dl, top1_on_end=top1)
    if aff_train_dl is not None:
        model.train()
        model.set_task(regression_task)
        model.train_model(
            aff_train_dl, epochs=epochs_affini, top1_on_end=top1,
            epoch_end_validation_set=aff_test_dl if val_on_epoch_end else None)
    if aff_test_dl is not None:
        model.eval()
        model.set_task(regression_task)
        model.val(aff_test_dl, top1_on_end=top1)
    return model


if __name__ == '__main__':
    main()
