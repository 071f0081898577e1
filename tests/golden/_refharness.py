"""Harness that imports the UNMODIFIED reference from the checkout PIML_REFERENCE names, or from the verbatim copy
__graft_entry__.build() stages in git-ignored baseline/_ref/.

Used by tests/golden/make_golden.py to generate the committed golden vectors, by tests/test_gpu_dropin.py to run the
real reference objects behind piml_b200.patch, and by bench.py's reference_pytorch timing; the product never imports it.
Works around two reference defects without editing it (SURVEY.md Appendix B-1/B-2): data files are
loaded by absolute path, and `args` is built programmatically instead of through main.py.
"""
import argparse
import contextlib
import io
import os
import sys

_COPY = os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "baseline", "_ref")
REF_ROOT = os.environ.get("PIML_REFERENCE") or _COPY
REF_SRC = os.path.join(REF_ROOT, "src")
REF_DATA = os.path.join(REF_ROOT, "data")


def import_reference():
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    import data.data as DATA          # noqa
    import models.model as MODEL      # noqa
    import models.mlapm as MLAPM      # noqa
    import models.simulators as SIM   # noqa
    import utils.utils as UTILS       # noqa
    return DATA, MODEL, MLAPM, SIM, UTILS


def default_args(**over):
    """main.py:26-112 defaults as a Namespace (hot-path relevant subset + what BaseSimulator reads)."""
    a = argparse.Namespace(
        exp_name='golden', user_name='golden', seed=666, finetune_flag=False,
        model='pinnsf_m', device='cpu', gpus='3', learning_rate=0.002, batch_size=3, ft_batch_size=4,
        shuffle=False, num_workers=0, weight_decay=5e-4, epochs=2, dropout=0.5, n_embedding=10,
        hidden_size=32, activation='relu', patience=1, ft_patience=5,
        topk_ped=6, topk_obs=10, sight_angle_ped=90, sight_angle_obs=90,
        dist_threshold_ped=4, dist_threshold_obs=4,
        encoder_hidden_size=128, processor_hidden_size=128, decoder_hidden_size=64,
        encoder_hidden_layers=3, processor_hidden_layers=16, decoder_hidden_layers=2,
        add_noise_flag=False, add_noise_std=0.05, correction_hidden_layers=1,
        finetune_lr_decay=1, finetune_wd_aug=1, num_history_velocity=1, skip_frames=25,
        valid_steps=5, time_decay=1, training_mode='normal', res_hidden_layers=3, ft_lr_decay2=0.,
        save_configs=False, reg_weight=0., collision_threshold=0.5, collision_loss_weight=10,
        val_coll_weight=30, hard_collision_penalty=10, teacher_weight=0, collision_pred_weight=10,
        collision_focus_weight=10, new_collision_loss_flag=0, tags='', iter_flag=0,
        iter_model_name_suffix='', pinnsf_interaction='sim', dataset_name='ucy', true_label_weight=0,
        collision_loss_version='v0', model_name_suffix='goldenxx',
        ped_feature_dim=6, obs_feature_dim=6, self_feature_dim=7, time_unit=0.08)
    for k, v in over.items():
        setattr(a, k, v)
    return a


@contextlib.contextmanager
def quiet():
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        yield


def load_raw(relpath):
    DATA, *_ = import_reference()
    raw = DATA.RawData()
    with quiet():
        raw.load_trajectory_data(os.path.join(REF_DATA, relpath))
    return raw


def make_time_indexed(args, raw):
    DATA, *_ = import_reference()
    d = DATA.TimeIndexedPedData()
    with quiet():
        d.make_dataset(args, raw)
        d.set_dataset_info(d, raw, list(range(len(d))))
    return d


GC_CLIP = "GC_Dataset/GC_Dataset_ped1-12685_time1000-1060_interp9_xrange5-25_yrange15-35.npy"
SYN_CLIP = "synthetic_data/GC_Dataset_ped1-12685_time1560-1620_interp9_xrange5-25_yrange15-35_simulation.npy"
UCY_CLIP = "UCY_dataset/UCY_Dataset_time0-54_timeunit0.08.npy"
TOY_CLIP = "GC_Dataset/GC_Dataset_toy5.npy"


def available():
    return os.path.isdir(REF_SRC) and os.path.isdir(REF_DATA)
