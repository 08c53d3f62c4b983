#!/usr/bin/env python
"""Drop-in for the reference's isprs_dilated_random.py on the B200-native hot path (libdrs.so).

Same positional command line (isprs:1987-2042):
  input_path output_path currentModelPath trainingInstances testing_instances learningRate weight_decay batch_size niter
  reference_crop_size reference_stride_crop net_type distribution_type probValues update_type process
process: training | validate_test | generate_final_maps.   Multi-GPU: launch under torchrun (one process per GPU).
DRS_NUM_SCALES=N (N > 1): validate_test evaluates at the N best patch sizes (multi-scale, isprs:1347-1474).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import drs_b200  # noqa: E402,F401
from drs_b200 import cli, host, loops  # noqa: E402
from drs_b200.host import BatchColors  # noqa: E402

NUM_CLASSES = 6
NET_TYPES = ('dilated_icpr_original', 'dilated_grsl', 'dilated_icpr_rate6_densely', 'dilated8_grsl', 'dilated_grsl_rate8',
             'dilated_icpr_rate6', 'dilated_icpr_rate6_small', 'dilated_icpr_rate6_nodilation', 'dilated_icpr_rate6_SE',
             'dilated_icpr_rate6_squeeze')


def main():
    list_params = ['input_path', 'output_path(for model, images, etc)', 'currentModelPath', 'trainingInstances',
                   'testing_instances', 'learningRate', 'weight_decay', 'batch_size', 'niter', 'reference_crop_size',
                   'reference_stride_crop', 'net_type[' + '|'.join(NET_TYPES) + ']',
                   'distribution_type[single_fixed|multi_fixed|uniform|multinomial]', 'probValues', 'update_type [acc|loss]',
                   'process [training|validate_test|generate_final_maps]']
    if len(sys.argv) < len(list_params) + 1:
        sys.exit('Usage: ' + sys.argv[0] + ' ' + ' '.join(list_params))
    cli.print_params(list_params)
    a = sys.argv
    input_path, output_path, former_model_path = a[1], a[2], a[3]
    dataset = input_path[:-1].split("/")[-1].lower()
    training_instances, testing_instances = a[4].split(','), a[5].split(',')
    lr_initial, weight_decay, batch_size, niter = float(a[6]), float(a[7]), int(a[8]), int(a[9])
    reference_crop_size, reference_stride_crop = int(a[10]), int(a[11])
    net_type, distribution_type = a[12], a[13]
    values = [int(i) for i in a[14].split(',')]
    update_type, process = a[15], a[16]
    # the reference hard-codes num_scales=1, eval_type='single_scale' (isprs:2128-2131); DRS_NUM_SCALES=N > 1 turns
    # validate_test into its multi-scale evaluation over the N best patch sizes of the saved score arrays
    num_scales = int(os.environ.get("DRS_NUM_SCALES", "1"))
    display_step = 50
    if dataset == 'vaihingen':
        resample_batch = 20
    elif dataset == 'postdam':
        resample_batch = 10
    else:
        print("Error! No dataset identified: ", dataset)
        resample_batch = 20
    if net_type not in NET_TYPES:
        print(BatchColors.FAIL + 'Error! Net type not identified: ' + net_type + BatchColors.ENDC)
        return
    patch_acc_loss, patch_occur, patch_chosen_values = host.init_score_arrays(distribution_type, values)
    probs = host.define_multinomial_probs(values) if distribution_type == 'multinomial' else None

    print(BatchColors.WARNING + 'Reading images...' + BatchColors.ENDC)
    training_data, training_labels = cli.load_npy_scenes(input_path, training_instances)
    testing_data, testing_labels = cli.load_npy_scenes(input_path, testing_instances)
    tag = os.getcwd() + '/dataset_' + dataset + '_crop_' + str(reference_crop_size) + '_stride_' + str(reference_stride_crop)
    training_class_distribution = testing_class_distribution = None
    if process == 'training':
        print(BatchColors.WARNING + 'Creating TRAINING class distribution...' + BatchColors.ENDC)
        training_class_distribution = host.create_distributions_over_classes(training_labels, reference_crop_size,
                                                                             reference_stride_crop, NUM_CLASSES)
        print(BatchColors.WARNING + 'Creating TESTING class distribution...' + BatchColors.ENDC)
        testing_class_distribution = host.create_distributions_over_classes(testing_labels, reference_crop_size,
                                                                            reference_stride_crop, NUM_CLASSES)
    def _rotation():
        if os.path.isfile(tag + '_rotation.npy'):
            r = np.load(tag + '_rotation.npy', allow_pickle=True)
            print(BatchColors.OKGREEN + 'Loaded training instance rotations' + BatchColors.ENDC)
            return r
        if training_class_distribution is None:
            return None
        r = host.create_rotation_distribution(training_class_distribution)
        cli.save_atomic(tag + '_rotation.npy', np.asarray(r, dtype=object), allow_pickle=True)
        print(BatchColors.OKGREEN + 'Created training instance rotations' + BatchColors.ENDC)
        return r

    def _mean_std():
        if os.path.isfile(tag + '_mean.npy') and os.path.isfile(tag + '_std.npy'):
            print(BatchColors.OKGREEN + 'Loaded Mean/Std from training instances' + BatchColors.ENDC)
            return np.load(tag + '_mean.npy'), np.load(tag + '_std.npy')
        distr = training_class_distribution
        if distr is None:
            distr = host.create_distributions_over_classes(training_labels, reference_crop_size, reference_stride_crop, NUM_CLASSES,
                                                           verbose=False)
        m, sd = host.dynamically_calculate_mean_and_std(training_data, distr, crop_size=25)
        cli.save_atomic(tag + '_std.npy', sd)
        cli.save_atomic(tag + '_mean.npy', m)
        print(BatchColors.OKGREEN + 'Created Mean/Std from training instances' + BatchColors.ENDC)
        return m, sd

    # under torchrun rank 0 creates the cache files, the other ranks wait and load them (no half-written reads, one table)
    training_rotation_distribution = cli.rank0_first(_rotation)
    mean_full, std_full = cli.rank0_first(_mean_std)

    channels = training_data[0].shape[-1]
    if process == 'training':
        be = cli.make_backend(net_type, channels, NUM_CLASSES, weight_decay, lr_initial, 0.5, list(training_data) + list(testing_data),
                              list(training_labels) + list(testing_labels), mean_full, std_full, True, True)
        loops.isprs_train(be, training_data, training_labels, training_class_distribution, training_rotation_distribution,
                          testing_data, testing_labels, testing_class_distribution, testing_instances, batch_size, niter,
                          update_type, distribution_type, values, patch_acc_loss, patch_occur, patch_chosen_values, probs,
                          resample_batch, output_path, display_step, dataset, former_model_path, NUM_CLASSES)
    elif process in ('validate_test', 'generate_final_maps'):
        be = cli.make_backend(net_type, channels, NUM_CLASSES, weight_decay, lr_initial, 0.5, list(testing_data),
                              list(testing_labels), mean_full, std_full, True, False)
        for model in former_model_path.split(","):
            be.restore(model)
            step = int(model.split('-')[-1]) if '-' in model else 0
            crop_size = int(values[0])
            if distribution_type in loops.DYNAMIC:       # isprs:1519-1545: best size from the saved score arrays
                pal = np.load(output_path + 'patch_acc_loss_step_' + str(step) + '.npy')
                occ = np.load(output_path + 'patch_occur_step_' + str(step) + '.npy')
                crop_size = host.select_best_patch_size(distribution_type, values, pal, occ, update_type, debug=True)
            if process == 'validate_test' and num_scales > 1:    # eval_type='multi_scale' (isprs:1347-1474)
                loops.isprs_validate_test_multiscale(be, testing_data, testing_labels, testing_instances, batch_size, step,
                                                     distribution_type, values, update_type, num_scales, False, output_path,
                                                     NUM_CLASSES)
            elif process == 'validate_test':
                loops.isprs_validate_test(be, testing_data, testing_labels, testing_instances, batch_size, crop_size, step,
                                          NUM_CLASSES)
            else:
                loops.isprs_generate_final_maps(be, testing_data, testing_instances, batch_size, crop_size, output_path, dataset)
    else:
        print(BatchColors.FAIL + "Process " + process + "not found!" + BatchColors.ENDC)


if __name__ == "__main__":
    main()
