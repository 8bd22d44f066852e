#!/usr/bin/env python
"""test.py -- same command line as the reference's test.py:120-161, RNN methods only: evaluates the
saved models of a configuration on the test set (first half of each sequence as input, second half
as goal, test.py:55-69)."""
import glob
import os
import re
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from sbr_b200.helpers import command_parser as parse   # noqa: E402
from sbr_b200.helpers import evaluation                 # noqa: E402
from sbr_b200.helpers.data_handling import DataHandler  # noqa: E402


def get_file_name(predictor, args):
    return args.dir + re.sub('_ml' + str(args.max_length), '_ml' + str(args.training_max_length),
                             predictor._get_model_filename(args.number_of_batches))


def find_models(predictor, dataset, args):
    file = dataset.dirname + "models/" + get_file_name(predictor, args)
    print(file)
    if args.number_of_batches == "*":
        file = np.array(glob.glob(file))
    return file


def save_file_name(predictor, dataset, args):
    if not args.save:
        return None
    return re.sub(r'_ne\*_', '_', dataset.dirname + 'results/' + get_file_name(predictor, args))


def run_tests(predictor, model_file, dataset, args, get_full_recommendation_list=False, k=10):
    predictor.load(model_file)
    evaluator = evaluation.Evaluator(dataset, k=k)
    if get_full_recommendation_list:
        k = min(dataset.n_items, 64)
    start = time.process_time()
    nb_of_dp = []
    for sequence, user_id in dataset.test_set(epochs=1):
        num_viewed = int(len(sequence) / 2)
        viewed = sequence[:num_viewed]
        goal = [int(i[0]) for i in sequence[num_viewed:]]
        if len(goal) == 0:
            raise ValueError
        if getattr(args, 'clusters', -1) > 0:     # the clustered RNN also returns how many items it scored (test.py:61-63)
            recommendations, n = predictor.top_k_recommendations(viewed, user_id=user_id, k=k)
            nb_of_dp.append(n)
        else:
            recommendations = predictor.top_k_recommendations(viewed, user_id=user_id, k=k)
        evaluator.add_instance(goal, recommendations)
    print('Timer: ', time.process_time() - start)
    evaluator.nb_of_dp = np.mean(nb_of_dp) if nb_of_dp else dataset.n_items
    return evaluator


def print_results(ev, metrics, file=None, n_batches=None, print_full_rank_comparison=False):
    for m in metrics:
        if m not in ev.metrics:
            raise ValueError('Unkown metric: ' + m)
        print(m + '@' + str(ev.k) + ': ', ev.metrics[m]())
    values = "\t".join(map(str, [ev.metrics[m]() for m in metrics]))
    if file is not None:
        if not os.path.exists(os.path.dirname(file)):
            os.makedirs(os.path.dirname(file))
        with open(file, "a") as f:
            f.write(str(n_batches) + values + "\n")
    else:
        print("-\t" + values, file=sys.stderr)
    if print_full_rank_comparison and file is not None:
        with open(file + "_full_rank", "a") as f:
            for data in ev.get_rank_comparison():
                f.write("\t".join(map(str, data)) + "\n")


def extract_number_of_epochs(filename):
    return float(re.search(r'_ne([0-9]+(\.[0-9]+)?)_', filename).group(1))


def get_last_tested_batch(filename):
    if filename is not None and os.path.isfile(filename):
        line = None
        with open(filename) as f:
            for line in f:
                pass
        return float(line.split()[0]) if line else 0
    return 0


def test_command_parser(parser):
    parser.add_argument('-d', dest='dataset', help='Directory name of the dataset.', default='', type=str)
    parser.add_argument('-i', dest='number_of_batches', help='Number of epochs, if not set it will compare all the '
                        'available models', default=-1, type=int)
    parser.add_argument('-k', dest='nb_of_predictions', help='Number of predictions to make. It is the "k" in '
                        '"prec@k", "rec@k", etc.', default=10, type=int)
    parser.add_argument('--metrics', help='List of metrics to compute, comma separated',
                        default='sps,recall,item_coverage,user_coverage,blockbuster_share', type=str)
    parser.add_argument('--save', help='Save results to a file', action='store_true')
    parser.add_argument('--dir', help='Model directory.', default="", type=str)
    parser.add_argument('--save_rank', help='Save the full comparison of goal and prediction ranking.', action='store_true')


def main(argv=None):
    args = parse.command_parser(parse.predictor_command_parser, test_command_parser, argv=argv)
    args.training_max_length = args.max_length
    if args.number_of_batches == -1:
        args.number_of_batches = "*"
    dataset = DataHandler(dirname=args.dataset)
    predictor = parse.get_predictor(args, device=args.device if args.device is not None else 0)
    predictor.set_dataset(dataset)
    predictor.prepare_model(dataset)
    file = find_models(predictor, dataset, args)
    metrics = args.metrics.split(',')
    results = []
    if args.number_of_batches == "*":
        output_file = save_file_name(predictor, dataset, args)
        last_tested_batch = get_last_tested_batch(output_file)
        batches = np.array([extract_number_of_epochs(f) for f in file])
        order = np.argsort(batches)
        for i, idx in enumerate(order):
            if batches[idx] > last_tested_batch:
                ev = run_tests(predictor, file[idx], dataset, args, get_full_recommendation_list=args.save_rank,
                               k=args.nb_of_predictions)
                print('-------------------')
                print('(', i + 1, '/', len(file), ') results on ' + file[idx])
                print_results(ev, metrics, file=output_file, n_batches=batches[idx],
                              print_full_rank_comparison=args.save_rank)
                results.append(ev)
    else:
        ev = run_tests(predictor, file, dataset, args, get_full_recommendation_list=args.save_rank,
                       k=args.nb_of_predictions)
        print_results(ev, metrics, file=save_file_name(predictor, dataset, args),
                      print_full_rank_comparison=args.save_rank)
        results.append(ev)
    return results


if __name__ == '__main__':
    main()
