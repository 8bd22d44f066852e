"""Command-line flags and the predictor factory -- host mirror of helpers/command_parser.py:22-127
restricted to the RNN method (the path this build accelerates).  Every flag of the reference's
parser is kept so existing command lines still parse; methods other than ``-m RNN`` raise NotImplementedError
(SURVEY.md §2 rows 9-10, 16-19).  ``-m RNN --clusters K`` builds the clustered RNN (command_parser.py:114-115)."""
import argparse

from ..neural_networks.recurrent_layers import get_recurrent_layers, recurrent_layers_command_parser
from ..neural_networks.rnn_cluster import RNNCluster
from ..neural_networks.rnn_margin import RNNMargin
from ..neural_networks.rnn_one_hot import RNNOneHot
from ..neural_networks.rnn_sampling import RNNSampling
from ..neural_networks.sequence_noise import get_sequence_noise, sequence_noise_command_parser
from ..neural_networks.target_selection import get_target_selection, target_selection_command_parser
from ..neural_networks.update_manager import get_update_manager, update_manager_command_parser
from .early_stopping import early_stopping_command_parser, get_early_stopper  # noqa: F401  (re-exported)

METHODS = ['RNN', 'SDA', 'BPRMF', 'FPMC', 'FISM', 'Fossil', 'LTM', 'UKNN', 'MM', 'POP']

# (flags, kwargs) in the reference's order (command_parser.py:35-76)
_PREDICTOR_FLAGS = [
    (('-m',), dict(dest='method', choices=METHODS, help='Method', default='RNN')),
    (('-b',), dict(dest='batch_size', help='Batch size', default=16, type=int)),
    (('-l',), dict(dest='learning_rate', help='Learning rate', default=0.01, type=float)),
    (('-r',), dict(dest='regularization', help='Regularization (positive for L2, negative for L1)', default=0., type=float)),
    (('-g',), dict(dest='gradient_clipping', help='Gradient clipping', default=100, type=int)),
    (('-H',), dict(dest='hidden', help='Number of hidden neurons (for LTM and BPRMF)', default=20, type=int)),
    (('-L',), dict(dest='layers', help='Layers (for SDA)', default="20", type=str)),
    (('--loss',), dict(help='Loss function, choose between TOP1, BPR and Blackout (Sampling), or hinge, logit and logsig '
                            '(multi-targets), or CCE (Categorical cross-entropy)', default='CCE', type=str)),
    (('--sampling',), dict(help='Number of sample for the computation of the loss in RNNSampling', default=32.0, type=float)),
    (('--sampling_bias',), dict(help='Sampling bias. 0. means uniform sampling, 1. means proportional to the item frequency', default=0., type=float)),
    (('--db',), dict(dest='diversity_bias', help='Diversity bias (for RNN with CCE, TOP1, BPR or Blackout loss)', default=0.0, type=float)),
    (('--in_do',), dict(dest='input_dropout', help='Input dropout (for SDA)', default=0.2, type=float)),
    (('--do',), dict(dest='dropout', help='Dropout (for SDA)', default=0.5, type=float)),
    (('--rf',), dict(help='Use rating features.', action='store_true')),
    (('--mf',), dict(help='Use movie features.', action='store_true')),
    (('--uf',), dict(help='Use users features.', action='store_true')),
    (('--ns',), dict(help='Neighborhood size (for UKNN).', default=80, type=int)),
    (('--pb',), dict(help='Popularity based (for RNNMargin).', action='store_true')),
    (('--balance',), dict(help='Balance between false positive and false negative error (for RNNMargin).', default=1., type=float)),
    (('--min_access',), dict(help='Estimation of minimum access probability (for RNNMargin).', default=0.05, type=float)),
    (('--k_cf',), dict(help='Number of features for the CF factorization (for FPMC).', default=32, type=int)),
    (('--k_mc',), dict(help='Number of features for the MC factorization (for FPMC).', default=32, type=int)),
    (('--init_sigma',), dict(help='Sigma of the gaussian initialization (for FPMC)', default=1, type=float)),
    (('--fpmc_bias',), dict(help='Sampling bias (for FPMC)', default=100., type=float)),
    (('--no_adaptive_sampling',), dict(help='No adaptive sampling (for FPMC)', action='store_true')),
    (('--cooling',), dict(help='Simulated annealing', default=1., type=float)),
    (('--ltm_damping',), dict(help='Temporal damping (for LTM)', default=0.8, type=float)),
    (('--ltm_window',), dict(help='Window for word2vec (for LTM)', default=5, type=int)),
    (('--ltm_no_trajectory',), dict(help='Do not use users trajectory in LTM, just use word2vec', action='store_true')),
    (('--max_length',), dict(help='Maximum length of sequences during training (for RNNs)', default=30, type=int)),
    (('--repeated_interactions',), dict(help='The model can recommend items with which the user already interacted', action='store_true')),
    (('--fism_alpha',), dict(help='Alpha parameter in FISM', default=0.2, type=float)),
    (('--fossil_order',), dict(help='Order of the markov chains in Fossil', default=1, type=int)),
    (('--c_sampling',), dict(help='Number of sample for the clustering loss.', default=-1, type=int)),
    (('--ignore_clusters',), dict(help="Don't use clusters during test.", action='store_true')),
    (('--clusters',), dict(help='Number of clusters. If unset, no clustering is used', default=-1, type=int)),
    (('--init_scale',), dict(help='Initial scale of the softmax and sigmoid in the clustering method.', default=1., type=float)),
    (('--scale_growing_rate',), dict(help='Rate of the geometric growth of the sigmoid/softmax scale in the clustering method.', default=1., type=float)),
    (('--max_scale',), dict(help='Max scale of the softmax and sigmoid in the clustering method.', default=50, type=float)),
    (('--csn',), dict(help='Cluster selection noise', default=0., type=float)),
    (('--cluster_type',), dict(choices=['softmax', 'mix', 'sigmoid'], help='Type of clusters.', default='mix', type=str)),
]

# flags added by this build (they do not change the meaning of any reference flag)
_B200_FLAGS = [
    (('--device',), dict(help='CUDA ordinal of this rank (default: LOCAL_RANK or 0)', default=None, type=int)),
    (('--seed',), dict(help='Seed of the python / numpy RNGs that drive batch construction', default=None, type=int)),
    (('--prefetch',), dict(help='Assemble this many mini-batches ahead in a background thread (the reference\'s '
                                'disabled threaded_generator); 0 = off', default=0, type=int)),
]


def command_parser(*sub_command_parser, argv=None):
    """sub_command_parser: callables that add their arguments to the parser (command_parser.py:22-32)."""
    parser = argparse.ArgumentParser()
    for scp in sub_command_parser:
        scp(parser)
    return parser.parse_args(argv)


def predictor_command_parser(parser):
    for flags, kw in _PREDICTOR_FLAGS + _B200_FLAGS:
        parser.add_argument(*flags, **kw)
    update_manager_command_parser(parser)
    recurrent_layers_command_parser(parser)
    sequence_noise_command_parser(parser)
    target_selection_command_parser(parser)


def get_predictor(args, **dist):
    """Build the predictor named by the flags (command_parser.py:84-125).  `dist` carries the
    data-parallel placement (device, n_ranks, rank, nccl_id)."""
    if args.method != 'RNN':
        raise NotImplementedError("-m %s: only the RNN method is on the B200 hot path (SURVEY.md §8)" % args.method)
    common = dict(interactions_are_unique=(not args.repeated_interactions), max_length=args.max_length,
                  updater=get_update_manager(args), target_selection=get_target_selection(args),
                  sequence_noise=get_sequence_noise(args), recurrent_layer=get_recurrent_layers(args),
                  use_ratings_features=args.rf, use_movies_features=args.mf, use_users_features=args.uf,
                  batch_size=args.batch_size, prefetch_batches=getattr(args, 'prefetch', 0))
    common.update(dist)
    if args.clusters > 0:       # checked before the loss dispatch, as in the reference
        return RNNCluster(cluster_selection_noise=args.csn, loss=args.loss, predict_with_clusters=(not args.ignore_clusters),
                          sampling_bias=args.sampling_bias, sampling=args.sampling, cluster_sampling=args.c_sampling,
                          init_scale=args.init_scale, scale_growing_rate=args.scale_growing_rate,
                          max_scale=args.max_scale, n_clusters=args.clusters, cluster_type=args.cluster_type, **common)
    if args.loss == 'CCE':
        return RNNOneHot(diversity_bias=args.diversity_bias, regularization=args.regularization, **common)
    if args.loss in ('hinge', 'logit', 'logsig'):
        return RNNMargin(loss_function=args.loss, balance=args.balance, popularity_based=args.pb,
                         min_access=args.min_access, n_targets=args.n_targets, **common)
    if args.loss in ('BPR', 'TOP1', 'Blackout'):
        return RNNSampling(loss_function=args.loss, diversity_bias=args.diversity_bias, sampling=args.sampling,
                           sampling_bias=args.sampling_bias, **common)
    raise ValueError('Unknown loss for the RNN model')
