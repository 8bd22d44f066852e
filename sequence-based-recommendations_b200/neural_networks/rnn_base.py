"""RNNBase -- Python 3 host mirror of the reference's neural_networks/rnn_base.py:58-642.

Same public API (``prepare_model``, ``train``, ``top_k_recommendations``, ``save`` / ``load`` /
``load_last``, ``_get_model_filename``) and the same three callables the reference obtains from
``theano.function`` (rnn_base.py:175-213):

    self.train_function(*batch)         -> cost      (in-place update of parameters + optimizer state)
    self.test_function(batch, k=10)     -> ids[k]
    self.predict_function(X, mask)      -> scores[B, n_items]

Here they are thin closures over one ``sbr_b200._capi.Engine`` handle, i.e. over the C ABI of
``libsbr_b200.so``; nothing is computed on the host and there is no CPU fallback.  Data
parallelism: one process per GPU, every rank builds the same global mini-batch (same seeds) and
steps on its own slice of rows; the library all-reduces the flat gradient buffer once per step.
"""
import glob
import os
import pickle
import queue
import random
import re
import sys
import threading
from time import time

import numpy as np

from .. import _capi
from ..helpers import evaluation
from .recurrent_layers import RecurrentLayers
from .sequence_noise import SequenceNoise
from .target_selection import SelectTargets
from .update_manager import Adagrad

MAX_LENGTH = 200
BATCH_SIZE = 10


class threaded_generator(object):
    """Run `generator` in a background thread, `num_cached` items ahead of the consumer.

    The reference defines a helper of this name (rnn_base.py:34-56) and leaves its only call commented out
    (rnn_base.py:273-274).  Here it pays: a train step returns as soon as its cost is known and spends its time
    inside the C library with the GIL released, so the ~0.5 ms of Python that assembles the next mini-batch
    (`_gen_mini_batch` + `_prepare_input`) overlaps the device work instead of adding to every step.

    Iteration order and content are exactly those of `generator`.  An exception raised by the producer is re-raised
    in the consumer at the position where it happened; `close()` (also called when the consumer is garbage
    collected) stops the producer.  The producer and the consumer share the global `random` / `numpy.random`
    state, so the consumer must not draw from them while the producer runs if a seeded run (or a multi-rank run,
    where every rank has to build the same global batches) is to stay reproducible.  The train loop does not; the
    periodic validation does not either: test batches of RNNSampling carry a constant sample vector (the test
    function ignores it) instead of fresh draws, and `--rand_test_target` is refused together with prefetching."""

    _END = object()

    def __init__(self, generator, num_cached=50):
        self._queue = queue.Queue(maxsize=max(1, int(num_cached)))
        self._stop = threading.Event()
        self._done = False
        self._thread = threading.Thread(target=self._produce, args=(generator,), daemon=True)
        self._thread.start()

    def _put(self, item):
        while not self._stop.is_set():
            try:
                self._queue.put(item, timeout=0.05)
                return True
            except queue.Full:
                continue
        return False

    def _produce(self, generator):
        try:
            for item in generator:
                if not self._put((None, item)):
                    return
            self._put((None, self._END))
        except BaseException as e:      # hand it to the consumer
            self._put((e, None))

    def __iter__(self):
        return self

    def __next__(self):
        if self._done:
            raise StopIteration
        err, item = self._queue.get()
        if err is not None:
            self._done = True
            raise err
        if item is self._END:
            self._done = True
            raise StopIteration
        return item

    def close(self):
        self._stop.set()
        self._done = True

    def __del__(self):
        self.close()


class CompactBatch(object):
    """A training mini-batch in the device-assembly form (SURVEY.md §8 f1): one (sequence index, start, length)
    triple per row into the sequences uploaded once with Engine.dataset_upload, plus the per-row targets.  The
    padded X / mask of the reference batch (rnn_one_hot.py:90-101) are built on the device from it."""
    __slots__ = ("seq", "start", "length", "Y", "pop")

    def __init__(self, seq, start, length, Y, pop):
        self.seq, self.start, self.length, self.Y, self.pop = seq, start, length, Y, pop

    def __len__(self):
        return len(self.seq)


class RNNBase(object):
    def __init__(self, sequence_noise=None, recurrent_layer=None, updater=None, target_selection=None,
                 interactions_are_unique=True, other_features=None, use_ratings_features=True, movies_features=None,
                 use_movies_features=True, users_features=None, use_users_features=True, max_length=MAX_LENGTH,
                 batch_size=BATCH_SIZE, device=0, n_ranks=1, rank=0, nccl_id=None, prefetch_batches=0, init_seed=None, control=None, device_batches=True):
        self.sequence_noise = sequence_noise if sequence_noise is not None else SequenceNoise()
        self.recurrent_layer = recurrent_layer if recurrent_layer is not None else RecurrentLayers()
        self.updater = updater if updater is not None else Adagrad()
        self.target_selection = target_selection if target_selection is not None else SelectTargets()
        self.interactions_are_unique = interactions_are_unique
        self.use_ratings_features = use_ratings_features
        self.use_movies_features = use_movies_features
        self.use_users_features = use_users_features
        self.max_length = max_length
        self.batch_size = batch_size
        self.device, self.n_ranks, self.rank, self.nccl_id = device, n_ranks, rank, nccl_id
        self.prefetch_batches = int(prefetch_batches)   # > 0: assemble mini-batches in a background thread
        # seed of the parameter initialisation.  The reference draws from the (unseeded) global numpy RNG through
        # lasagne.random.get_rng(); data-parallel replicas must start identical, so with several ranks the default
        # is a fixed seed, with one rank the global numpy RNG like the reference.
        self.init_seed = init_seed
        # multi-rank control plane (helpers/rendezvous.Control) or None; used to make wall-clock decisions collective
        self.control = control
        # build the padded mini-batch tensors on the device from (sequence, start, length) triples when the model
        # supports it (RNNOneHot; no sequence noise: the uploaded sequences must be the ones the rows are cut from)
        self.device_batches = bool(device_batches)
        self._uploaded = None       # user id -> index of its sequence in the uploaded CSR
        if batch_size % n_ranks != 0:
            raise ValueError("batch_size (%d) must be a multiple of the number of ranks (%d)" % (batch_size, n_ranks))
        self.local_batch = batch_size // n_ranks
        self._input_type = 'int32'
        self.name = "RNN base"
        self.metrics = {'recall': {'direction': 1}, 'sps': {'direction': 1}, 'user_coverage': {'direction': 1},
                        'item_coverage': {'direction': 1}, 'ndcg': {'direction': 1},
                        'blockbuster_share': {'direction': -1}}
        self.engine = None

    # ------------------------------------------------------------------ model construction
    loss_name = "CCE"

    def prepare_model(self, dataset):
        """Must be called before train, load or top_k_recommendations (rnn_base.py:106-109)."""
        self._prepare_networks(dataset.n_items)

    def _engine_extra_kwargs(self):
        return {}

    def _prepare_networks(self, n_items):
        """Replaces the symbolic graph construction of the subclasses' _prepare_networks
        (rnn_one_hot.py:37-77, rnn_sampling.py:93-137, rnn_margin.py:70-109): one sbr_create."""
        if self.use_movies_features or self.use_users_features:
            raise NotImplementedError("--mf / --uf need external feature tables that the reference defaults to None "
                                      "(rnn_base.py:27-29); they are outside the B200 hot path")
        self.n_items = n_items
        kw = dict(n_items=n_items, loss=self.loss_name, max_length=self.max_length, batch_size=self.local_batch,
                  n_extra_ids=self._n_optional_features(), ids_per_step=self._input_size(), device=self.device,
                  n_ranks=self.n_ranks, rank=self.rank, nccl_id=self.nccl_id, global_batch=self.batch_size)
        kw.update(self.recurrent_layer.engine_kwargs())
        kw.update(self.updater.engine_kwargs())
        kw.update(self._engine_extra_kwargs())
        self.engine = _capi.Engine(**kw)
        self._init_parameters()

    last_layer_init = 1.0   # GlorotUniform gain of the output layer (RNNSampling overrides it, rnn_sampling.py:131)

    def _init_parameters(self):
        """Lasagne's initialisers for a freshly built network, in add_param order (the library allocates the
        parameter arena zeroed): Gate W_in / W_hid / W_cell ~ Normal(std 0.1), b = 0 (lasagne Gate defaults used at
        sparse_lstm.py:156-159,590-593,960-961); learned cell_init / hid_init = 0; EmbeddingLayer.W ~ Normal(std
        0.01) (recurrent_layers.py:47); Dense / Blackout W ~ GlorotUniform(gain) (rnn_one_hot.py:65,
        rnn_sampling.py:131, rnn_margin.py:103), b = 0."""
        rng = self._init_rng()
        vals = [self._initial_value(rng, name, shape) for name, shape in self.engine.param_infos()]
        self.engine.set_all_param_values(vals)

    def _init_rng(self):
        if self.init_seed is None:
            return np.random.RandomState(20160901) if self.n_ranks > 1 else np.random
        return np.random.RandomState(self.init_seed)

    def _initial_value(self, rng, name, shape):
        leaf = name.split(".")[1]
        if name == "emb.W":
            v = rng.normal(0.0, 0.01, size=shape)
        elif name == "out.W":
            a = float(self.last_layer_init) * np.sqrt(6.0 / (shape[0] + shape[1]))
            v = rng.uniform(-a, a, size=shape)
        elif leaf in ("W_in_to_hid", "W_hid_to_hid"):
            # Vanilla layers with a dense input are lasagne.layers.RecurrentLayer (recurrent_layers.py:98-99),
            # whose weights default to lasagne.init.Uniform() = U(-0.01, 0.01)
            v = rng.uniform(-0.01, 0.01, size=shape)
        elif leaf.startswith("W_"):
            v = rng.normal(0.0, 0.1, size=shape)
        else:
            v = np.zeros(shape, dtype=np.float32)
        return np.asarray(v, dtype=np.float32)     # drawn in float64 like Lasagne, stored as floatX

    def _common_filename(self, epochs):
        """Common part of the checkpoint filename across sub classes (rnn_base.py:111-130)."""
        parts = ["ml" + str(self.max_length), "bs" + str(self.batch_size), "ne" + str(epochs),
                 self.recurrent_layer.name, self.updater.name, self.target_selection.name]
        filename = "_".join(parts)
        if self.sequence_noise.name != "":
            filename += "_" + self.sequence_noise.name
        if not self.interactions_are_unique:
            filename += "_ri"
        if not (self.use_ratings_features or self.use_movies_features or self.use_users_features):
            filename += "_nf"
        if self.use_ratings_features:
            filename += "_rf"
        if self.use_movies_features:
            filename += "_mf"
        if self.use_users_features:
            filename += "_uf"
        return filename

    def _get_model_filename(self, iterations):
        raise NotImplementedError

    # ------------------------------------------------------------------ features (rnn_base.py:517-642)
    def _n_ratings_features(self):
        return 10 if self.use_ratings_features else 0

    def _n_optional_features(self):
        return self._n_ratings_features()

    def _input_size(self):
        """ids per timestep: the item id, plus one rating-bucket id with --rf (rnn_base.py:615-622)."""
        return 2 if self.use_ratings_features else 1

    def _features_of(self, sequence):
        """[L, K] int32 ids of a [L,2] (item, rating) array (rnn_base.py:578-593,624-642)."""
        sequence = np.asarray(sequence, dtype=np.float64).reshape(-1, 2)
        ids = np.empty((len(sequence), self._input_size()), dtype=np.int32)
        ids[:, 0] = sequence[:, 0]
        if self.use_ratings_features:
            ids[:, 1] = self.n_items + (np.floor(sequence[:, 1] * 2 + 0.5).astype(np.int64) - 1) % 10
        return ids

    def _get_features(self, item, user_id=None):
        return self._features_of(np.asarray([item], dtype=np.float64))[0]

    # ------------------------------------------------------------------ compiled callables
    def _split_rows(self, arr):
        """This rank's rows of a global-batch array."""
        if self.n_ranks == 1:
            return arr
        lo = self.rank * self.local_batch
        return arr[lo:lo + self.local_batch]

    def _compile_train_function(self):
        raise NotImplementedError

    def _compile_predict_function(self):
        """predict_function(X, mask) -> deterministic network output (rnn_base.py:188-194)."""
        self.predict_function = lambda X, mask: self.engine.scores(X, mask)

    _test_softmax = False

    def _compile_test_function(self):
        """test_function(batch, k) -> k best ids of the first row (rnn_base.py:196-213).  The batch is
        the tuple made by _prepare_input; its last entry carries the items to exclude (dense [B,N] like
        the reference, or a ragged list of id lists)."""
        def test_function(inputs, k=10):
            return self.test_function_batched(inputs, k)[0]
        self.test_function = test_function

    def test_function_batched(self, inputs, k=10):
        X, mask, exclude = inputs[0], inputs[1], inputs[-1]
        excl = None
        if self.interactions_are_unique and exclude is not None:
            if isinstance(exclude, np.ndarray) and exclude.ndim == 2:
                excl = [np.nonzero(row)[0].tolist() for row in exclude]
            else:
                excl = [list(e) for e in exclude]
        return self.engine.topk(X, mask, k=k, exclude=excl, softmax=self._test_softmax, neg_inf=False)

    def top_k_recommendations(self, sequence, user_id=None, k=10, exclude=None):
        """k recommendations (item ids, best first) for a sequence of (id, rating) (rnn_base.py:132-159)."""
        if exclude is None:
            exclude = []
        sequence = np.asarray(sequence, dtype=np.float64).reshape(-1, 2)
        tail = sequence[-min(self.max_length, len(sequence)):]
        X = np.zeros((1, self.max_length, self._input_size()), dtype=np.int32)
        X[0, :len(tail), :] = self._features_of(tail)
        mask = np.zeros((1, self.max_length), dtype=np.float32)
        mask[0, :len(tail)] = 1
        banned = list(exclude)
        if self.interactions_are_unique:
            banned += sequence[:, 0].astype(np.int64).tolist()
        ids = self.engine.topk(X, mask, k=k, exclude=[banned], softmax=False, neg_inf=True)
        return list(ids[0])

    # ------------------------------------------------------------------ training loop (rnn_base.py:215-356)
    def set_dataset(self, dataset):
        self.dataset = dataset
        self.target_selection.set_dataset(dataset)

    def get_pareto_front(self, metrics, metrics_names):
        costs = np.zeros((len(metrics[metrics_names[0]]), len(metrics_names)))
        for i, m in enumerate(metrics_names):
            costs[:, i] = np.array(metrics[m]) * self.metrics[m]['direction']
        is_efficient = np.ones(costs.shape[0], dtype=bool)
        for i, c in enumerate(costs):
            if is_efficient[i]:
                is_efficient[is_efficient] = np.any(costs[is_efficient] >= c, axis=1)
        return np.where(is_efficient)[0].tolist()

    def train(self, dataset, max_time=np.inf, progress=2.0, time_based_progress=False, autosave='All', save_dir='',
              min_iterations=0, max_iter=np.inf, max_progress_interval=np.inf, load_last_model=False,
              early_stopping=None, validation_metrics=['sps']):
        """Same arguments and return value as the reference (rnn_base.py:215-356)."""
        self.set_dataset(dataset)
        if len(set(validation_metrics) & set(self.metrics.keys())) < len(validation_metrics):
            raise ValueError('Incorrect validation metrics. Metrics must be chosen among: ' + ', '.join(self.metrics.keys()))
        if not hasattr(self, 'train_function'):
            self._compile_train_function()
        if not hasattr(self, 'test_function'):
            self._compile_test_function()

        iterations = 0
        epochs_offset = 0
        if load_last_model:
            epochs_offset = self.load_last(save_dir)

        if (self.device_batches and self._supports_device_batches and self.sequence_noise.name == ""
                and self._uploaded is None and dataset.training_set.lines):
            self._upload_training_sequences(dataset)
        batch_generator = self._gen_mini_batch(self.sequence_noise(dataset.training_set()))
        if self.prefetch_batches > 0 and not getattr(self.target_selection, 'determinist_test', True):
            raise ValueError("--prefetch and --rand_test_target draw from the same RNG streams in two threads; "
                             "use one or the other")
        if self.prefetch_batches > 0:       # the call the reference keeps commented out (rnn_base.py:273-274)
            batch_generator = threaded_generator(batch_generator, num_cached=self.prefetch_batches)
        start_time = time()
        next_save = int(progress)
        train_costs, current_train_cost, epochs = [], [], []
        metrics = {name: [] for name in self.metrics.keys()}
        filename = {}
        first_metric = list(self.metrics.keys())[0]
        # Every rank must execute the same number of train steps (each one ends in a collective all-reduce) and take the
        # same validate / stop decisions.  Decisions that depend on a wall clock are therefore taken on rank 0's clock:
        # it is broadcast once per iteration, and only when such a decision exists (--max_time, --time_based_progress).
        clock_matters = self.n_ranks > 1 and (time_based_progress or np.isfinite(max_time))
        if clock_matters and self.control is None:
            raise ValueError("max_time / time_based_progress with several ranks need the control plane "
                             "(helpers/rendezvous.Control) so that all ranks stop on the same iteration")

        def elapsed():
            e = time() - start_time
            return self.control.broadcast(e) if clock_matters else e

        try:
            while iterations < max_iter:
                now = elapsed()
                if not now < max_time:
                    break
                try:
                    batch = next(batch_generator)
                    cost = self.train_function(*batch)
                    if np.isnan(cost):
                        raise ValueError("Cost is NaN")
                except StopIteration:
                    break
                current_train_cost.append(cost)
                iterations += 1
                progress_indicator = int(elapsed()) if time_based_progress else iterations
                if progress_indicator >= next_save:
                    if progress_indicator >= min_iterations:
                        epochs.append(epochs_offset + dataset.training_set.epochs)
                        train_costs.append(np.mean(current_train_cost))
                        current_train_cost = []
                        metrics = self._compute_validation_metrics(metrics)
                        self._print_progress(iterations, epochs[-1], start_time, train_costs, metrics, validation_metrics)
                        run_nb = len(metrics[first_metric]) - 1
                        if self.rank == 0:
                            if autosave == 'All':
                                filename[run_nb] = save_dir + self._get_model_filename(round(epochs[-1], 3))
                                self.save(filename[run_nb])
                            elif autosave == 'Best':
                                pareto_runs = self.get_pareto_front(metrics, validation_metrics)
                                if run_nb in pareto_runs:
                                    filename[run_nb] = save_dir + self._get_model_filename(round(epochs[-1], 3))
                                    self.save(filename[run_nb])
                                    for run in [r for r in filename if r not in pareto_runs]:
                                        try:
                                            os.remove(filename[run])
                                        except OSError:
                                            print('Warning : Previous model could not be deleted')
                                        del filename[run]
                        if early_stopping is not None:
                            if all([early_stopping(epochs, metrics[m]) for m in validation_metrics]):
                                break
                    if isinstance(progress, int):
                        next_save += min(progress, max_progress_interval)
                    else:
                        next_save += min(max_progress_interval, next_save * (progress - 1))
        except KeyboardInterrupt:
            print('Training interrupted')
        finally:
            if isinstance(batch_generator, threaded_generator):
                batch_generator.close()

        if len(metrics[validation_metrics[0]]) == 0:
            return ({m: None for m in self.metrics.keys()}, time() - start_time, None)
        best_run = np.argmax(np.array(metrics[validation_metrics[0]]) * self.metrics[validation_metrics[0]]['direction'])
        return ({m: metrics[m][best_run] for m in self.metrics.keys()}, time() - start_time, filename.get(best_run))

    def _compute_validation_metrics(self, metrics):
        """One validation pass (rnn_base.py:358-371).  The reference evaluates one user per compiled
        call; here validation users are packed local_batch rows at a time into the fused
        exclude + top-k kernel -- identical instances, identical metrics."""
        ev = evaluation.Evaluator(self.dataset, k=10)
        gen = self._gen_mini_batch(self.dataset.validation_set(epochs=1), test=True)
        pending = []

        def flush():
            if not pending:
                return
            X = np.concatenate([p[0][0] for p in pending], axis=0)
            mask = np.concatenate([p[0][1] for p in pending], axis=0)
            excl = [p[0][-1][0] for p in pending]
            preds = self.test_function_batched((X, mask, excl), 10)
            for (_, goal), pred in zip(pending, preds):
                ev.add_instance(goal, pred)
            del pending[:]

        for batch_input, goal in gen:
            pending.append((batch_input, goal))
            if len(pending) == self.local_batch:
                flush()
        flush()
        metrics['recall'].append(ev.average_recall())
        metrics['sps'].append(ev.sps())
        metrics['ndcg'].append(ev.average_ndcg())
        metrics['user_coverage'].append(ev.user_coverage())
        metrics['item_coverage'].append(ev.item_coverage())
        metrics['blockbuster_share'].append(ev.blockbuster_share())
        return metrics

    _supports_device_batches = False

    def _upload_training_sequences(self, dataset):
        """Encode every training sequence once ([L, K] ids) and hand the CSR to the library."""
        lines = dataset.training_set.lines
        feats = [self._features_of(seq) for _, seq in lines]
        off = np.zeros(len(lines) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(f) for f in feats])
        if off[-1] >= 2 ** 31:
            return False
        ids = np.concatenate(feats, axis=0) if feats else np.zeros((0, self._input_size()), np.int32)
        self.engine.dataset_upload(off.astype(np.int32), ids)
        self._uploaded = {uid: i for i, (uid, _) in enumerate(lines)}
        return True

    def _plain_first_target(self):
        """True when a row's target is simply the item that follows its input window: one target, no shuffling, no
        popularity-biased skipping (target_selection.py:41-53 then draws nothing from the RNGs)."""
        ts = self.target_selection
        return (type(ts) is SelectTargets and ts.n_targets == 1 and not ts.shuffle and ts.bias < 0
                and hasattr(self, '_compact_from_triples'))

    def _gen_compact_batches(self, sequence_generator, max_reuse_sequence=np.inf):
        """_gen_mini_batch for the device-assembly form, one numpy pass per USER instead of one python iteration per
        ROW: the same `random.sample` calls in the same order as the row loop below (so the rows, and a seeded run,
        are identical), but the windows / targets of a user's rows are cut with array arithmetic.  With several ranks
        every process still walks the same global batch, now at a cost that does not grow with the row count."""
        T, Bsz = self.max_length, self.batch_size
        while True:
            j = 0
            seq_idx, starts, lens, ys = [], [], [], []
            while j < Bsz:
                try:
                    sequence, user_id = next(sequence_generator)
                except StopIteration:
                    return
                n_pick = int(min([Bsz - j, len(sequence) - 2, max_reuse_sequence]))
                if n_pick <= 0:
                    continue
                ls = np.array(sorted(random.sample(range(2, len(sequence)), n_pick)), dtype=np.int64)
                st = np.maximum(0, ls - T)
                seq_idx.append(np.full(n_pick, self._uploaded[user_id], dtype=np.int32))
                starts.append(st)
                lens.append(ls - st)
                ys.append(sequence[ls, 0])
                j += n_pick
            yield self._compact_from_triples(np.concatenate(seq_idx), np.concatenate(starts).astype(np.int32),
                                             np.concatenate(lens).astype(np.int32),
                                             np.concatenate(ys).astype(np.int32))

    def _gen_mini_batch(self, sequence_generator, test=False, max_reuse_sequence=np.inf):
        """Mini-batch generator with the reference's semantics (rnn_base.py:373-420): a training batch
        is made of nested prefixes -- sorted random split points l in [2, len) of as few user
        sequences as needed to fill exactly batch_size rows; row = (user, seq[max(0,l-T):l],
        targets chosen in seq[l:]).  test=True: one row per user, split in the middle."""
        if not test and self._uploaded is not None and self._plain_first_target():
            yield from self._gen_compact_batches(sequence_generator, max_reuse_sequence)
            return
        while True:
            j = 0
            sequences = []
            batch_size = 1 if test else self.batch_size
            while j < batch_size:
                try:
                    sequence, user_id = next(sequence_generator)
                except StopIteration:
                    return
                if not test:
                    n_pick = int(min([batch_size - j, len(sequence) - 2, max_reuse_sequence]))
                    seq_lengths = sorted(random.sample(range(2, len(sequence)), n_pick)) if n_pick > 0 else []
                else:
                    seq_lengths = [int(len(sequence) / 2)]
                skipped_seq = 0
                # the rows of one user are windows of the same sequence: encode it once, hand every row a view
                # (4th element, consumed by _fill_inputs; the first three are the reference's [user, input, targets])
                ids = self._features_of(sequence) if len(seq_lengths) > 1 else None
                for l in seq_lengths:
                    target = self.target_selection(sequence[l:], test=test)
                    if len(target) == 0:
                        skipped_seq += 1
                        continue
                    start = max(0, l - self.max_length)
                    row = [user_id, sequence[start:l], target]
                    if not test and self._uploaded is not None:
                        row.append(None)
                        row.append((self._uploaded[user_id], start, l - start))     # device-assembly triple
                    elif ids is not None:
                        row.append(ids[start:l])
                    sequences.append(row)
                j += len(seq_lengths) - skipped_seq
            if test:
                self._assembling_test_batch = True      # validation must not draw from the training RNG streams
                try:
                    batch_input = self._prepare_input(sequences)
                finally:
                    self._assembling_test_batch = False
                yield batch_input, [int(i[0]) for i in sequence[seq_lengths[0]:]]
            else:
                yield self._prepare_input(sequences)

    def _fill_inputs(self, sequences):
        """Ragged -> padded, left-aligned tensors (rnn_one_hot.py:90-101): X [B,T,K] int32, mask [B,T]
        float32, plus the ragged list of seen item ids (the reference's dense `exclude` rows)."""
        B = len(sequences)
        X = np.zeros((B, self.max_length, self._input_size()), dtype=np.int32)
        lens = np.empty(B, dtype=np.int64)
        seen = []
        for i, row in enumerate(sequences):
            in_seq = row[1]
            n = len(in_seq)
            X[i, :n, :] = row[3] if (len(row) > 3 and row[3] is not None) else self._features_of(in_seq)   # pre-encoded view
            lens[i] = n
            seen.append(X[i, :n, 0])
        mask = (np.arange(self.max_length)[None, :] < lens[:, None]).astype(np.float32)
        return X, mask, seen

    def _print_progress(self, iterations, epochs, start_time, train_costs, metrics, validation_metrics):
        if self.rank != 0:
            return
        print(self.name, iterations, "batchs, ", epochs, " epochs in", time() - start_time, "s")
        print("Last train cost : ", train_costs[-1])
        for m in self.metrics:
            print(m, ': ', metrics[m][-1])
            if m in validation_metrics:
                d = self.metrics[m]['direction']
                print('Best ', m, ': ', max(np.array(metrics[m]) * d) * d)
        print('-----------------')
        # machine-readable progress line on stderr (rnn_base.py:433-434)
        print(iterations, epochs, time() - start_time, train_costs[-1],
              ' '.join(map(str, [metrics[m][-1] for m in self.metrics])), file=sys.stderr)

    # ------------------------------------------------------------------ checkpoints (rnn_base.py:470-515)
    def save(self, filename):
        """Weights only, as a pickled python list of numpy arrays in lasagne get_all_param_values
        order (protocol 2, readable from Python 2)."""
        print('Save model in ' + filename)
        d = os.path.dirname(filename)
        if d and not os.path.exists(d):
            os.makedirs(d)
        with open(filename, 'wb') as f:
            pickle.dump(self.engine.get_all_param_values(), f, protocol=2)

    def load_last(self, save_dir):
        def extract_number_of_epochs(filename):
            m = re.search(r'_ne([0-9]+(\.[0-9]+)?)_', filename)
            return float(m.group(1))
        files = glob.glob(save_dir + self._get_model_filename("*"))
        if len(files) == 0:
            print('No previous model, starting from scratch')
            return 0
        epochs = [extract_number_of_epochs(f) for f in files]
        last = int(np.argmax(epochs))
        print('Starting from model ' + files[last])
        self.load(files[last])
        return epochs[last]

    def load(self, filename):
        with open(filename, 'rb') as f:
            param = pickle.load(f, encoding='latin1')
        self.engine.set_all_param_values([np.asarray(p, dtype=np.float32) for p in param])
