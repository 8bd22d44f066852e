"""RNNCluster -- host mirror of neural_networks/rnn_cluster.py:19-539: a sampled-output RNN trained together with a
soft assignment of the items to clusters; at test time only the items of the cluster the user's state selects are
scored.  The arithmetic is `sbr_train_step_cluster`, `sbr_cluster_test_topk`, `sbr_cluster_build` and
`sbr_cluster_topk` (include/sbr_b200.h).

Deliberate difference: the cluster-selection noise (--csn) is drawn on the host from the global numpy RNG and passed
in with the batch, instead of Theano's MRG stream on the device."""
import os
import pickle
import random
import sys
from bisect import bisect
from time import time

import numpy as np

from ..helpers import evaluation
from . import rnn_base as rnn

LOSSES = ("Blackout", "lin", "BPRelu", "BPR", "TOP1", "CCE")


class RNNCluster(rnn.RNNBase):
    def __init__(self, n_clusters=10, loss="Blackout", cluster_type='mix', sampling=100, cluster_sampling=-1,
                 sampling_bias=0., predict_with_clusters=True, cluster_selection_noise=0., init_scale=1.,
                 scale_growing_rate=1., max_scale=50, **kwargs):
        super().__init__(**kwargs)
        self.n_clusters = int(n_clusters)
        # float32 like the reference's np.cast[floatX] (they are also what _get_model_filename prints)
        self.init_scale = np.float32(init_scale)
        self.effective_scale = np.float32(init_scale)
        self.scale_growing_rate = np.float32(scale_growing_rate)
        self.max_scale = np.float32(max_scale)    # stored, never applied (as in the reference)
        if cluster_type not in ('softmax', 'mix', 'sigmoid'):
            raise ValueError("Unknown cluster type")
        self.cluster_type = cluster_type
        self.sampling_bias = sampling_bias
        if loss not in LOSSES:
            raise ValueError('Unknown cluster loss')
        self.loss = loss
        self.cluster_selection_noise = cluster_selection_noise
        self.predict_with_clusters = predict_with_clusters
        self.n_samples = int(sampling)
        if self.n_samples < 1:
            raise ValueError("RNNCluster needs at least one sample (--sampling %s)" % sampling)
        self.n_cluster_samples = int(cluster_sampling)
        self.name = "RNN Cluster with categorical cross entropy"
        self.metrics = {'recall': {'direction': 1}, 'cluster_recall': {'direction': 1}, 'sps': {'direction': 1},
                        'cluster_sps': {'direction': 1}, 'ignored_items': {'direction': -1}, 'assr': {'direction': 1},
                        'cluster_use': {'direction': 1}, 'cluster_use_std': {'direction': -1},
                        'cluster_size': {'direction': 1}}

    loss_name = "Blackout"

    def _get_model_filename(self, epochs):
        """rnn_cluster.py:120-149."""
        filename = "rnn_clusters" + str(self.n_clusters) + "_sc" + str(self.init_scale)
        if self.scale_growing_rate != 1.:
            filename += "-" + str(self.scale_growing_rate) + "-" + str(self.max_scale)
        filename += "_"
        if self.sampling_bias > 0.:
            filename += "p" + str(self.sampling_bias)
        filename += "s" + str(self.n_samples)
        if self.n_cluster_samples > 0:
            filename += "_"
            if self.sampling_bias > 0.:
                filename += "p" + str(self.sampling_bias)
            filename += "cs" + str(self.n_cluster_samples)
        if self.cluster_type == 'softmax':
            filename += "_softmax"
        elif self.cluster_type == 'mix':
            filename += "_mix"
        if self.cluster_selection_noise > 0.:
            filename += '_n' + str(self.cluster_selection_noise)
        filename += "_c" + self.loss
        return filename + "_" + self._common_filename(epochs)

    # ------------------------------------------------------------------ model construction
    def _engine_extra_kwargs(self):
        return dict(n_samples=self.n_samples,
                    clusters=dict(n_clusters=self.n_clusters, cluster_type=self.cluster_type, loss=self.loss,
                                  n_cluster_samples=max(0, self.n_cluster_samples)))

    def _init_parameters(self):
        """The stack and out.* as RNNBase draws them, then Wc ~ GlorotUniform (the DenseLayer of :235), then
        R = 0.1 randn (:182-189, created after it at :241)."""
        rng = self._init_rng()
        vals = [self._initial_value(rng, name, shape) for name, shape in self.engine.param_infos()[:-2]]
        h_last, C = self.engine.param_infos()[-1][1]
        a = np.sqrt(6.0 / (h_last + C))
        Wc = rng.uniform(-a, a, size=(h_last, C)).astype(np.float32)
        R = (0.1 * rng.randn(self.n_items, C)).astype(np.float32)
        self.engine.set_all_param_values(vals + [R, Wc])

    # ------------------------------------------------------------------ compiled callables
    def _compile_train_function(self):
        """train_function(X, mask, Y, samples, cluster_samples, noise, scale, exclude) -> cost (rnn_cluster.py:272).
        The scale travels with the batch so that batches assembled ahead of time (--prefetch) keep their own."""
        def train_function(X, mask, Y, samples, cluster_samples, noise, scale, exclude=None):
            sl = self._split_rows
            cs = None if self.n_cluster_samples <= 0 else cluster_samples
            cost, self.last_cluster_cost = self.engine.train_step_cluster(
                sl(X), sl(mask), sl(Y), samples, cluster_samples=cs, noise=None if noise is None else sl(noise),
                scale=scale, Y_all=Y, row_offset=self.rank * self.local_batch)
            return cost
        self.train_function = train_function

    def _compile_test_function(self):
        """test_function(batch) -> (ids1, ids2, c, n_used) of the first row (rnn_cluster.py:345-351)."""
        def test_function(inputs, k=10):
            full, clus, sel, used = self.test_function_batched(inputs, k)
            return full[0], clus[0], sel[0], used[0]
        self.test_function = test_function

    def test_function_batched(self, inputs, k=10):
        X, mask, exclude = inputs[0], inputs[1], inputs[-1]
        excl = [list(e) for e in exclude] if (self.interactions_are_unique and exclude is not None) else None
        return self.engine.cluster_test_topk(X, mask, k=k, exclude=excl)

    def _popularity_sample(self):
        if not hasattr(self, '_cumsum'):
            self._cumsum = np.cumsum(np.power(self.dataset.item_popularity, self.sampling_bias))
        return bisect(self._cumsum, random.uniform(0, self._cumsum[-1]))

    def _draw(self, n):
        if self.sampling_bias > 0.:
            return np.array([self._popularity_sample() for _ in range(n)], dtype=np.int32)
        return np.random.choice(self.n_items, n).astype(np.int32)

    def _prepare_input(self, sequences):
        """(X, mask, Y, samples, cluster_samples, noise, scale, exclude) (rnn_cluster.py:363-407): samples, then
        cluster samples, then the selection noise, from the global RNGs; validation batches draw nothing."""
        X, mask, seen = self._fill_inputs(sequences)
        Y = np.array([int(t[2][0][0]) for t in sequences], dtype=np.int32)
        if getattr(self, '_assembling_test_batch', False):
            z = np.zeros(self.n_samples, dtype=np.int32)
            return (X, mask, Y, z, z, None, self.effective_scale, seen)
        samples = self._draw(self.n_samples)
        cluster_samples = self._draw(self.n_cluster_samples) if self.n_cluster_samples > 0 else samples
        noise = None
        if self.cluster_selection_noise > 0.:
            noise = np.random.normal(0.0, self.cluster_selection_noise, size=(len(sequences), self.n_clusters))
            noise = noise.astype(np.float32)
        self._update_scale()
        return (X, mask, Y, samples, cluster_samples, noise, self.effective_scale, seen)

    def _update_scale(self):
        """rnn_cluster.py:397-405: the first batch records the epoch counter; afterwards, once more than one epoch has
        passed since, the scale is multiplied by rate ** whole epochs (max_scale is never applied)."""
        epochs = self.dataset.training_set.epochs
        if not hasattr(self, '_last_epoch'):
            self._last_epoch = epochs
        elif epochs > self._last_epoch + 1 and self.scale_growing_rate != 1.:
            self.effective_scale = np.float32(self.effective_scale * self.scale_growing_rate ** int(epochs - self._last_epoch))
            self._last_epoch += int(epochs - self._last_epoch)
            if self.rank == 0:
                print("New scale: ", self.effective_scale)

    # ------------------------------------------------------------------ validation
    def _compute_validation_metrics(self, metrics):
        """rnn_cluster.py:409-445, with the validation users packed local_batch rows per call."""
        clusters = np.zeros(self.n_clusters, dtype="int")
        used_items = []
        ev = evaluation.Evaluator(self.dataset, k=10)
        ev_clusters = evaluation.Evaluator(self.dataset, k=10)
        pending = []

        def flush():
            if not pending:
                return
            X = np.concatenate([p[0][0] for p in pending], axis=0)
            mask = np.concatenate([p[0][1] for p in pending], axis=0)
            excl = [p[0][-1][0] for p in pending]
            full, clus, sel, used = self.test_function_batched((X, mask, excl), 10)
            for i, (_, goal) in enumerate(pending):
                ev.add_instance(goal, full[i])
                ev_clusters.add_instance(goal, clus[i])
                clusters[sel[i]] += 1
                used_items.append(float(used[i]))
            del pending[:]

        for batch_input, goal in self._gen_mini_batch(self.dataset.validation_set(epochs=1), test=True):
            pending.append((batch_input, goal))
            if len(pending) == self.local_batch:
                flush()
        flush()
        R = self.engine.get_all_param_values()[-2]
        if self.cluster_type == 'softmax':
            ignored_items = 0
            cluster_size = np.histogram(R.argmax(axis=1), bins=range(self.n_clusters + 1))[0].tolist()
        elif self.cluster_type == 'mix':
            ignored_items = 0
            sig_clusters = R > 0.
            sig_clusters[np.arange(self.n_items), R.argmax(axis=1)] = True
            cluster_size = sig_clusters.sum(axis=0)
        else:
            ignored_items = (R.max(axis=1) < 0.).sum()
            cluster_size = (R > 0.).sum(axis=0)
        metrics['recall'].append(ev.average_recall())
        metrics['cluster_recall'].append(ev_clusters.average_recall())
        metrics['sps'].append(ev.sps())
        metrics['cluster_sps'].append(ev_clusters.sps())
        metrics['assr'].append(self.n_items / np.mean(used_items))
        metrics['ignored_items'].append(ignored_items)
        metrics['cluster_use'].append(clusters)
        metrics['cluster_use_std'].append(np.std(clusters))
        metrics['cluster_size'].append(cluster_size)
        return metrics

    def _print_progress(self, iterations, epochs, start_time, train_costs, metrics, validation_metrics):
        """rnn_cluster.py:447-459."""
        if self.rank != 0:
            return
        print(self.name, iterations, "batchs, ", epochs, " epochs in", time() - start_time, "s")
        print("Last train cost : ", train_costs[-1])
        for m in self.metrics.keys():
            print(m, ': ', metrics[m][-1])
            if m in validation_metrics:
                print('Best ', m, ': ', max(np.array(metrics[m]) * self.metrics[m]['direction']) * self.metrics[m]['direction'])
        print('-----------------')
        print(iterations, epochs, time() - start_time, train_costs[-1], metrics['sps'][-1], metrics['cluster_sps'][-1],
              metrics['recall'][-1], metrics['cluster_recall'][-1], metrics['assr'][-1], metrics['ignored_items'][-1],
              metrics['cluster_use_std'][-1], file=sys.stderr)

    # ------------------------------------------------------------------ recommendation
    def prepare_tests(self):
        """Hard clusters of the current R, built and kept on the device (rnn_cluster.py:461-487)."""
        self.cluster_sizes = self.engine.cluster_build()

    def top_k_recommendations(self, sequence, user_id=None, k=10, exclude=None):
        """(ids, number of scored items) (rnn_cluster.py:489-513, :293-322)."""
        if exclude is None:
            exclude = []
        if self.predict_with_clusters and not hasattr(self, 'cluster_sizes'):
            self.prepare_tests()
        sequence = np.asarray(sequence, dtype=np.float64).reshape(-1, 2)
        tail = sequence[-min(self.max_length, len(sequence)):]
        X = np.zeros((1, self.max_length, self._input_size()), dtype=np.int32)
        X[0, :len(tail), :] = self._features_of(tail)
        mask = np.zeros((1, self.max_length), dtype=np.float32)
        mask[0, :len(tail)] = 1
        banned = sequence[:, 0].astype(np.int64).tolist() if self.interactions_are_unique else []
        banned += list(exclude)
        ids, n, _ = self.engine.cluster_topk(X, mask, k=k, exclude=[banned], use_clusters=self.predict_with_clusters)
        return [int(i) for i in ids[0] if i >= 0], int(n[0])

    # ------------------------------------------------------------------ checkpoints (rnn_cluster.py:515-539)
    def save(self, filename):
        """get_all_param_values(l_out), then R, then [Wc]; pickle protocol 2."""
        print('Save model in ' + filename)
        d = os.path.dirname(filename)
        if d and not os.path.exists(d):
            os.makedirs(d)
        vals = self.engine.get_all_param_values()
        with open(filename, 'wb') as f:
            pickle.dump(vals[:-2] + [vals[-2], [vals[-1]]], f, protocol=2)

    def load(self, filename):
        with open(filename, 'rb') as f:
            param = pickle.load(f, encoding='latin1')
        vals = [np.asarray(p, dtype=np.float32) for p in param[:-2]]
        vals += [np.asarray(param[-2], dtype=np.float32), np.asarray(param[-1][0], dtype=np.float32)]
        self.engine.set_all_param_values(vals)
        self.prepare_tests()
