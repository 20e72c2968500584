"""Learned dynamics model s' - s = f(s, a): API of the reference's ``Dyn_Model``
(smartstart/RLContinuousAlgorithms/NN_Dynamics_Model/dynamics_model.py).

The reference builds a float64 TF1 graph (feedforward_network.py:3-23) and trains it with
Adam / MSE on a mix of the initial random-policy data and the replay-buffer data
(dynamics_model.py:52-171), feeding numpy batches through ``sess.run``.  Here the model lives in
the CUDA engine: ``train`` uploads the two data sets once, draws the batch row indices with the
reference's numpy calls (same stream of ``npr`` draws, hence the same batches for the same seed)
and runs every epoch's Adam steps on the device (csrc/dyn_train.cu, one index upload and one loss
read-back per epoch, no host copy of a batch); the trained parameters are handed to the rollout
kernels on the device (``Engine.dyn_commit``).  ``precision="fp64"`` trains in float64 like the
reference's graph (data, parameters, Adam moments and every step), so the weights stay the reference's
up to the summation order of the GEMMs; the default "fp32" is the faster FP32 trainer.  ``do_forward_sim`` keeps the reference's signature
and runs on the engine as well.  There is no CPU path: a missing engine raises.
"""
from __future__ import annotations

import math
import time

import numpy as np
import numpy.random as npr


def _xavier_normal(rng, shape, fan_in, fan_out):
    """tf.contrib.layers.xavier_initializer(uniform=False): truncated normal,
    stddev sqrt(1.3 * 2 / (fan_in + fan_out)) (feedforward_network.py:8)."""
    std = math.sqrt(1.3 * 2.0 / (fan_in + fan_out))
    x = rng.normal(0.0, std, size=shape)
    bad = np.abs(x) > 2 * std
    while bad.any():
        x[bad] = rng.normal(0.0, std, size=int(bad.sum()))
        bad = np.abs(x) > 2 * std
    return x


class Dyn_Model:
    def __init__(self, inputSize, outputSize, sess, learning_rate, batchsize, num_fc_layers,
                 depth_fc_layers, mean_x, mean_y, mean_z, std_x, std_y, std_z, tf_datatype, verbose,
                 engine=None, seed=None, *, precision="fp32"):
        """precision: arithmetic of the device trainer, "fp32" or "fp64" (the reference's float64; set on the
        engine here, before the initial weights).  tf_datatype is accepted and unused."""
        if engine is None:
            raise RuntimeError("Dyn_Model needs a CUDA engine (there is no CPU implementation of this path)")
        engine.dyn_set_precision(precision)
        self.precision = precision
        self.sess = sess                      # accepted for signature compatibility, unused
        self.batchsize = batchsize
        self.inputSize = inputSize
        self.outputSize = outputSize
        self.mean_x, self.mean_y, self.mean_z = mean_x, mean_y, mean_z
        self.std_x, self.std_y, self.std_z = std_x, std_y, std_z
        self.verbose = verbose
        self.engine = engine
        self.learning_rate = learning_rate
        self.num_fc_layers = num_fc_layers
        self.depth_fc_layers = depth_fc_layers
        rng = np.random.default_rng(seed)
        sizes = [inputSize] + [depth_fc_layers] * num_fc_layers + [outputSize]
        weights, biases = [], []
        for fi, fo in zip(sizes[:-1], sizes[1:]):
            # weights AND biases use the Xavier initialiser in the reference (:14-23)
            weights.append(_xavier_normal(rng, (fi, fo), fi, fo))
            biases.append(_xavier_normal(rng, (fo,), fo, fo))
        self._old_data_token = None
        self.set_weights(weights, biases)

    # ------------------------------------------------------------------ parameters
    def norm(self):
        return dict(mean_x=self.mean_x, std_x=self.std_x, mean_y=self.mean_y, std_y=self.std_y,
                    mean_z=self.mean_z, std_z=self.std_z)

    def export(self):
        """(weights, biases) as float64 numpy, [in, out] / [out] (read back from the device)."""
        return self.engine.dyn_get_params()

    @property
    def weights(self):
        return self.export()[0]

    @property
    def biases(self):
        return self.export()[1]

    def set_weights(self, weights, biases):
        """Assign the parameters (initialisation, checkpoints): Engine.set_model uploads them and
        re-packs them for the rollout kernels; the Adam moments of the device trainer survive an
        assignment of the same shape, like the optimizer slots of the reference's graph."""
        self.engine.set_model([np.asarray(w, dtype=np.float64) for w in weights],
                              [np.asarray(b, dtype=np.float64).reshape(-1) for b in biases], self.norm())
        self._old_data_token = None           # a new model may follow a shape change: data re-uploaded

    def push_to_engine(self):
        """Make the rollout kernels use the current parameters (device-side re-packing)."""
        self.engine.dyn_commit()

    # ------------------------------------------------------------------ training (device)
    def _upload_old(self, dataX, dataZ):
        token = (id(dataX), id(dataZ), dataX.shape, dataZ.shape)
        if token != self._old_data_token:      # the initial data set never changes: uploaded once
            self.engine.dyn_set_data(0, dataX, dataZ)
            self._old_data_token = token

    def train(self, dataX, dataZ, dataX_new, dataZ_new, nEpoch, save_dir, fraction_use_new,
              save_results=True):
        """dynamics_model.py:52-171: nEpoch epochs; each batch = batchsize*(1-fraction) rows of the
        shuffled old data + batchsize*fraction rows drawn from the new data.  Returns
        (mean training loss of the last epoch, old_loss, new_loss)."""
        start = time.time()
        eng = self.engine
        dataX, dataZ = np.asarray(dataX, dtype=np.float64), np.asarray(dataZ, dtype=np.float64)
        dataX_new, dataZ_new = np.asarray(dataX_new, dtype=np.float64), np.asarray(dataZ_new, dtype=np.float64)
        n_old, n_new = dataX.shape[0], dataX_new.shape[0]
        self._upload_old(dataX, dataZ)
        eng.dyn_set_data(1, dataX_new, dataZ_new)
        losses = []
        if n_new < self.batchsize * fraction_use_new:                       # :62-65
            new_per_batch = n_new
        else:
            new_per_batch = int(self.batchsize * fraction_use_new)
        old_per_batch = int(self.batchsize - new_per_batch)                 # :68
        range_of_indeces = np.arange(n_old)
        new_order = np.arange(n_new)           # "train completely from new set": the data is re-shuffled per epoch
        avg, nb = 0.0, 0
        for epoch in range(nEpoch):
            old_indeces = npr.choice(range_of_indeces, size=(n_old,), replace=False)     # :76, drawn in every branch
            if old_per_batch > 0:
                nb = int(math.floor(n_old / old_per_batch))
                idx_new = np.empty((nb, new_per_batch), dtype=np.int32)
                for b in range(nb):
                    if n_new:
                        idx_new[b] = npr.randint(0, n_new, (new_per_batch,))              # :88
                idx_old = old_indeces[:nb * old_per_batch].reshape(nb, old_per_batch)
            else:
                nb = int(math.floor(n_new / new_per_batch))
                idx_old = np.empty((nb, 0), dtype=np.int32)
                idx_new = new_order[:nb * new_per_batch].reshape(nb, new_per_batch)
            if nb:
                ep = eng.dyn_train_batches(idx_old, idx_new, self.learning_rate)
                losses.extend(ep.tolist())
                avg = float(ep.sum())
            if old_per_batch <= 0:
                new_order = new_order[npr.permutation(n_new)]                             # :124-126
            if save_results and save_dir:
                np.save(save_dir + '/training_losses.npy', losses)
            if self.verbose and epoch % 10 == 0:
                print("\n=== Epoch {} ===".format(epoch))
                print("loss: ", avg / max(nb, 1))
        if self.verbose:
            print("Training set size: ", n_old + n_new)
            print("Training duration: {:0.2f} s".format(time.time() - start))
        old_loss, nb_old = eng.dyn_eval_loss(0, self.batchsize)             # :139-150
        new_loss, nb_new = eng.dyn_eval_loss(1, self.batchsize)             # :153-166 (0 when no full batch)
        self.push_to_engine()
        return avg / max(nb, 1), old_loss, (new_loss if nb_new else 0)

    def run_validation(self, inputs, outputs, quiet=False):
        """Mean batch MSE over the full batches of (inputs, outputs) (dynamics_model.py:174-197)."""
        self.engine.dyn_set_data(1, np.asarray(inputs, dtype=np.float64), np.asarray(outputs, dtype=np.float64))
        loss, _ = self.engine.dyn_eval_loss(1, self.batchsize)
        if self.verbose and not quiet:
            print("Validation set size: ", np.shape(inputs)[0])
            print("Validation set's total loss: ", loss)
        return loss

    # ------------------------------------------------------------------ inference (engine)
    def do_forward_sim(self, forwardsim_x_true, forwardsim_y, many_in_parallel, *, precision="fp32"):
        """Multi-step open-loop prediction (dynamics_model.py:199-270) on the GPU engine.
        Returns a list of H+1 arrays [N, d] (parallel) or [d] (single sequence).

        many_in_parallel, forwardsim_y = N action sequences [N, H, da]:
          * len(forwardsim_x_true) == 2: the reference's [state, 0] form, forwardsim_x_true[0] starts every
            sequence.  As in the reference, a [2, d] array of two start states takes this branch too: its first
            row starts all N sequences.
          * otherwise forwardsim_x_true holds the N start states ([N, d] array or a list of N arrays of length d),
            sequence n starts at row n (multi-step prediction from many start states, e.g. k-step validation).
            Any other shape raises ValueError.
        precision: "fp32" (default), "bf16_tc", "auto" or "fp64" (the reference's float64 arithmetic)."""
        y = np.asarray(forwardsim_y, dtype=np.float64)
        if many_in_parallel:
            if len(forwardsim_x_true) == 2:
                start = forwardsim_x_true[0]
            else:
                start = np.asarray(forwardsim_x_true, dtype=np.float64)
                if start.ndim != 2 or y.ndim != 3 or start.shape != (y.shape[0], self.outputSize):
                    raise ValueError("per-sequence start states must be [N, d] = [%s, %d], got shape %s"
                                     % (y.shape[0] if y.ndim == 3 else "N", self.outputSize, start.shape))
            states = self.engine.forward_sim(start, y, precision)
            return [states[t] for t in range(states.shape[0])]
        states = self.engine.forward_sim(forwardsim_x_true[0], y[None, :, :], precision)
        return [states[t, 0] for t in range(states.shape[0])]
