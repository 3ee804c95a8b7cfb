"""The reference's training script (`train.py`) as a function over a config object.

`TrainConfig` keeps the script's module-level parameter names and defaults verbatim
(`train.py:22-57`); `run(config, ...)` is the script body: build reader + model, compile,
optional donor weights (`:136-145`), the epoch loop with early stopping (`:147-177`) and the two
test procedures (`:202-254`). Dataset dimensions come from `metadata` (the reference reads
`./datasets_metadata.json`, which is not in its tree) or from a ready `data_reader`.
"""
from __future__ import annotations

import datetime
import json
import os
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from .data_reader import data_reader as DataReader
from .model import load_model, omni_model
from .optimizers import Adagrad, get as get_optimizer


@dataclass
class TrainConfig:
    # Dataset parameters (train.py:22-24)
    dataset: str = "ml1m"
    useTimestamps: bool = False
    reverse_user_item_data: bool = True
    # Training parameters (train.py:27-40)
    max_epochs: int = 500
    train_sparsity: List[float] = field(default_factory=lambda: [1.0, 1.0])
    test_sparsities: List[float] = field(default_factory=lambda: [0.0, 0.1, 0.4, 0.5, 0.6, 0.9])
    batch_size: int = 128
    patience: int = 0
    shuffle_data_every_epoch: bool = True
    val_split: List[float] = field(default_factory=lambda: [0.8, 0.1, 0.1])
    useJSON: bool = True
    early_stopping_metric: str = "val_accurate_MSE"
    eval_mode: str = "fixed_split"
    l2_weight_regulatization: Optional[float] = None
    pass_through_input_training: bool = True
    dropout_probability: Optional[float] = 0.2
    # Model parameters (train.py:43-57)
    numlayers: int = 1
    num_hidden_units: object = 512
    use_causal_info: bool = False
    auxilliary_mask_type: Optional[str] = None
    aux_var_value: float = -1
    model_save_path: str = "models/"
    model_loss: str = "mean_squared_error"
    learning_rate: float = 0.005
    optimizer: object = None                   # None -> Adagrad(lr=learning_rate, epsilon=1e-08, decay=0.0), train.py:51
    activation_type: str = "sigmoid"
    use_sparse_representation: bool = False
    use_experimental_sparse_masking_layer: bool = False
    load_weights_from: Optional[str] = None
    perform_finetuning: bool = False

    def model_save_name(self) -> str:
        """train.py:59,76-80 (the timestamp suffix is appended by run())."""
        name = ("stackedDenoising_WITHfinetuning_" + str(self.train_sparsity) + "trainSparsity_" + str(self.batch_size)
                + "bs_" + str(self.numlayers) + "lay_" + str(self.num_hidden_units) + "hu_" + str(self.learning_rate)
                + "lr_" + str(self.l2_weight_regulatization) + "regul_" + str(self.auxilliary_mask_type) + "_"
                + str(self.activation_type))
        if self.reverse_user_item_data:
            name += "_itemUserReverse"
        return name + "_" + self.dataset + "_"


def compute_full_RMSE(predictions, targets, ratings_count):
    """train.py:243-252."""
    sum_squared_error = 0
    for cur_preds, cur_tars in zip(predictions, targets):
        sum_squared_error += np.sum(np.square(np.subtract(cur_preds, cur_tars, dtype=np.float64)))
    return float(np.sqrt(sum_squared_error / ratings_count))


def run(config: TrainConfig, reader: Optional[DataReader] = None, metadata: Optional[dict] = None,
        rating_range: Optional[float] = None, save_models: bool = True, verbose: int = 1,
        reference_first_epoch_fallback: bool = False, ranking_ks: Optional[List[int]] = None,
        ranking_min_value: Optional[float] = None) -> dict:
    """The body of `train.py`. Returns a dict with the history, the best epoch and test results.

    `reference_first_epoch_fallback`: the reference never saves epoch 1 (train.py:164-165), so when epoch 1 stays
    the best its reload of "the best model" fails and it tests the LIVE model, i.e. the last epoch's weights
    (train.py:194-197). False (default) tests epoch 1's weights, which is what the script means to do; True
    reproduces what it does.

    `ranking_ks`: also rank the test targets against the full catalogue (`OmniNet.evaluate_ranking`, seen items
    excluded, targets with a value below `ranking_min_value` not relevant) and report HR / precision / recall /
    NDCG at every k, MRR and AUC in results["test_ranking"] (ablation: one entry per test sparsity). It runs after
    every test procedure of the script, so the other results and their NumPy stream are those of a run without it."""
    c = config
    if c.useTimestamps or c.use_sparse_representation or c.use_experimental_sparse_masking_layer:
        raise NotImplementedError("timestamps / sparse representation / experimental masking layer are out of scope")
    if reader is None:
        if metadata is None:
            with open("./datasets_metadata.json", "r") as f:           # train.py:62-69
                metadata = json.load(f)
        d = metadata[c.dataset]
        num_items, num_users = d["num_items"], d["num_users"]
        rating_range = d["rating_range"] if rating_range is None else rating_range
        if c.reverse_user_item_data:                                   # train.py:71-76
            num_items, num_users = num_users, num_items
        print("Loading data for " + c.dataset)
        reader = DataReader(num_items, num_users, d["data_path"], nonsequentialusers=d["nonsequentialusers"],
                            use_json=c.useJSON, eval_mode=c.eval_mode, useTimestamps=c.useTimestamps,
                            reverse_user_item_data=c.reverse_user_item_data)
    num_items = reader.num_items
    if rating_range is None:
        rating_range = 1.0
    if c.eval_mode == "ablation":
        reader.split_for_validation(c.val_split)                       # train.py:85-86
    use_both_masks = c.auxilliary_mask_type == "both"                  # train.py:92-95
    omni_m = omni_model(c.numlayers, c.num_hidden_units, num_items, c.batch_size, dense_activation=c.activation_type,
                        use_causal_info=c.use_causal_info, use_timestamps=c.useTimestamps, use_both_masks=use_both_masks,
                        l2_weight_regulatization=c.l2_weight_regulatization,
                        sparse_representation=c.use_sparse_representation, dropout_probability=c.dropout_probability,
                        use_sparse_masking_layer=c.use_experimental_sparse_masking_layer,
                        auxilliary_mask_type=c.auxilliary_mask_type)
    m = omni_m.model
    optimizer = c.optimizer if c.optimizer is not None else Adagrad(lr=c.learning_rate, epsilon=1e-08, decay=0.0)
    m.compile(optimizer=get_optimizer(optimizer), loss=c.model_loss, rating_range=rating_range)   # train.py:131-133
    if c.load_weights_from is not None:                                # train.py:136-145
        print("Loading weights from ", c.load_weights_from)
        donor = load_model(os.path.join(c.model_save_path, c.load_weights_from))
        if c.perform_finetuning:
            print("Fine tuning")
            omni_m.manually_load_all_weights(donor)
        else:
            omni_m.load_and_fix_for_denoising_autoencoders(donor)
    save_name = c.model_save_name() + datetime.datetime.now().strftime("%I_%M%p_%B_%d_%Y")
    if save_models:
        os.makedirs(c.model_save_path, exist_ok=True)

    def gen(which, sparsity, **kw):
        return reader.data_gen(c.batch_size, sparsity, train_val_test=which, shuffle=c.shuffle_data_every_epoch,
                               auxilliary_mask_type=c.auxilliary_mask_type, aux_var_value=c.aux_var_value,
                               sparse_representation=c.use_sparse_representation, **kw)

    min_loss, best_epoch, best_weights = None, 0, None
    val_history, history = [], []
    last_epoch = 0
    for i in range(c.max_epochs):                                      # train.py:150-177
        if verbose:
            print("Starting epoch ", i + 1)
        train_gen = gen("train", c.train_sparsity, pass_through_input_training=c.pass_through_input_training)
        valid_gen = gen("valid", c.train_sparsity)
        hist = m.fit_generator(train_gen, np.floor(reader.train_set_size / c.batch_size) - 1,
                               validation_data=valid_gen,
                               validation_steps=np.floor(reader.val_set_size / c.batch_size) - 1, verbose=verbose)
        history.append({k: v[-1] for k, v in hist.history.items()})
        val_loss = hist.history[c.early_stopping_metric][-1]
        val_history.extend(hist.history[c.early_stopping_metric])
        last_epoch = i
        if min_loss is None:
            # the reference does not save here (train.py:164-165); keeping the weights makes
            # "best model" defined from epoch 1 without changing any stopping decision
            min_loss, best_weights = val_loss, m.get_weights()
        elif min_loss > val_loss:
            min_loss, best_epoch, best_weights = val_loss, i, m.get_weights()
            if save_models:
                m.save(os.path.join(c.model_save_path, save_name + "_epoch_" + str(i + 1) + "_bestValidScore"))
        elif i - best_epoch > c.patience:
            print("Stopping early at epoch ", i + 1)
            print("Best epoch was ", best_epoch + 1)
            print("Val history: ", val_history)
            break
    # Testing (train.py:181-199): the best-validation weights, optimizer state dropped
    if not (reference_first_epoch_fallback and best_epoch == 0):
        m.set_weights(best_weights)
    if save_models:
        m.save(os.path.join(c.model_save_path, save_name + "_bestValidScore"))
    print("Testing model from epoch: ", best_epoch + 1)
    results = {"history": history, "best_epoch": best_epoch, "epochs_run": last_epoch + 1,
               "val_history": val_history, "model": omni_m, "save_name": save_name}
    test_steps = np.floor(reader.test_set_size / c.batch_size) - 1
    if c.eval_mode == "ablation":                                      # train.py:202-213
        print("\nEvaluating model with ablations")
        results["test"] = {}
        for test_sparsity in c.test_sparsities:
            test_results = m.evaluate_generator(gen("test", test_sparsity), test_steps)
            print("\nTest results with sparsity: ", test_sparsity)
            for name, v in zip(m.metrics_names, test_results):
                print(name, " : ", v)
            results["test"][test_sparsity] = dict(zip(m.metrics_names, test_results))
    else:                                                              # train.py:215-255
        print("\nEvaluating model with fixed split")
        test_results = m.evaluate_generator(gen("test", None), test_steps)
        print("Test results with fixed split")
        for name, v in zip(m.metrics_names, test_results):
            print(name, " : ", v)
        results["test"] = dict(zip(m.metrics_names, test_results))
        print("Testing manually")
        manual = gen("test", None, return_target_count=True)
        sse, ratings_count = 0.0, 0
        for _ in range(int(np.floor(reader.test_set_size / c.batch_size))):
            batch = next(manual)
            # sum((mask*full - t)^2) over the batch == the step's sum of squared errors; the
            # dense predict()/subtract of train.py:239-249 is available as m.predict(batch)
            m.test_on_batch(batch, sync=False)
            first = m.read_metrics(m.steps_logged() - 1, 1)
            sse += float(first[0, 6])
            ratings_count += batch.target_count
        rmse = float(np.sqrt(sse / ratings_count)) if ratings_count else float("nan")
        print("Manual test RMSE is ", rmse)
        results["manual_test_rmse"] = rmse
    if ranking_ks is not None:
        print("\nEvaluating ranking of the test targets")
        if c.eval_mode == "ablation":
            results["test_ranking"] = {}
            for test_sparsity in c.test_sparsities:
                results["test_ranking"][test_sparsity] = m.evaluate_ranking(
                    gen("test", test_sparsity), test_steps, ks=ranking_ks, min_value=ranking_min_value)
        else:
            results["test_ranking"] = m.evaluate_ranking(gen("test", None), test_steps, ks=ranking_ks,
                                                         min_value=ranking_min_value)
        if verbose:
            print("Test ranking: ", results["test_ranking"])
    return results

