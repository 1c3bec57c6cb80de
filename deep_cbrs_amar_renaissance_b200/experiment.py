"""Thin experiment driver with the command line, the file formats and the build / train / evaluate sequence of
/root/reference/src/experiment.py:47-318, so that the reference's `config.yaml` and `econfigs/*.yaml` grids run on the
CUDA path unchanged:

    python -m deep_cbrs_amar_renaissance_b200.experiment -c config.yaml -e econfigs/basic-gnn.yaml [--out runs]

What is kept: base config + 'linear' / 'grid' experiment sections (MultiExperimenter, experiment.py:243-311), class
and loader lookup by name (:107-118), loader / optimiser keyword filtering by signature (:120-134), the constructor
dispatch on the model family (:136-153), compile -> one call to create the weights -> summary (:155-170), fit with the
log callback (:172-188), evaluate -> predict -> per-user top-5 / top-10 written as
predictions/top_<k>/predictions_1.tsv -> P/R/F1@k (:190-222), one failed experiment does not stop the others (:299-302).
What is added, off unless a config sets the top-level key `catalog_metrics: true`: P/R/F1@k of full-catalog top-k lists
(every item ranked for every user, the user's training items excluded) against the test ratings, reported as
catalog_{precision,recall,f1}_at_{k}; `catalog_metrics: all` adds catalog_{ndcg,map,hit_rate,mrr}_at_{k}.  The metrics
are computed on the device from the lists and the test ratings (utilities.metrics.catalog_ranking_metrics).
What is replaced: MLflow run management by a directory per run holding config.yaml, log.txt, metrics.json;
ruamel.yaml by PyYAML with the YAML-1.2 float forms the files use (`1e-4`); the Java evaluator by
utilities.metrics.top_k_metrics.
"""
import argparse
import copy
import importlib
import inspect
import json
import os
import re
import time
import traceback

import numpy as np
import yaml

from . import models  # noqa: F401  (model modules are looked up by name below)
from .data import loaders
from .keras_like import set_seed
from .models.basic import BasicGNN, BasicKnowledgeGCN, BasicRS, BasicTSGNN, BasicTWGNN
from .models.hybrid import HybridBertGNN, HybridCBRS
from .training import Adam
from .utilities.keras import LogCallback, get_total_parameters
from .scoring import ItemLists
from .utilities.metrics import RANKING_METRICS, catalog_ranking_metrics, top_k_metrics, top_k_predictions
from .utilities.utils import get_experiment_logger, make_grid, nested_dict_update

PARAMS_PATH = 'config.yaml'
EXPERIMENTS_PATH = 'experiments.yaml'
RUNS_PATH = './runs'
LOG_FREQUENCY = 100
METRICS_TOP_KS = [5, 10]
CATALOG_METRICS = ("precision", "recall", "f1")   # catalog_metrics: true; `all` reports every RANKING_METRICS entry


class _Loader(yaml.SafeLoader):
    """PyYAML follows YAML 1.1, where `1e-4` is a string; the reference reads its files with ruamel (YAML 1.2),
    where it is a float (config.yaml:9, every l2_regularizer list of the grids)."""


_Loader.add_implicit_resolver(
    'tag:yaml.org,2002:float',
    re.compile(r'^[-+]?(?:[0-9][0-9_]*\.[0-9_]*(?:[eE][-+]?[0-9]+)?|\.[0-9_]+(?:[eE][-+]?[0-9]+)?'
               r'|[0-9][0-9_]*[eE][-+]?[0-9]+|\.(?:inf|Inf|INF)|\.(?:nan|NaN|NAN))$'),
    list('-+0123456789.'))


def load_yaml(path):
    with open(path) as fp:
        return yaml.load(fp, Loader=_Loader)


class Config(dict):
    """attribute access on a nested dict (what EasyDict gives the reference, experiment.py:53)"""

    def __init__(self, mapping=()):
        super().__init__()
        for key, value in dict(mapping).items():
            self[key] = Config(value) if isinstance(value, dict) else value

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError:
            raise AttributeError(key)

    def __setattr__(self, key, value):
        self[key] = value

    def plain(self):
        return {k: v.plain() if isinstance(v, Config) else v for k, v in self.items()}


def _by_signature(fn, mapping):
    """the entries of `mapping` that `fn` takes (experiment.py:125-127,131-133)"""
    accepted = inspect.signature(fn).parameters.keys()
    return {k: mapping[k] for k in mapping.keys() & accepted}


class Experimenter:
    def __init__(self, config, exp_path):
        config = copy.deepcopy(config)
        self.config = Config(config)
        set_seed(self.config.seed)
        name = self.config.model.name
        module_name, class_name = name.split('.')
        self.model_class = getattr(importlib.import_module(models.__name__ + '.' + module_name), class_name)
        catalog = self.config.get('catalog_metrics')
        self.catalog_metrics = bool(catalog)
        self.catalog_metric_names = RANKING_METRICS if catalog == 'all' else CATALOG_METRICS
        if self.catalog_metrics and not hasattr(self.model_class, 'recommend_top_k'):
            raise ValueError("catalog_metrics: {} scores pre-computed embedding rows and has no full-catalog top-k "
                             "(recommend_top_k); use a graph model".format(name))
        self.exp_name = time.strftime("%m_%d-%H_%M") + '-' + name
        if BasicRS.__name__ in name:
            pass
        elif HybridCBRS.__name__ in name:
            self.exp_name += '-feature' if self.config.model.feature_based else '-entity'
        else:
            self.exp_name += '-{}-{}'.format(self.config.model.l2_regularizer, self.config.model.final_node)
        if self.config.get('details'):
            self.exp_name += '-' + str(self.config.details)
        run_dir, k = os.path.join(exp_path, self.exp_name), 1
        while os.path.exists(run_dir):
            k += 1
            run_dir = os.path.join(exp_path, "{}.{}".format(self.exp_name, k))
        self.dest = os.path.join(run_dir, 'artifacts')
        self.predictions_dest = os.path.join(self.dest, "predictions")
        os.makedirs(self.predictions_dest)
        with open(os.path.join(self.dest, "config.yaml"), 'w') as fp:
            yaml.safe_dump(config, fp)
        self.logger = get_experiment_logger(self.dest)
        self.logger.info('CONFIG\n' + yaml.safe_dump(config))
        self.load_function = getattr(loaders, self.config.dataset.load_function_name)
        if self.config.parameters.optimizer.name != 'Adam':
            raise NotImplementedError("optimizer '{}' (the reference's configs use Adam)".format(self.config.parameters.optimizer.name))
        self.trainset = self.testset = self.model = self.optimizer = self.callback = None
        self.parameters = self.config.parameters
        self.metrics = {}

    def build_dataset(self):
        self.trainset, self.testset = self.load_function(**_by_signature(self.load_function, self.config.dataset))

    def build_optimizer(self):
        self.optimizer = Adam(**_by_signature(Adam.__init__, self.parameters.optimizer))

    def build_model(self):
        self.logger.info('Building model...')
        cls, kw = self.model_class, self.config.model.plain()
        if issubclass(cls, (BasicKnowledgeGCN, BasicTSGNN, BasicTWGNN)):
            self.model = cls(len(self.trainset.users), len(self.trainset.items), self.trainset.adj_matrix, **kw)
        elif issubclass(cls, (BasicGNN, HybridBertGNN)):
            self.model = cls(self.trainset.adj_matrix, **kw)
        else:
            self.model = cls(**kw)
        self.model.compile(loss=self.parameters.loss, optimizer=self.optimizer, metrics=self.parameters.metrics)
        self.model(self.trainset[0][0])  # one prediction creates the weights
        self.model.summary(print_fn=self.logger.info, expand_nested=True)
        trainable, non_trainable = get_total_parameters(self.model)
        self.metrics.update(trainable_params=trainable, non_trainable_params=non_trainable)

    def train(self):
        self.logger.info("Experiment folder: " + self.dest)
        self.build_dataset()
        self.build_optimizer()
        self.build_model()
        self.logger.info('Training:')
        self.callback = LogCallback(self.logger, LOG_FREQUENCY)
        history = self.model.fit(self.trainset, epochs=self.parameters.epochs, workers=self.config.n_workers,
                                 callbacks=[self.callback])
        self.metrics.update(batch_time=self.callback.get_batch_time(), training_time=self.callback.training_time,
                            history=history.history)

    def evaluate(self):
        loss, accuracy = self.model.evaluate(self.testset)
        self.metrics.update(test_loss=loss, test_accuracy=accuracy)
        predictions = self.model.predict(self.testset)
        ratings_pred = np.concatenate([self.testset.ratings[:, [0, 1]], predictions], axis=1)
        for k in METRICS_TOP_KS:
            top = top_k_predictions(ratings_pred, self.trainset.users, self.trainset.items, k=k)
            top_k_dest = os.path.join(self.predictions_dest, "top_{}".format(k))
            os.makedirs(top_k_dest, exist_ok=True)
            top.to_csv(os.path.join(top_k_dest, "predictions_1.tsv"), sep='\t', header=False, index=False)
            res = top_k_metrics(self.config.dataset.test_ratings_filepath, top_k_dest)[k]
            self.metrics.update({"precision_at_{}".format(k): res["precision"], "recall_at_{}".format(k): res["recall"],
                                 "f1_at_{}".format(k): res["f1"]})
        rows = [("", m) for m in CATALOG_METRICS]
        if self.catalog_metrics:
            self.evaluate_catalog()
            rows += [("catalog_", m) for m in self.catalog_metric_names]
        table = "\n".join("{}{}@{}: {:.6f}".format(p, m, k, self.metrics["{}{}_at_{}".format(p, m, k)])
                          for p, m in rows for k in METRICS_TOP_KS)
        self.logger.info('\n' + table)
        print('\n' + table)

    def evaluate_catalog(self):
        """P/R/F1@k (with `catalog_metrics: all` also NDCG, MAP, hit rate and MRR @k) of each user's top-k over the WHOLE
        catalog, its training items excluded, against the test ratings: the items a user rated >= 1 in the test set are
        its relevant items, as in the RiVal restatement of the test-pair metrics.  Lists and relevance stay on the
        device; one kernel computes every metric at both cutoffs."""
        users, items = self.trainset.users, self.trainset.items
        if isinstance(self.model, HybridBertGNN) and self.model.content_table is None:
            self.model.set_content_table(self.trainset.embeddings.embeddings)
        seen = ItemLists.from_ratings(self.trainset.ratings, len(users), len(items), device="cuda")
        ids, _ = self.model.recommend_top_k(len(users), len(items), max(METRICS_TOP_KS), exclude=seen)
        # the loader maps every test id into the training vocabulary, so the test ratings index the same catalog
        relevant = ItemLists.from_ratings(self.testset.ratings, len(users), len(items), device="cuda", min_rating=1,
                                          distinct=True)
        res = catalog_ranking_metrics(ids, relevant, cutoffs=METRICS_TOP_KS, metrics=self.catalog_metric_names)
        self.metrics.update({"catalog_" + key: value for key, value in res.items() if key != "users"})

    def run(self):
        try:
            self.train()
            self.evaluate()
        finally:
            self.close()
        return self.metrics

    def close(self):
        with open(os.path.join(self.dest, "metrics.json"), "w") as fp:
            json.dump(self.metrics, fp, indent=1, default=float)
        for handler in list(self.logger.handlers):
            handler.close()
            self.logger.removeHandler(handler)


class MultiExperimenter:
    """base config + the experiments of an experiment file ('linear': named overrides, 'grid': cartesian products)"""

    def __init__(self, params_path, experiments_path, exp_path):
        self.exp_path = exp_path
        self.base_config = load_yaml(params_path)
        config = load_yaml(experiments_path) or {}
        self.experiments = dict(config.get('linear') or {})
        for grid in (config.get('grid') or {}).values():
            self.experiments.update({str(elem): elem for elem in make_grid(grid)})
        print("Retrieved experiments: {}".format(len(self.experiments)))
        for exp in self.experiments:
            print(exp)
        self.results = {}

    def run_experiment(self, exp_name):
        config = copy.deepcopy(self.base_config)
        if self.experiments[exp_name]:  # None runs the base config
            config = nested_dict_update(config, self.experiments[exp_name])
        print('-----------------------------------------------\n{}\n-----------------------------------------------\n'.format(exp_name))
        try:
            self.results[exp_name] = Experimenter(config, self.exp_path).run()
        except Exception as e:  # one failed experiment does not stop the grid (experiment.py:299-302)
            print(e)
            traceback.print_exc()
            self.results[exp_name] = None

    def run(self, only=None):
        names = list(self.experiments)[:only]
        for k, exp_name in enumerate(names):
            print("Experiment {}/{}".format(k + 1, len(names)))
            self.run_experiment(exp_name)
        return self.results


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument("-c", "--config", dest='config', type=str, help="Config input file", default=PARAMS_PATH)
    parser.add_argument("-e", "--experiments", dest='experiments', type=str, help="Experiment (grid search) file",
                        default=EXPERIMENTS_PATH)
    parser.add_argument("--exp_name", dest='exp_name', type=str, help="Name of the group of runs", default='cbrs')
    parser.add_argument("--out", dest='out', type=str, help="Where the runs are stored", default=RUNS_PATH)
    parser.add_argument("--only", dest='only', type=int, default=None, help="Run only the first N experiments")
    args = parser.parse_args(argv)
    exp_path = os.path.join(args.out, re.sub(r'[^A-Za-z0-9_.-]+', '_', args.exp_name))
    os.makedirs(exp_path, exist_ok=True)
    return MultiExperimenter(args.config, args.experiments, exp_path).run(args.only)


if __name__ == "__main__":
    main()
