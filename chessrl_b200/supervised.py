"""supervised: drop-in for the reference's entry point (supervised.py:36-95)

    python -m chessrl_b200.supervised modeldir datadir [--epochs 1] [--bs 8] [--debug]
        [--targets played|search] [--temperature 50] [--value-weight 0.5]

Contract kept: `train(model_dir, dataset_path, epochs=1, batch_size=8)` resumes from the newest `model-<n>.h5` of the
directory (or starts fresh when there is none), trains with a 25 % validation split and writes the weights back under
the same name; the same command-line flags.  The training step itself is chessrl_b200/training.py.
--targets search (opt-in) trains games recorded by `gen_data --scores` on the search's soft policy and score-value targets
(DESIGN.md 3.8); the default, played, is the reference's one-hot of the move played and the game's result.
"""

from __future__ import annotations

import argparse
import os

from .agent import Agent
from .dataset import DatasetGame
from .lib.logger import Logger
from .selfplay import get_model_path

VALIDATION_SPLIT = 0.25          # supervised.py:60-61

_FLAGS = (
    (("model_dir",), dict(metavar="modeldir", help="where to store (and load from) the trained model and the logs")),
    (("data_path",), dict(metavar="datadir", help="Path of .JSON dataset.")),
    (("--epochs",), dict(metavar="epochs", type=int, default=1)),
    (("--bs",), dict(metavar="bs", type=int, default=8, help="Batch size. Default 8")),
    (("--debug",), dict(action="store_true", default=False, help="Log debug messages on screen. Default false.")),
    (("--precision",), dict(choices=("fp32", "tf32", "bf16"), default=None,
                            help="arithmetic of the training step (default fp32 = the parity setting; tf32 / bf16 run the "
                                 "convolutions on the tensor cores, 8-10 x faster, gradients no longer parity-grade)")),
    (("--targets",), dict(choices=("played", "search"), default="played",
                          help="played: one-hot of the move played and the result (default); search: softmax of the "
                               "recorded root scores and a score-blended value (games from gen_data --scores)")),
    (("--temperature",), dict(type=float, default=50.0, help="search targets: softmax temperature in centipawns")),
    (("--value-weight",), dict(type=float, default=0.5,
                               help="search targets: weight w of tanh(score / 400) in the value target, 0..1")),
)


def _resume(weights_file):
    """An Agent carrying the weights of `weights_file` if that file exists, else a freshly initialised one."""
    agent = Agent(color=True)
    try:
        agent.load(weights_file)
        return agent, True
    except OSError:                       # the reference's rule: a missing checkpoint means "train a new model"
        return agent, False


def train(model_dir, dataset_path, epochs=1, batch_size=8, targets="played", temperature=50.0, value_weight=0.5):
    """targets "played" (the reference's) or "search" (DESIGN.md 3.8, with `temperature` and `value_weight`)."""
    from . import training
    if targets not in ("played", "search"):
        raise ValueError("targets: 'played' or 'search', got %r" % (targets,))
    search = training.check_targets(training.SearchTargets(float(temperature), float(value_weight))) \
        if targets == "search" else None
    log = Logger.get_instance()
    games = DatasetGame()
    games.load(dataset_path)
    log.info("%d games read from %s" % (len(games), dataset_path))
    weights_file = get_model_path(model_dir)
    agent, resumed = _resume(weights_file)
    if resumed:
        log.info("resuming from %s" % weights_file)
    else:
        log.warning("no checkpoint at %s: training a fresh model" % weights_file)
    if search is not None:
        log.info("search targets: %d of %d games carry root scores"
                 % (sum(g.search_scores is not None for g in games.games), len(games)))
    agent.train(games, epochs=epochs, batch_size=batch_size, validation_split=VALIDATION_SPLIT, logdir=model_dir,
                targets=search)
    agent.save(weights_file)
    log.info("weights written to %s" % weights_file)


def main(argv=None):
    cli = argparse.ArgumentParser(description="Trains the newest model of a directory on a dataset of recorded games.")
    for names, options in _FLAGS:
        cli.add_argument(*names, **options)
    opts = cli.parse_args(argv)
    Logger.get_instance().set_level(0 if opts.debug else 1)
    if opts.precision:
        os.environ["CRL_TRAIN_PRECISION"] = opts.precision
    train(opts.model_dir, opts.data_path, epochs=opts.epochs, batch_size=opts.bs, targets=opts.targets,
          temperature=opts.temperature, value_weight=opts.value_weight)


if __name__ == "__main__":
    main()
