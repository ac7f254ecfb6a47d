"""Times the UNMODIFIED Python reference (staged in baseline/_ref by stage_ref.py) on the host cores
of the box the GPU numbers are taken on (SURVEY.md §8(d) "CPU baseline timing", BASELINE.md §4):

  (i)  configs[0]: the reference's HarmoniesGameState in a single process, 2-player uniform-random
       playouts (random.choice over action-index-sorted legal moves -> apply_move) -> steps/s/core;
  (ii) the reference's own parallel self-play layout (trainer.py:104-107): a multiprocessing Pool
       over games, one CPU ModelManager per worker with torch.set_num_threads(1), default network
       (random init), 100 simulations per move through the reference's get_best_action_and_pi
       (MCTS.py:272) -> aggregate sims/s, with the reference's file loggers enabled (as shipped)
       and disabled.  A worker plays a bounded number of moves of one game instead of a whole game
       (a whole game is ~62 moves x 100 sims at ~13 ms each, i.e. minutes per core).

Used by bench.py (cpu_baseline.python_reference and --impl reference); never by the product.
"""

import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")


def available():
    return os.path.exists(os.path.join(REF, "harmonies_engine.py")) and os.path.isdir(os.path.join(REF, "run", "logs"))


def _import_ref():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import harmonies_engine  # noqa: F401  (the reference module, unmodified)
    import process_game_state  # noqa: F401

    return harmonies_engine, process_game_state


def steps_per_core(budget_s=4.0, seed=0):
    """(i): single-process random playouts on the reference engine."""
    import random

    he, pgs = _import_ref()
    random.seed(seed)
    steps = games = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        g = he.HarmoniesGameState()
        while not g.is_game_over():
            moves = sorted(g.get_legal_moves(), key=pgs.get_action_index)
            g = g.apply_move(random.choice(moves))
            steps += 1
        games += 1
    dt = time.perf_counter() - t0
    return {"value": steps / dt, "unit": "steps/s", "cores": 1, "games": games, "steps": steps, "seconds": dt,
            "what": "harmonies_engine.py random playouts, one process (harmonies_engine.py:145,210)"}


def _mcts_worker(args):
    """One Pool task = one game's first ``moves`` moves, exactly the loop body of self_play_worker
    (trainer.py:468-509) with its own CPU ModelManager (trainer.py:455-457)."""
    moves, sims, loggers_on, seed = args
    import random

    import numpy as np
    import torch

    torch.set_num_threads(1)
    he, _ = _import_ref()
    import config
    import loggers
    import MCTS
    from model import ModelManager

    for name in ("logger_mcts", "logger_main", "logger_tourney", "logger_memory", "logger_model"):
        getattr(loggers, name).disabled = not loggers_on
    random.seed(seed)
    np.random.seed(seed % (2**32))
    torch.manual_seed(seed)
    tc = dict(config.training_config_default, device="cpu")
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        mm = ModelManager(config.model_config_default, tc)
    mm.model.eval()
    mc = dict(config.mcts_config_default, num_simulations=sims)
    game = he.HarmoniesGameState()
    t0 = time.perf_counter()
    done = 0
    for m in range(moves):
        if game.is_game_over():
            break
        move, _pi = MCTS.get_best_action_and_pi(game.clone(), mm, mc, m)
        game = game.apply_move(move)
        done += sims
    return done, time.perf_counter() - t0


def pool_sims_per_s(workers=None, moves=2, sims=100, loggers_on=True):
    """(ii): the reference's Pool layout; returns aggregate sims/s over ``workers`` processes."""
    import multiprocessing as mp

    workers = workers or (os.cpu_count() or 1)
    ctx = mp.get_context("spawn")             # main.py:27
    t0 = time.perf_counter()
    with ctx.Pool(processes=workers) as pool:
        res = pool.map(_mcts_worker, [(moves, sims, loggers_on, 1000 + i) for i in range(workers)])
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return {"value": total / busy, "unit": "sims/s", "cores": workers, "sims": total, "seconds_search": busy, "seconds_wall_incl_spawn": wall,
            "per_core": total / busy / workers, "loggers": "enabled (as shipped)" if loggers_on else "disabled",
            "what": f"MCTS.get_best_action_and_pi, default net on CPU (1 torch thread per worker), {sims} sims/move, {moves} moves per worker, "
                    f"Pool({workers}) as trainer.py:104-107"}


def measure(engine_budget_s=4.0, moves=2, sims=100, both_logger_modes=True):
    if not available():
        return {"unavailable": "baseline/_ref not staged (python baseline/stage_ref.py --src <checkout of the reference>, "
                               "or with HZ_REFERENCE_ROOT set)"}
    out = {"cores": os.cpu_count() or 1, "engine": steps_per_core(engine_budget_s)}
    out["mcts_loggers_on"] = pool_sims_per_s(moves=moves, sims=sims, loggers_on=True)
    if both_logger_modes:
        out["mcts_loggers_off"] = pool_sims_per_s(moves=moves, sims=sims, loggers_on=False)
    return out


if __name__ == "__main__":
    import json

    print(json.dumps(measure(), indent=1))
