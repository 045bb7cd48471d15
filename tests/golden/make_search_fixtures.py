"""Generates tests/golden/searchfake.npz from the REFERENCE Search (oracle/_ref/kgref_driver searchfake ...).

The reference's MCTS (search/search.cpp, searchexplorehelpers.cpp, searchupdatehelpers.cpp) runs single-threaded with a
deterministic hash-based fake net as its NeuralNet backend (oracle/ref_driver.cpp), restricted to the SearchParams subset
the device loop implements (DESIGN.md §8).  Stored per case: the move prefix, maxVisits, and for the root: each child's
visit count, the post-processed NN policy and the utility average.  The device loop is given the same fake net
(debug_fake_nn) and must reproduce the visit counts."""
import json, os, subprocess, sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DRIVER = os.path.join(HERE, "..", "..", "oracle", "_ref", "kgref_driver")
MODEL = os.path.join(HERE, "models", "torchref_b2c16.bin.gz")   # only supplies a ModelDesc (version 15) to NNEvaluator


def prefix_from_stream(name, n):
    d = np.load(os.path.join(HERE, name))
    mv = d["moves"][:n]
    out = []
    for x, y, _ in mv:
        out.append(None if x < 0 else (int(x), int(y)))
    for i, (a, b) in enumerate(zip(out, out[1:])):
        if a is None and b is None:      # two passes in a row would end the game: stop the prefix before the second one
            return out[:i + 1]
    return out


SCORE_KEYS = ("staticScoreUtilityFactor", "dynamicScoreUtilityFactor", "dynamicScoreCenterZeroWeight", "dynamicScoreCenterScale")
# the search part of cpp/configs/training/selfplay8mainb18.cfg that the device loop implements
SELFPLAY8B18 = {"staticScoreUtilityFactor": 0.05, "dynamicScoreUtilityFactor": 0.30, "dynamicScoreCenterZeroWeight": 0.25,
                "dynamicScoreCenterScale": 0.50, "cpuctExploration": 1.05, "cpuctExplorationLog": 0.28, "fpuReductionMax": 0.2,
                "rootFpuReductionMax": 0.0, "valueWeightExponent": 0.5, "fpuParentWeightByVisitedPolicy": 1,
                "fpuParentWeightByVisitedPolicyPow": 2.0, "rootDesiredPerChildVisitsCoeff": 2}


LCB = {"useLcbForSelection": 1, "lcbStdevs": 5.0, "minVisitPropForLCB": 0.15, "useNonBuggyLcb": 1, "chosenMoveSubtract": 0, "chosenMovePrune": 1}
BIAS = {"subtreeValueBiasFactor": 0.30, "subtreeValueBiasWeightExponent": 0.8}


def run(X, Y, visits, moves, score=None, driver=None, model=None, env=None, frame=None, answer=None):
    """answer(args, env) -> the driver's stdout, in place of running it (tests: the stored answers of tests/reference_runs.py)."""
    s = " ".join("pass" if m is None else f"{m[0]},{m[1]}" for m in moves)
    if score is None:
        score = {}
    elif not isinstance(score, dict):
        score = dict(zip(SCORE_KEYS, score))
    extra = [f"{k}={float(v)!r}" for k, v in score.items() if k != "fullHistoryRules"]
    if frame is not None:      # the evaluator's frame is frame x frame, the board X x Y in its corner: positions are y * frame + x
        env = dict(env or {}, KGREF_NN_LEN=str(frame))
    args = ["searchfake", model or MODEL, str(X), str(Y), str(visits), s] + extra
    if answer is not None:
        out = answer(args, env)
    else:
        out = subprocess.run([driver or DRIVER] + args, capture_output=True, text=True, check=True, env=(dict(os.environ, **env) if env else None)).stdout
    bx = X
    if frame is not None:
        X = Y = frame
    v = np.zeros(X * Y + 1, np.int32); u = np.zeros(X * Y + 1, np.float64); pol = None; root = None; center = 0.0
    psv = np.full(X * Y + 1, -1.0, np.float64); threadseed = ""
    cstats = np.zeros((X * Y + 1, 5), np.float64); rstats = np.zeros(5, np.float64)
    for ln in out.splitlines():
        f = ln.split()
        if f[0] == "rootvisits":
            root = (int(f[1]), float(f[3]))
        elif f[0] == "threadseed":
            threadseed = ln.split(" ", 1)[1]
        elif f[0] == "playselection":
            for j in range(2, len(f), 3):
                x, y = int(f[j]), int(f[j + 1])
                psv[X * Y if x < 0 else y * X + x] = float(f[j + 2])
        elif f[0] == "recentScoreCenter":
            center = float(f[1])
        elif f[0] == "child":
            x, y = int(f[1]), int(f[2])
            i = X * Y if x < 0 else y * X + x
            v[i] = int(f[3]); u[i] = float(f[4]); cstats[i] = [float(t) for t in f[5:10]]
        elif f[0] == "rootstats":
            rstats[:] = [float(t) for t in f[1:6]]
        elif f[0] == "policy":
            pol = np.array([float(t) for t in f[1:]], np.float32)
    return root, v, u, pol, center, psv, threadseed, cstats, rstats


# Black builds a two-eyed (pass-alive) group in the corner while White, after two stones, passes four times: Black to move, the
# opponent's last four moves are passes -> Search::isAllowedRootMove refuses Black's own eyes (0,0), (2,0) and nothing else.
PRUNE_7X7 = [(1, 0), (5, 5), (0, 1), (5, 4), (1, 1), None, (2, 1), None, (3, 0), None, (3, 1), None]
# both sides own a two-eyed corner group; Black adds four stones in the centre while White passes four times
PRUNE_9X9 = [(1, 0), (7, 8), (0, 1), (8, 7), (1, 1), (7, 7), (2, 1), (6, 7), (3, 0), (5, 8), (3, 1), (5, 7),
             (4, 4), None, (4, 3), None, (3, 4), None, (3, 3), None]


if __name__ == "__main__":
    cases = [
        (9, 9, 100, prefix_from_stream("boardstream_9x9_multisuicide.npz", 0)),
        (9, 9, 400, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12)),
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31)),
        (19, 19, 200, prefix_from_stream("boardstream_19x19_multisuicide.npz", 0)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 131)),
        (13, 7, 300, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20)),
        (5, 5, 500, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9)),
        # score utility on (a21): static, dynamic, dynamicScoreCenterZeroWeight, dynamicScoreCenterScale
        (9, 9, 500, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), (0.05, 0.30, 0.25, 0.50)),    # selfplay8mainb18.cfg
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), (0.05, 0.30, 0.25, 0.50)),
        (19, 19, 400, prefix_from_stream("boardstream_19x19_multisuicide.npz", 131), (0.3, 0.0, 0.0, 1.0)),   # SearchParams defaults
        (13, 7, 300, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), (0.1, 0.3, 0.25, 0.5)),
        (5, 5, 600, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), (0.05, 0.30, 0.25, 0.50)),      # reaches terminal nodes
        # value weighting, FPU blending, utility-stdev exploration scaling, root per-child visit floor (a19/a20 widened)
        (9, 9, 400, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), {"valueWeightExponent": 0.5}),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), {"valueWeightExponent": 0.5}),
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), SELFPLAY8B18),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), SELFPLAY8B18),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 0), SELFPLAY8B18),
        (13, 7, 500, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), SELFPLAY8B18),
        (5, 5, 600, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), SELFPLAY8B18),
        (9, 9, 500, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12),
         {"valueWeightExponent": 0.25, "cpuctUtilityStdevScale": 0.85, "cpuctUtilityStdevPrior": 0.4, "cpuctUtilityStdevPriorWeight": 2.0,
          "fpuParentWeight": 0.3, "fpuLossProp": 0.1, "rootFpuLossProp": 0.05, "staticScoreUtilityFactor": 0.1}),
        # subtree value bias (a23, tree search): entries shared by nodes reached by the same local move
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), dict(SELFPLAY8B18, **BIAS)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), dict(SELFPLAY8B18, **BIAS)),
        (19, 19, 400, prefix_from_stream("boardstream_19x19_multisuicide.npz", 0), dict(SELFPLAY8B18, **BIAS)),
        (13, 7, 500, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), dict(SELFPLAY8B18, **BIAS)),
        (5, 5, 600, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), dict(SELFPLAY8B18, **BIAS)),
        (9, 9, 500, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), {"subtreeValueBiasFactor": 0.45, "subtreeValueBiasWeightExponent": 0.5}),
        # graph search (a23): transpositions share nodes
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), {"useGraphSearch": 1}),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), {"useGraphSearch": 1}),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), {"useGraphSearch": 1}),
        (9, 9, 800, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS)),
        (13, 7, 600, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS)),
        (5, 5, 1000, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS)),
        # root policy temperature (a22), early-game interpolation by turn number
        (9, 9, 400, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), {"rootPolicyTemperature": 1.1, "rootPolicyTemperatureEarly": 1.5}),
        (19, 19, 500, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40),
         dict(SELFPLAY8B18, useGraphSearch=1, rootPolicyTemperature=1.1, rootPolicyTemperatureEarly=1.5, chosenMoveTemperatureHalflife=19, **BIAS)),
        (13, 7, 400, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), {"rootPolicyTemperature": 0.8, "chosenMoveTemperatureHalflife": 10}),
        # play selection values with LCB (a22 / §8f move choice): selfplay8mainb18.cfg and variants
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS, **LCB)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS, **LCB)),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), dict(SELFPLAY8B18, useGraphSearch=1, **BIAS, **LCB)),
        (13, 7, 500, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20),
         {"useLcbForSelection": 1, "lcbStdevs": 3.0, "minVisitPropForLCB": 0.05, "chosenMoveSubtract": 2.0, "chosenMovePrune": 3.0, "valueWeightExponent": 0.5}),
        # rootNumSymmetriesToSample (a22): the root's evaluation is the average over symmetries drawn from the search thread's Rand
        (9, 9, 400, prefix_from_stream("boardstream_9x9_multisuicide.npz", 12), {"rootNumSymmetriesToSample": 4}),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 40),
         dict(SELFPLAY8B18, useGraphSearch=1, rootNumSymmetriesToSample=4, rootPolicyTemperature=1.1, rootPolicyTemperatureEarly=1.5, **BIAS, **LCB)),
        (13, 7, 300, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), {"rootNumSymmetriesToSample": 8, "valueWeightExponent": 0.5}),
        (5, 5, 500, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), {"rootNumSymmetriesToSample": 2, "staticScoreUtilityFactor": 0.1}),
        # ko rules inside the search (a3): superko bans and repetition endings along the playout paths
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 9), {"koRule": 1}),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), dict(SELFPLAY8B18, useGraphSearch=1, koRule=2, **BIAS)),
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), dict(SELFPLAY8B18, useGraphSearch=1, koRule=1, **BIAS, **LCB)),
        (5, 5, 1000, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {"fullHistoryRules": 1, "useGraphSearch": 1}),
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 55), dict(SELFPLAY8B18, fullHistoryRules=1)),
        (5, 5, 1000, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {"fullHistoryRules": 1}),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {"koRule": 2}),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {"useGraphSearch": 1}),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {}),
        # the two root options the stock self-play configs switch on (a21 / a22): rootEndingBonusPoints (the fake net's ownership head puts about
        # half of the points beyond |0.95|) and rootPruneUselessMoves (positions with pass-alive groups reached while the opponent passed four times)
        (9, 9, 600, prefix_from_stream("boardstream_9x9_multisuicide.npz", 31), dict(SELFPLAY8B18, useGraphSearch=1, rootEndingBonusPoints=0.5, **BIAS, **LCB)),
        (19, 19, 600, prefix_from_stream("boardstream_19x19_multisuicide.npz", 131),
         dict(SELFPLAY8B18, useGraphSearch=1, rootNumSymmetriesToSample=4, rootPolicyTemperature=1.1, rootPolicyTemperatureEarly=1.5, rootEndingBonusPoints=0.5,
              rootPruneUselessMoves=1, **BIAS, **LCB)),
        (5, 5, 800, prefix_from_stream("boardstream_5x5_multisuicide.npz", 20), {"rootEndingBonusPoints": 0.5, "fullHistoryRules": 1, "staticScoreUtilityFactor": 0.1}),
        (13, 7, 500, prefix_from_stream("boardstream_13x7_nosuicide.npz", 20), dict(SELFPLAY8B18, rootEndingBonusPoints=1.0, rootNumSymmetriesToSample=2)),
        (7, 7, 400, PRUNE_7X7, dict(SELFPLAY8B18, rootPruneUselessMoves=1)),
        (7, 7, 400, PRUNE_7X7, dict(SELFPLAY8B18, useGraphSearch=1, rootPruneUselessMoves=1, rootEndingBonusPoints=0.5, rootNumSymmetriesToSample=4, **BIAS, **LCB)),
        (9, 9, 500, PRUNE_9X9, dict(SELFPLAY8B18, useGraphSearch=1, rootPruneUselessMoves=1, rootEndingBonusPoints=0.5, **BIAS, **LCB)),
        (9, 9, 500, PRUNE_9X9[:-2], dict(SELFPLAY8B18, rootPruneUselessMoves=1, rootEndingBonusPoints=0.5)),     # only three opponent passes: nothing pruned
    ]
    store = {"num_cases": len(cases)}
    for i, case in enumerate(cases):
        X, Y, visits, moves = case[:4]
        score = case[4] if len(case) > 4 else None
        root, v, u, pol, center, psv, threadseed, cstats, rstats = run(X, Y, visits, moves, score)
        store[f"c{i}_child_stats"] = cstats; store[f"c{i}_root_stats"] = rstats
        store[f"c{i}_thread_seed"] = np.array(threadseed)
        store[f"c{i}_play_selection"] = psv
        if score is not None and not isinstance(score, dict):
            score = dict(zip(SCORE_KEYS, score))
        store[f"c{i}_params"] = np.array(json.dumps(score or {}))
        store[f"c{i}_recent_score_center"] = np.float64(center)
        assert root[0] == visits and v.sum() == visits - 1, (root, v.sum())
        store[f"c{i}_shape"] = np.array([X, Y, visits], np.int32)
        store[f"c{i}_moves"] = np.array([(-1, -1) if m is None else m for m in moves], np.int8).reshape(-1, 2)
        store[f"c{i}_visits"] = v; store[f"c{i}_util"] = u; store[f"c{i}_policy"] = pol
        store[f"c{i}_root_util"] = np.float64(root[1])
        print(i, X, Y, visits, len(moves), "children", int((v > 0).sum()), "max visits", int(v.max()), "root util", root[1])
    np.savez_compressed(os.path.join(HERE, "searchfake.npz"), **store)
