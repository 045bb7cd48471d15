"""Komi-bisection searches (katago_b200/komi_search.py): PlayUtils::getNaiveEvenKomiHelper / adjustKomiToEven / computeLead as generators, and the
side loop that runs them on the device."""
import math
import os
import random
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from katago_b200.komi_search import KomiSearcher, adjust_komi_to_even, compute_lead, naive_even_komi


def _run(gen, oracle):
    asked = [gen.send(None)]
    while True:
        try:
            asked.append(gen.send(oracle(asked[-1])))
        except StopIteration as st:
            return st.value, asked[:-1] if False else asked


def test_generators_find_the_even_komi_of_a_synthetic_position():
    """A position in which white's lead at komi k is k - 3.2 and the win/loss value a smooth function of it: the helpers converge on 3.2 with the
    reference's sequence of queries (first the lead-sized shift, then the window around it), never asking a komi twice."""
    oracle = lambda k, even=3.2: (k - even, math.tanh((k - even) / 4.0))
    (even, _), asked = _run(naive_even_komi(7.5, 19, 19), oracle)
    assert abs(even - 3.2) < 0.01 and asked[0] == 7.5 and asked[1] == 3.0 and len(asked) == len(set(asked)) <= 6, asked
    assert all(a * 2 == round(a * 2) for a in asked)
    fair, _ = _run(adjust_komi_to_even(7.5, 19, 19, random.Random(1)), oracle)
    assert fair in (3.0, 3.5)
    lead, _ = _run(compute_lead(7.5, 19, 19), oracle)
    assert abs(lead - 4.3) < 0.01
    lead, _ = _run(compute_lead(-40.0, 9, 9), oracle)
    assert abs(lead + 43.2) < 0.01
    # a hopeless position: the window grows to its limit (32 points) and the answer stays inside the komi clip range of the board
    lead, asked = _run(compute_lead(7.5, 9, 9), lambda k: (k + 300.0, 1.0))
    assert all(abs(a) <= 20 + 81 for a in asked) and lead > 30


class _Loop:
    """The part of SelfPlay the KomiSearcher drives, with a scripted evaluator: lead(komi) = komi - even(position)."""

    def __init__(self, n):
        self.num_games, self.x, self.y, self.max_visits = n, 9, 9, 6
        self.moves = [[] for _ in range(n)]; self.komi = np.full(n, 7.5, np.float32); self.next_komi = self.komi.copy()
        self.visits = np.zeros(n, np.int32); self.loads = 0

    def set_game_setup(self, setups, also_current_games=False):
        pass

    def set_komi(self, komis, also_current_games=False):
        self.next_komi = np.array(komis, np.float32)

    def play_moves_game(self, g, moves):
        for m in moves:
            self.moves[g].append(m)
            if len(self.moves[g]) >= 2 and self.moves[g][-1] is None and self.moves[g][-2] is None:      # two passes: next game, next komi
                self.moves[g] = []; self.komi[g] = self.next_komi[g]
        self.visits[g] = 0; self.loads += 1

    def game(self, g):
        return None, dict(move_num=len(self.moves[g]))

    def run(self, waves):
        self.visits = np.minimum(self.visits + waves, self.max_visits)

    def root_visits(self):
        return self.visits.copy()

    def root_value_stats(self, g):
        even = 2.0 + len(self.moves[g])          # the "position" is its number of moves
        lead = float(self.komi[g]) - even
        return None, np.array([math.tanh(lead / 3.0), 0.0, lead, lead * lead, lead])


def test_komi_searcher_schedules_jobs_over_its_slots():
    loop = _Loop(3)
    ks = KomiSearcher(loop)
    got = {}
    for i in range(7):                          # more jobs than slots
        ks.submit(compute_lead(7.5, 9, 9), (9, 9, 0, 1), [(k % 9, k // 9) for k in range(i)], lambda v, i=i: got.__setitem__(i, v))
    assert ks.pending() == 7 and len(ks.running) == 3
    ks.drain()
    assert ks.pending() == 0 and sorted(got) == list(range(7))
    for i, v in got.items():
        assert abs(v - (7.5 - (2.0 + i))) < 0.05, (i, v)


def _komitable_cases():
    import gzip, json
    return json.loads(gzip.open(os.path.join(ROOT, "tests", "golden", "komitable.json.gz"), "rb").read())["cases"]


@pytest.mark.parametrize("case", _komitable_cases(), ids=lambda c: c["name"])
def test_compute_lead_lands_on_the_reference_value_given_the_reference_searches(case):
    """PlayUtils::computeLead of the unmodified reference (trained g170-b6c96 net on host cores) against `compute_lead` driven by the function the
    reference's komi bisection saw: tests/golden/komitable.json.gz holds, per position, (lead, winLoss) of PlayUtils::getWhiteScoreValues for every
    komi the board allows and the reference's own result.  The generator must reach that result to the last bit (float32, as the reference
    returns it) - i.e. bracket, bisect and interpolate exactly like getNaiveEvenKomiHelper / computeLead - asking only for rounded, clipped komis
    and never twice for the same one (scoreWLCache)."""
    table = case["table"]
    assert len(case["leads"]) >= 25
    for start, ref_lead in case["leads"].items():      # the case's own komi and ~25 more starting komis over the whole range the board allows
        start, asked = float(start), []

        def oracle(k):
            assert k == float(np.float32(k)) and 2 * k == int(2 * k) and abs(k) <= 20 + case["x"] * case["y"], k
            asked.append(k)
            return tuple(table["%.1f" % k])
        lead, _ = _run(compute_lead(start, case["x"], case["y"]), oracle)
        assert len(set(asked)) == len(asked), asked
        assert np.float32(lead) == np.float32(ref_lead), (start, lead, ref_lead, asked)
        # the even komi that adjustKomiToEven rounds is the one this lead was taken from (coarse area-scoring granularity aside)
        (naive, _), asked_naive = _run(naive_even_komi(start, case["x"], case["y"]), lambda k: tuple(table["%.1f" % k]))
        assert asked_naive == asked[:len(asked_naive)] and abs((start - naive) - lead) <= 1.0


@pytest.fixture(scope="module")
def cpp_komi_driver(tmp_path_factory):
    exe = tmp_path_factory.mktemp("komi") / "komi_table_driver"
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", ROOT, os.path.join(ROOT, "tests", "cpp", "komi_table_driver.cpp"), "-o", str(exe),
                    "-L", os.path.join(ROOT, "katago_b200"), "-lkgb200", "-lz", "-Wl,-rpath," + os.path.join(ROOT, "katago_b200")], check=True)
    return str(exe)


def test_cpp_compute_lead_lands_on_the_reference_value_too(cpp_komi_driver):
    """integration/b200_komi.h - the C++ host's twin of the generators, written as a plain function that is re-run from the top whenever an evaluation
    is missing - against the same 472 reference results: the reference's lead bit for bit, and exactly the komis, in exactly the order, that the
    Python generator asks for."""
    total = 0
    for case in _komitable_cases():
        table = case["table"]
        text = f"{case['x']} {case['y']} {len(table)}\n" + "".join(f"{k} {v[0]!r} {v[1]!r}\n" for k, v in table.items()) + "".join(f"{k}\n" for k in case["leads"])
        out = subprocess.run([cpp_komi_driver], input=text, capture_output=True, text=True, check=True).stdout.splitlines()
        assert len(out) == len(case["leads"])
        for line, (start, ref_lead) in zip(out, case["leads"].items()):
            parts = line.split()
            assert parts[0] == "lead" and parts[2] == "asked", line
            asked_py = []

            def oracle(k):
                asked_py.append(k)
                return tuple(table["%.1f" % k])
            _run(compute_lead(float(start), case["x"], case["y"]), oracle)
            assert np.float32(float(parts[1])) == np.float32(ref_lead), (case["name"], start, line)
            assert [float(v) for v in parts[3:]] == asked_py, (case["name"], start)
            total += 1
    assert total >= 470


@pytest.mark.gpu
@pytest.mark.parametrize("stream,size,prefix_len,komi,visits", [("boardstream_9x9_multisuicide.npz", 9, 12, 7.5, 6), ("boardstream_9x9_multisuicide.npz", 9, 31, 0.5, 10),
                                                               ("boardstream_19x19_multisuicide.npz", 19, 40, 7.5, 6)])
def test_lead_of_a_position_equals_the_reference_computeLead(golden_dir, stream, size, prefix_len, komi, visits):
    """PlayUtils::computeLead of the UNMODIFIED reference (its Search + NNEvaluator on libkgb200, fp32-equivalent, trained g170-b6c96 net,
    symmetry 0, no cache; its answers stored by tests/reference_runs.py) against the same computation as jobs on the device's side loop:
    the same komis are searched with the same few visits, so the interpolated lead agrees to the evaluator's rounding."""
    sys.path.insert(0, golden_dir)
    import make_search_fixtures as F
    from katago_b200 import NeuralNet, SelfPlay
    from reference_runs import reference_run
    model = os.path.join(golden_dir, "models", "g170-b6c96-s175395328-d26788732.bin.gz")
    moves = F.prefix_from_stream(stream, prefix_len)
    s = " ".join("pass" if m is None else f"{m[0]},{m[1]}" for m in moves)
    out = reference_run("kgref_driver_b200", ["computelead", model, size, size, visits, repr(komi), s])
    ref = float([ln.split()[1] for ln in out.splitlines() if ln.startswith("lead ")][0])
    lm = NeuralNet.loadModelFile(model)
    ctx = NeuralNet.createComputeContext([0], size, size, False, lm)
    h = NeuralNet.createComputeHandle(ctx, lm, 4, False, True, 0)
    kw = KomiSearcher.noiseless_kwargs(dict(cpuct_exploration=1.0, cpuct_exploration_log=0.45, cpuct_exploration_base=500.0, fpu_reduction_max=0.2, root_fpu_reduction_max=0.1))
    sp = SelfPlay(h, 4, visits, komi=7.5, multi_stone_suicide_legal=True, seed=1, debug_hold_at_max_visits=True, debug_fixed_symmetry=0, full_history_rules=True, **kw)
    ks = KomiSearcher(sp)
    got = []
    ks.submit(compute_lead(komi, size, size), (size, size, 0, 1), moves, got.append)
    ks.drain()
    print(f"{size}x{size} after {len(moves)} moves at komi {komi}, {visits} visits per search, {ks.searches} searches: lead {got[0]:.4f} (reference {ref:.4f})")
    assert abs(got[0] - ref) < 0.02, (got, ref)
    sp.free(); h.free(); ctx.free()


def test_fork_manager_picks_the_move_the_net_scores_best():
    """Play::maybeForkGame: early forks near the start, late forks anywhere; among the drawn legal moves the one with the best whiteScoreMean for
    the player to move; the pool hands positions out at random and empties."""
    from katago_b200.fork_play import ForkManager
    settings = dict(early_fork_game_prob=1.0, early_fork_game_expected_move_prop=0.05, fork_game_prob=0.0, fork_game_min_choices=3, early_fork_game_max_choices=5,
                    fork_game_max_choices=5, fork_compensate_komi_prob=0.0)
    fm = ForkManager(settings, random.Random(3))
    game = [(k % 9, k // 9) for k in range(40)]
    legal = np.ones(82, bool); legal[:10] = False
    scores = lambda moves: 0.1 * (moves[-1][0] + 9 * moves[-1][1]) if moves and moves[-1][0] >= 0 else 100.0       # white likes high positions and the pass most
    for trial in range(20):
        gen = fm.job(game, (9, 9, 0, 1), 7.5, 9)
        q = gen.send(None)
        idx = len(q["moves"])
        assert q["moves"] == game[:idx] and q["komi"] == 7.5 and idx <= 39
        asked, answer = [], dict(legal=legal, nn_score_mean=0.0, lead=0.0, win_loss=0.0)
        try:
            while True:
                q = gen.send(answer)
                asked.append(q["moves"][-1])
                assert q["moves"][:-1] == game[:idx] and (q["moves"][-1] == (-1, -1) or q["moves"][-1][1] * 9 + q["moves"][-1][0] >= 10)
                answer = dict(legal=legal, nn_score_mean=scores(q["moves"]), lead=0.0, win_loss=0.0)
        except StopIteration as st:
            fork = st.value
        assert 3 <= len(asked) <= 5 and fork[:-1] == game[:idx]
        best = (min if idx % 2 == 0 else max)(asked, key=lambda m: scores([m]))          # black (even index) wants white's score low
        assert scores([fork[-1]]) == scores([best])
        fm.add(fork, (9, 9, 0, 1), 7.5)
    assert fm.forks_made == 20 and len(fm.pool) == 20
    seen = [fm.pop() for _ in range(20)]
    assert fm.pop() is None and len({tuple(f["moves"]) for f in seen}) >= 10 and all(f["setup"] == (9, 9, 0, 1) for f in seen)
    off = ForkManager(dict(settings, early_fork_game_prob=0.0), random.Random(1))
    assert not off.enabled and off.job(game, (9, 9, 0, 1), 7.5, 9) is None


def test_forking_move_distribution_and_side_position_bookkeeping():
    """chooseRandomForkingMove: never the banned move, mostly policy-proportional; and the recorder's bookkeeping of side positions that are still being
    searched when their game ends (the game is written once they are back, with them attached)."""
    from katago_b200.game_recorder import choose_random_forking_move
    pol = np.full(26, -1.0, np.float32)
    pol[[3, 7, 11, 25]] = [0.6, 0.3, 0.1, 0.0]                      # three moves with mass, a legal pass with none
    r = random.Random(5)
    draws = [choose_random_forking_move(pol, 5, r, ban_pos=7) for _ in range(4000)]
    assert 7 not in draws and set(draws) <= {3, 11, 25}
    f3 = draws.count(3) / 4000
    # 70 %: 0.6 / 0.7 = 0.857; 25 %: sqrt weights 0.775 / (0.775 + 0.316) = 0.710; 5 %: uniform over {3, 11, 25} = 1/3
    assert abs(f3 - (0.70 * 0.857 + 0.25 * 0.710 + 0.05 / 3)) < 0.03, f3
    assert 0 < draws.count(25) / 4000 < 0.04                         # the mass-less pass only through the uniform 5 %
    assert choose_random_forking_move(np.full(5, -1.0, np.float32), 2, r, ban_pos=0) is None
