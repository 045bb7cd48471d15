"""Per-turn training targets and the game recorder (SURVEY §8f rows 1-2).

CPU: the target functions of katago_b200/game_recorder.py against what the reference derives from its own finished `Search`
(tests/golden/searchtargets.npz, generator tests/golden/make_searchtargets_fixture.py).
GPU: whole games recorded from the device loop in hold mode and written as training rows."""
import os, sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from katago_b200 import game_recorder as R
from katago_b200 import npz_writer as W

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _cases():
    d = np.load(os.path.join(GOLDEN, "searchtargets.npz"))
    return d, int(d["num_cases"])


def test_value_targets_match_reference_get_node_values():
    d, n = _cases()
    for i in range(n):
        got = R.value_targets_from_root(d[f"c{i}_root_stats"])
        assert [np.float32(v) for v in got[:4]] == list(d[f"c{i}_value_targets"]), i


def test_q_targets_match_reference_extract_q_value_targets():
    d, n = _cases()
    for i in range(n):
        X = int(d[f"c{i}_shape"][0])
        q, mask = d[f"c{i}_q"], d[f"c{i}_q_mask"]
        got = R.q_targets_from_children(d[f"c{i}_child_stats"], np.where(mask, q[:, 2], 0).astype(np.int64), X)
        assert len(got) == int(mask.sum()) > 0
        for (x, y, wl, sc, v) in got:
            pos = len(mask) - 1 if x < 0 else y * X + x
            assert mask[pos] and wl == np.float32(q[pos, 0]) and sc == np.float32(q[pos, 1]) and v == int(q[pos, 2]), (i, pos)


def test_policy_surprise_and_entropies_match_reference():
    d, n = _cases()
    for i in range(n):
        got = R.policy_surprise_and_entropy(d[f"c{i}_play_selection"], d[f"c{i}_policy"])
        # the fixture's policy is printed with 9 significant digits and the sums run in child order there, position order here
        assert np.allclose(got, d[f"c{i}_surprise"], rtol=1e-9, atol=1e-12), (i, got, d[f"c{i}_surprise"])


def test_policy_target_matches_reference_extract_policy_target():
    """Including the case where one move has more than 30000 visits (everything is scaled to fit int16)."""
    d, n = _cases()
    saw_cap = False
    for i in range(n):
        X = int(d[f"c{i}_shape"][0])
        want = d[f"c{i}_policy_target"]
        got = R.policy_target_moves(d[f"c{i}_play_selection"], X)
        dense = np.full(len(want), -1, np.int32)
        for (x, y, v) in got:
            dense[len(want) - 1 if x < 0 else y * X + x] = v
        assert np.array_equal(dense, want), (i, np.flatnonzero(dense != want)[:5])
        saw_cap |= int(want.max()) == 30000
    assert saw_cap


def test_value_surprise_and_surprise_weights_match_reference_run_game():
    """Six whole games of the reference's own Play::runGame (CPU, fake net; tests/golden/make_rungame_fixtures.py): from each turn's
    value targets, raw net values and policy surprise our restatement reproduces runGame's value surprise (1e-12) and its
    surprise-weighted target weights (float32, bit for bit) - both variants of the value surprise, several weight settings."""
    import gzip, json
    games = json.loads(gzip.open(os.path.join(GOLDEN, "rungame.json.gz"), "rb").read())
    assert len(games) >= 6 and {g["useSearchValueSurprise"] for g in games} == {0, 1}
    for g in games:
        n = g["turns"]
        vs = R.compute_value_surprise_by_turn(g["valueTargets"], g["rawNN"], g["size"] ** 2, bool(g["useSearchValueSurprise"]))
        assert np.allclose(vs, g["valueSurprise"], rtol=1e-12, atol=1e-15), np.abs(np.array(vs) - np.array(g["valueSurprise"])).max()
        w = R.surprise_target_weights([1.0] * n, g["policySurprise"], g["valueSurprise"], g["policySurpriseDataWeight"], g["valueSurpriseDataWeight"])
        assert [float(x) for x in w] == [float(np.float32(x)) for x in g["targetWeightUnrounded"]]
        assert abs(float(np.sum(w, dtype=np.float64)) - n) < 1e-3          # the game's total weight is kept
        # what runGame then wrote: each weight resolved to one of its two neighbouring integers
        assert all(r in (np.floor(u), np.floor(u) + 1) for r, u in zip(g["targetWeight"], g["targetWeightUnrounded"]))


def test_resolve_target_weight_keeps_the_expectation():
    rand = W.RowRand("resolve")
    draws = [float(R.resolve_target_weight(1.3, rand)) for _ in range(4000)]
    assert set(draws) == {1.0, 2.0} and abs(np.mean(draws) - 1.3) < 0.03
    assert float(R.resolve_target_weight(-0.5, rand)) == 0.0 and float(R.resolve_target_weight(2.0, rand)) == 2.0


# ---- the recorder's host logic against a scripted stand-in for the device loop ------------------------------------------------------
class ScriptedSlots:
    """Stands in for nn_backend.SelfPlay in hold mode: every slot replays a move stream of the reference `Board` (boardstream
    fixture: moves, position after each move, area) and reports made-up but reproducible search statistics."""

    def __init__(self, stream, lengths, max_visits):
        self.s, self.lengths, self.max_visits = stream, lengths, max_visits
        self.x = self.y = int(stream["X"])
        self.num_games = len(lengths)
        self.t = [0] * self.num_games                 # moves played in the slot's current game
        self.index = [0] * self.num_games
        self.released = [False] * self.num_games
        self.last = [None] * self.num_games
        self.waves = 0

    def _board(self, t):
        return np.zeros((self.y, self.x), np.uint8) if t == 0 else self.s["colors"][t - 1]

    def _rng(self, g):
        return np.random.default_rng(1000 * self.index[g] + 37 * g + self.t[g])

    def run(self, n):
        self.waves += n
        for g in range(self.num_games):
            if not self.released[g]:
                continue
            self.released[g] = False
            t = self.t[g]
            x, y, pla = (int(v) for v in self.s["moves"][t])
            over = t + 1 >= self.lengths[g]
            area = self.s["area"][t]
            self.last[g] = dict(pos=self.x * self.y if x < 0 else y * self.x + x, xy=(x, y), game_over=over, no_result=False, hit_move_limit=over,
                                move_num=t, game_index=self.index[g], final_colors=self.s["colors"][t].copy(), final_area=area.copy(),
                                final_white_minus_black_score=float((area == 2).sum()) - float((area == 1).sum()) + 6.5)
            self.t[g] = 0 if over else t + 1
            self.index[g] += 1 if over else 0

    def root_visits(self):
        return np.full(self.num_games, self.max_visits, np.int32)

    def game(self, g):
        t = self.t[g]
        return self._board(t).copy(), dict(move_num=t, black_to_move=(t % 2 == 0), ko=-1, cap_b=0, cap_w=0, root_visits=self.max_visits + g)

    def root_row(self, g):
        b = self._board(self.t[g]).reshape(-1)
        own = 1 if self.t[g] % 2 == 0 else 2
        sp = np.zeros((self.x * self.y, 22), np.float32)
        sp[:, 0] = 1; sp[:, 1] = b == own; sp[:, 2] = b == 3 - own
        return sp, np.full(19, 0.25 * self.t[g], np.float32)

    def _children(self, g):
        r = self._rng(g)
        legal = np.append(self.s["legal_next"][self.t[g] - 1].reshape(-1) if self.t[g] else np.ones(self.x * self.y, np.uint8), 1).astype(bool)
        visits = np.where(legal & (r.random(legal.size) < 0.4), r.integers(1, 30, legal.size), 0).astype(np.int32)
        x, y, _ = self.s["moves"][self.t[g]]
        visits[self.x * self.y if x < 0 else y * self.x + x] += 5      # the move that will be played has been searched
        return r, legal, visits

    def root_children(self, g):
        r, legal, visits = self._children(g)
        pol = np.where(legal, r.random(legal.size), 0).astype(np.float32)
        pol = np.where(legal, pol / pol.sum(), -1).astype(np.float32)
        return visits, pol, np.zeros(legal.size)

    def root_value_stats(self, g):
        r, legal, visits = self._children(g)
        ch = np.zeros((legal.size, 5))
        ch[:, 0] = np.where(visits > 0, r.uniform(-1, 1, legal.size), 0); ch[:, 2] = np.where(visits > 0, r.uniform(-20, 20, legal.size), 0)
        return ch, np.array([0.2 - 0.01 * self.t[g], 0.0, 1.5 * g - 0.1 * self.t[g], 30.0, 0.0])

    def play_selection_values(self, g):
        _, _, visits = self._children(g)
        return np.where(visits > 0, visits.astype(np.float64), -1.0)

    def root_extra(self, g):
        _, _, visits = self._children(g)
        return dict(child_node_visits=visits + (visits > 0), root_nn_moments=np.array([0.1, 0.0, 2.0, 9.0, 0.0]))

    def release(self, mask=None):
        self.released = [True] * self.num_games if mask is None else [bool(m) for m in mask]

    def last_move(self, g):
        return self.last[g]


def test_recorder_applies_surprise_weights_to_finished_games():
    """PlaySettings policySurpriseDataWeight / valueSurpriseDataWeight in the recorder: a finished game's weights are the restated runGame
    weighting of its own policy surprises, value targets and raw net values; the game's total weight is kept; with a weight Rand the
    weights the writer gets are integers and the fractional ones stay available for the game record."""
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))
    sp = ScriptedSlots(stream, [15, 9], 30)
    games = []
    rec = R.GameRecorder(sp, None, 6.5, on_game=lambda g, d: games.append(d), policy_surprise_data_weight=0.5, value_surprise_data_weight=0.1,
                         weight_rand=W.RowRand("weights"))
    for _ in range(15):
        rec.step()
    assert len(games) == 2
    for d in games:
        n = len(d.moves)
        vs = d.value_surprise_by_turn
        assert len(vs) == n and all(0.0 <= v <= 1.0 for v in vs)
        want = R.surprise_target_weights([1.0] * n, d.policy_surprise_by_turn, vs, 0.5, 0.1)
        assert [float(x) for x in d.target_weight_by_turn_unrounded] == [float(x) for x in want]
        assert abs(sum(float(x) for x in want) - n) < 1e-3 and len({float(x) for x in want}) > 1
        assert all(float(r) in (np.floor(float(u)), np.floor(float(u)) + 1) for r, u in zip(d.target_weight_by_turn, want))
        assert "weight=%.2f" % float(want[0]) in W.write_sgf(d, "b", "w")


def test_recorder_refuses_configurations_that_give_no_root_row():
    """Evaluation cache on + a single root evaluation: the new root is a cache hit and the loop produces no input row for it."""
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))

    class Cfg:
        nn_cache_size_power_of_two, root_num_symmetries_to_sample, ladder_nodes_per_wave, ko_rule, multi_stone_suicide_legal = 16, 1, 0, 0, 1
    sp = ScriptedSlots(stream, [5], 10)
    sp.cfg = Cfg()
    with pytest.raises(ValueError, match="root must be evaluated"):
        R.GameRecorder(sp, None, 6.5)
    sp.cfg.root_num_symmetries_to_sample = 4
    R.GameRecorder(sp, None, 6.5)
    sp.cfg.ladder_nodes_per_wave = 256          # a ladder budget is fine: the root's row is kept on the device, not read off the last wave
    R.GameRecorder(sp, None, 6.5)
    # and at run time: a row that is not the root's is detected
    sp = ScriptedSlots(stream, [5], 10)
    rec = R.GameRecorder(sp, None, 6.5)
    rec.step()
    good = sp.root_row
    sp.root_row = lambda g: (np.roll(good(g)[0], 1, axis=0), good(g)[1])
    with pytest.raises(RuntimeError, match="did not evaluate the new root"):
        rec.step()


class UnevenSlots(ScriptedSlots):
    """Slots whose searches finish at different times: slot g needs 3 + 2 g waves per move."""

    def __init__(self, *a):
        super().__init__(*a)
        self.progress = [0] * self.num_games

    def run(self, n):
        was_released = list(self.released)
        super().run(n)
        for g in range(self.num_games):
            self.progress[g] = 0 if was_released[g] else self.progress[g] + n

    def root_visits(self):
        return np.array([self.max_visits if self.progress[g] >= 3 + 2 * g else self.progress[g] for g in range(self.num_games)], np.int32)


def test_pump_records_slots_as_they_finish():
    """Without lockstep: a slot is recorded and released as soon as its own search is finished; slow slots do not hold fast ones
    back, unreleased slots are left alone, and the games that come out are the same as under lockstep."""
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))
    lengths = [6, 6, 6]
    sp = UnevenSlots(stream, lengths, 50)
    games = []
    rec = R.GameRecorder(sp, None, 6.5, on_game=lambda g, data: games.append((g, data)))
    recorded = 0
    for _ in range(40):
        recorded += rec.pump(1)
    # slot g needs 3 + 2 g search waves per move: the fast slot has played twice as many moves as the slow one by now
    moves = [sp.index[g] * 6 + sp.t[g] for g in range(3)]
    assert recorded == rec.moves_recorded == sum(moves) and moves == [15, 10, 7]
    assert [[g for g, _ in games].count(k) for k in range(3)] == [2, 1, 1]
    lock = ScriptedSlots(stream, lengths, 50)
    ref_games = []
    rec2 = R.GameRecorder(lock, None, 6.5, on_game=lambda g, data: ref_games.append((g, data)))
    for _ in range(6):
        rec2.step()
    first = {g: d for g, d in reversed(games)}
    for g, d in ref_games:
        assert first[g].moves == d.moves and first[g].policy_targets_by_turn == d.policy_targets_by_turn
        assert all(np.array_equal(a, b) for a, b in zip(first[g].boards_by_turn, d.boards_by_turn))


class _JobSink:
    """Stands in for komi_search.KomiSearcher: keeps what the recorder submits; the test answers the jobs when and in the order it likes."""

    def __init__(self):
        self.jobs = []

    def submit(self, gen, setup, moves, on_done):
        self.jobs.append(dict(gen=gen, setup=tuple(setup), moves=list(moves), on_done=on_done))


def test_recorder_holds_a_finished_game_until_its_lead_and_side_jobs_are_back():
    """Host logic only (no GPU).  With estimateLeadProb the drawn turns of a finished game get a computeLead job for the position BEFORE that turn's
    move (play.cpp:2290-2324) and the game is written when the last answer is in - the slot plays on meanwhile and a later game may overtake it;
    the answers land in the turns' value targets as (hasLead, lead).  With side positions (play.cpp:1846-1860) a job carries the game so far plus a
    forking move that is not the move played; a finished game also waits for those, and the searched positions become the game's side positions."""
    import random
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))
    sp = ScriptedSlots(stream, [5], 50)
    lead_jobs, side_jobs, games = _JobSink(), _JobSink(), []
    rec = R.GameRecorder(sp, None, 6.5, on_game=lambda g, data: games.append(data), lead_estimator=lead_jobs, estimate_lead_prob=0.6, lead_rand=random.Random(1),
                         side_searcher=side_jobs, side_position_prob=0.7)
    moves = [tuple(int(v) for v in stream["moves"][t][:2]) for t in range(5)]
    for _ in range(5):
        rec.step()
    # the first game (A) is over: nothing is written while its jobs are out
    assert games == [] and rec.games_written == 0 and rec.games_waiting_for_lead == 1
    lead_a, side_a = list(lead_jobs.jobs), list(side_jobs.jobs)
    assert 1 <= len(lead_a) <= 5 and all(j["setup"] == (9, 9, 0, 1) for j in lead_a)
    turns = [len(j["moves"]) for j in lead_a]
    assert turns == sorted(set(turns)) and all(j["moves"] == moves[:t] for j, t in zip(lead_a, turns))      # the position before turn t's move
    assert 1 <= len(side_a) <= 4                      # (never after the move that ended the game)
    for j in side_a:                                   # the game up to some turn, then ONE other move than the one played there
        q = j["gen"].send(None)
        n = len(q["moves"]) - 1
        assert q["komi"] == 6.5 and q["moves"][:n] == moves[:n] and tuple(q["moves"][n]) != moves[n] and j["setup"] == (9, 9, 0, 1)
    # all but one lead answer of A, in reverse order: still waiting
    for k, j in enumerate(reversed(lead_a[1:])):
        j["on_done"](10.0 + k)
    assert games == [] and rec.games_waiting_for_lead == 1
    # the slot plays on: its second game (B) ends, and waits as well
    for _ in range(5):
        rec.step()
    lead_b, side_b = lead_jobs.jobs[len(lead_a):], side_jobs.jobs[len(side_a):]
    assert rec.games_waiting_for_lead == (2 if (lead_b or side_b) else 1)

    def answer_side(j, started):
        side_loop = ScriptedSlots(stream, [30], 50)            # a side loop whose slot holds some searched position: read like a game turn
        side_loop.t[0] = 3
        if not started:
            j["gen"].send(None)
        try:
            j["gen"].send(dict(lead=0.0, win_loss=0.0, nn_score_mean=0.0, legal=None, loop=side_loop, slot=0))
        except StopIteration as st:
            j["on_done"](st.value)
    # B's jobs come back first: B overtakes A
    for j in side_b:
        answer_side(j, False)
    for j in lead_b:
        j["on_done"](1.5)
    assert len(games) == 1 and games[0].game_hash != rec.game_hash_fn(0, 0) and rec.games_waiting_for_lead == 1
    b = games[0]
    assert len(b.side_positions) == len(side_b) and [len(v) > 4 and v[4] == 1 for v in b.white_value_targets_by_turn[:5]].count(True) == len(lead_b)
    # A: its side positions, then the last lead answer
    for j in side_a:
        answer_side(j, True)
    assert len(games) == 1
    lead_a[0]["on_done"](-3.25)
    assert len(games) == 2 and rec.games_waiting_for_lead == 0 and rec.games_written == 2
    a = games[1]
    assert a.game_hash == rec.game_hash_fn(0, 0) and a.moves == moves
    for t in range(5):
        v = a.white_value_targets_by_turn[t]
        if t in turns:
            want = -3.25 if t == turns[0] else 10.0 + list(reversed(turns[1:])).index(t)
            assert v[4] == 1 and v[5] == np.float32(want), (t, v)
        else:
            assert len(v) < 5 or v[4] == 0
    assert len(a.side_positions) == len(side_a) and all(isinstance(x, W.SidePosition) for x in a.side_positions)
    assert all(x.turn_idx >= 1 and x.unreduced_num_visits == 50 and x.next_player == 2 for x in a.side_positions)


class LimitedSlots(ScriptedSlots):
    """ScriptedSlots with the device's per-root search limits (kgb_selfplay_set_next_search_limits): a root's budget and plain flag are the ones handed
    over for "after this slot's next move" - entry 0 when the game goes on, entry 1 when a new game starts."""

    def __init__(self, stream, lengths, max_visits):
        super().__init__(stream, lengths, max_visits)
        n = self.num_games
        self.budget, self.plain = np.full(n, max_visits, np.int32), np.zeros(n, np.uint8)
        self.next_budget, self.next_plain = np.full((n, 2), max_visits, np.int32), np.zeros((n, 2), np.uint8)
        self.roots = [[] for _ in range(n)]           # (game index, move number, budget, plain) of every root the slot has searched

    def set_next_search_limits(self, visits2, plain2=None, also_current_roots=False):
        self.next_budget = np.array(visits2, np.int32).reshape(self.num_games, 2)
        self.next_plain = np.zeros((self.num_games, 2), np.uint8) if plain2 is None else np.array(plain2, np.uint8).reshape(self.num_games, 2)
        if also_current_roots:
            self.budget, self.plain = self.next_budget[:, 0].copy(), self.next_plain[:, 0].copy()

    def search_limits(self):
        return self.budget.copy(), self.plain.copy()

    def root_visits(self):
        return self.budget.copy()

    def run(self, n):
        moving = [g for g in range(self.num_games) if self.released[g]]
        for g in moving:
            self.roots[g].append((self.index[g], self.t[g], int(self.budget[g]), int(self.plain[g])))
        super().run(n)
        for g in moving:
            k = 1 if self.last[g]["game_over"] else 0
            self.budget[g], self.plain[g] = self.next_budget[g, k], self.next_plain[g, k]


def test_recorder_hands_search_limits_over_one_root_ahead():
    """Host logic only (no GPU).  Cheap searches (play.cpp:1093-1223): the limits of a root are drawn while the slot's PREVIOUS move is recorded and
    handed to the device for "the root after the next move" - once for the game going on, once for a new game.  Every recorded turn's target weight
    and cheap flag must describe the search the device really ran for that root: a cheap turn has cheapSearchVisits visits and the cheap weight,
    any other the full budget and weight 1; an unrecorded cheap search (weight 0) runs with a plain root."""
    import random
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))
    for cheap_weight in (0.25, 0.0):
        sp = LimitedSlots(stream, [7, 4, 11], 50)
        games = []
        ps = dict(cheap_search_prob=0.4, cheap_search_visits=12, cheap_search_target_weight=cheap_weight)
        rec = R.GameRecorder(sp, None, 6.5, on_game=lambda g, data: games.append((g, data)), play_settings=ps, limits_rand=random.Random(11))
        for _ in range(40):
            rec.pump(1)
        assert len(games) >= 12
        seen = {g: 0 for g in range(3)}
        cheap_turns = total = 0
        for g, data in games:
            n = len(data.moves)
            roots = sp.roots[g][seen[g]:seen[g] + n]
            seen[g] += n
            assert [r[1] for r in roots] == list(range(n)) and len({r[0] for r in roots}) == 1          # this game's roots, in order
            for t, (_, _, budget, plain) in enumerate(roots):
                w = data.target_weight_by_turn[t]
                total += 1
                if budget == 12:
                    cheap_turns += 1
                    assert w == np.float32(cheap_weight) and plain == (1 if cheap_weight == 0.0 else 0), (g, t, w, plain)
                else:
                    assert budget == 50 and w == 1.0 and plain == 0, (g, t, budget, w, plain)
        assert 0.25 < cheap_turns / total < 0.55, (cheap_turns, total)


def test_recorder_assembles_finished_games_from_scripted_slots():
    """Host logic only (no GPU): three slots replaying reference move streams of different lengths.  Every finished game carries the
    scripted moves, positions, per-turn targets and final area; rows reach the writer game by game; slots restart independently."""
    stream = np.load(os.path.join(GOLDEN, "boardstream_9x9_multisuicide.npz"))
    lengths = [12, 7, 20]
    sp = ScriptedSlots(stream, lengths, 50)
    flushed, games = [], []
    writer = W.TrainingDataWriter(None, 100000, 1.0, 9, "scripted", on_flush=lambda b: flushed.append({k: v[:b.cur_rows].copy() for k, v in b.arrays.items()}))
    rec = R.GameRecorder(sp, writer, 6.5, on_game=lambda g, data: games.append((g, data)))
    for _ in range(21):
        rec.step()
    writer.flush_if_nonempty()
    # 21 moves per slot: slot 0 finishes 1 game (12 moves), slot 1 three (7 each), slot 2 one (20)
    assert [g for g, _ in games] == [1, 0, 1, 2, 1] and rec.games_written == 5 and rec.moves_recorded == 63
    rows = flushed[0]
    assert rows["globalTargetsNC"].shape[0] == 7 + 12 + 7 + 20 + 7 == writer.row_count
    at = 0
    for g, data in games:
        n = lengths[g]
        assert data.moves == [tuple(int(v) for v in stream["moves"][t][:2]) for t in range(n)]
        assert data.hit_turn_limit and not data.end_finished and not data.end_no_result
        assert (data.boards_by_turn[0] == 0).all() and all(np.array_equal(data.boards_by_turn[t + 1], stream["colors"][t].reshape(-1)) for t in range(n))
        assert np.array_equal(data.final_ownership, stream["area"][n - 1].reshape(-1)) and data.final_full_area is data.final_ownership
        score = float((stream["area"][n - 1] == 2).sum()) - float((stream["area"][n - 1] == 1).sum()) + 6.5
        assert data.white_value_targets_by_turn[-1][:4] == (1.0 if score > 0 else 0.0, 0.0 if score > 0 else 1.0, 0.0, np.float32(score))
        for t in range(n):
            assert data.next_player_by_turn[t] == 1 + t % 2 and data.target_weight_by_turn[t] == 1.0
            moves, visits = data.policy_targets_by_turn[t]
            assert visits == 50 + g and tuple(data.moves[t]) in {(x, y) for x, y, _ in moves}
            assert data.white_value_targets_by_turn[t][3] == np.float32(1.5 * g - 0.1 * t)
            assert data.nn_raw_stats_by_turn[t][:2] == (0.1, 2.0)
            assert all(v >= 2 for *_, v in data.white_q_value_targets_by_turn[t])     # node visits, not edge visits
            # the row written for this turn: the slot's input row of that position, the turn index, the game's outcome
            assert rows["globalInputNC"][at + t, 0] == np.float32(0.25 * t) and rows["globalTargetsNC"][at + t, 51] == t
            assert rows["globalTargetsNC"][at + t, 52] == 1.0 and rows["globalTargetsNC"][at + t, 62] == 0.0       # hit the move limit, not finished
            planes = np.unpackbits(rows["binaryInputNCHWPacked"][at + t], axis=1)[:, :81]
            assert np.array_equal(planes[1], (data.boards_by_turn[t] == data.next_player_by_turn[t]).astype(np.uint8))
        assert len({data.game_hash for _, data in games}) == len(games)
        sgf = W.write_sgf(data, "b", "w")          # the record of a game cut off by the move limit: no result tag, one node per move
        assert sgf.startswith("(;FF[4]GM[1]SZ[9]PB[b]PW[w]HA[0]KM[6.5]RU[koSIMPLEscoreAREAtaxNONEsui1]C[startTurnIdx=0,") and sgf.count(";") == n + 1 and "RE[" not in sgf
        at += n


# ---- the C++ recorder + the reference's writer against the Python recorder + writer, both fed by the same CPU mock of the ABI ----------
class ReplaySlots:
    """nn_backend.SelfPlay as the mock library (tests/mock/kgb200_mock.cpp) behaved in a finished run: replays its JSON-lines log."""

    def __init__(self, log_path, num_games, size, max_visits):
        import json
        self.x = self.y = size
        self.num_games, self.max_visits = num_games, max_visits
        self.queues = [[] for _ in range(num_games)]
        for ln in open(log_path):
            ev = json.loads(ln)
            self.queues[ev["slot"]].append(ev)
        self.root = [q.pop(0) for q in self.queues]
        self.last = [None] * num_games
        self.released = [False] * num_games

    def run(self, n):
        for g in range(self.num_games):
            if self.released[g] and self.queues[g]:
                self.released[g] = False
                self.last[g] = self.queues[g].pop(0); assert self.last[g]["ev"] == "move"
                if self.queues[g]:               # (a log of a single game ends with its last move)
                    self.root[g] = self.queues[g].pop(0); assert self.root[g]["ev"] == "root"

    def release(self, mask=None):
        self.released = [True] * self.num_games

    def root_visits(self):
        return np.full(self.num_games, self.max_visits, np.int32)

    def game(self, g):
        r = self.root[g]
        return np.array(r["colors"], np.uint8).reshape(self.y, self.x), dict(move_num=r["move_num"], black_to_move=bool(r["black_to_move"]), ko=-1, cap_b=0,
                                                                          cap_w=0, root_visits=r.get("root_visits", self.max_visits + g))

    def root_row(self, g):
        r = self.root[g]
        return np.array(r["row_spatial"], np.float32).reshape(self.x * self.y, 22), np.array(r["row_global"], np.float32)

    def root_children(self, g):
        r = self.root[g]
        return np.array(r["edge_visits"], np.int32), np.array(r["policy"], np.float32), np.zeros(len(r["policy"]))

    def root_value_stats(self, g):
        r = self.root[g]
        return np.array(r["child_stats"]).reshape(-1, 5), np.array(r["root_stats"])

    def play_selection_values(self, g):
        return np.array(self.root[g]["psv"])

    def root_extra(self, g):
        return dict(child_node_visits=np.array(self.root[g]["node_visits"], np.int32), root_nn_moments=np.array(self.root[g]["root_nn"]))

    def last_move(self, g):
        m = self.last[g]
        pos, fl = m["pos"], m["flags"]
        n = self.x * self.y
        return dict(pos=pos, xy=(-1, -1) if pos == n else (pos % self.x, pos // self.x), game_over=bool(fl & 1), no_result=bool(fl & 2), hit_move_limit=bool(fl & 4),
                    move_num=m["move_num"], game_index=m["game_index"], game_hash=m.get("game_hash"), final_white_minus_black_score=float(m["score"]),
                    final_colors=np.array(m["final_colors"] or [0] * n, np.uint8), final_area=np.array(m["final_area"] or [0] * n, np.uint8))


@pytest.mark.parametrize("size,ko_rule,komi,max_moves", [(9, 0, 6.5, 40), (5, 1, 7.0, 60)])
def test_cpp_recorder_against_python_recorder_on_scripted_slots(tmp_path, size, ko_rule, komi, max_moves):
    """No GPU: oracle/ref_record_driver.cpp (integration/b200record.h + the reference's own TrainingDataWriter) linked against a CPU mock
    of the recording ABI that plays random legal games on the reference's Board (oracle/_ref/kgref_record_mock; tests/reference_runs.py).
    The C++ recorder's own checks (legality, game end, final score and area) ran on every move; its rows - planes recomputed by the
    reference - must equal the rows the Python recorder and writer produce from the mock's log: input planes bit for bit, integer
    targets exactly, floats to the text sink's 6 digits."""
    import ctypes
    from katago_b200.nn_backend import SelfplayConfig
    from reference_runs import reference_run
    from test_npz_writer import _parse_text_dump
    G, V, NUM = 3, 20, 5
    c = SelfplayConfig()
    c.num_games, c.max_visits, c.max_moves, c.multi_stone_suicide_legal, c.komi, c.seed = G, V, max_moves, 1, komi, 5 + size
    c.debug_hold_at_max_visits, c.draw_equivalent_wins_for_white, c.ko_rule, c.full_history_rules = 1, 0.5, ko_rule, 1
    (tmp_path / "cfg.bin").write_bytes(ctypes.string_at(ctypes.addressof(c), ctypes.sizeof(c)))
    (tmp_path / "model.bin").write_bytes(b"unused")
    log = tmp_path / "log.jsonl"
    reference_run("kgref_record_mock", [tmp_path / "model.bin", size, tmp_path / "cfg.bin", NUM, tmp_path / "rows.txt"], env={"KGB_MOCK_LOG": log})
    want = _parse_text_dump((tmp_path / "rows.txt").read_text())
    assert len(want) == 1

    sp = ReplaySlots(str(log), G, size, V)
    sp.cfg = c
    got, games = [], []
    writer = W.TrainingDataWriter(None, 4096, 1.0, size, "recorder-test", on_flush=lambda b: got.append({k: v[:b.cur_rows].copy() for k, v in b.arrays.items()}))

    class FirstGames:
        def write_game(self, data):
            if len(games) < NUM:
                writer.write_game(data)
            games.append(data)
    rec = R.GameRecorder(sp, FirstGames(), komi)
    while len(games) < NUM:
        rec.step()
    writer.flush_if_nonempty()
    fw, fg = want[0], got[0]
    n = len(fw["globalTargetsNC"])
    assert n == fg["globalTargetsNC"].shape[0] == sum(len(d.moves) for d in games[:NUM]) > 0
    assert [bytes.fromhex(x) for x in fw["binaryInputNCHWPacked"]] == [fg["binaryInputNCHWPacked"][i].tobytes() for i in range(n)]
    for name in ("policyTargetsNCMove", "scoreDistrN", "valueTargetsNCHW", "qValueTargetsNCMove"):
        a = np.stack(fw[name]).astype(np.int64)
        b = fg[name].reshape(n, -1).astype(np.int64)
        assert np.array_equal(a, b), (name, np.argwhere(a != b)[:5])
    for name in ("globalInputNC", "globalTargetsNC"):
        a = np.stack(fw[name])
        b = fg[name].reshape(n, -1).astype(np.float64)
        assert np.allclose(a, b, rtol=2e-5, atol=1e-30), (name, np.argwhere(~np.isclose(a, b, rtol=2e-5, atol=1e-30))[:5])
    assert any(d.end_finished for d in games[:NUM]) or size == 9        # the small board also sees games that end by passes


@pytest.mark.parametrize("size,visits,max_moves,seed,psw,vsw", [(9, 40, 50, 3, 0.5, 0.1), (7, 60, 200, 12, 0.3, 0.2), (13, 25, 70, 5, 0.0, 0.0)])
def test_recorder_chain_against_a_whole_reference_selfplay_game(tmp_path, size, visits, max_moves, seed, psw, vsw):
    """The whole host chain against the reference's own self-play: `kgref_driver rungame` plays a game with Play::runGame (CPU, fake
    net), logs what the device loop's getters would have exposed after every search, and lets the reference's TrainingDataWriter write
    the FinishedGameData runGame produced.  The Python recorder, fed only with that log, must arrive at the same rows: per-turn
    targets, game-end targets, surprise weights (left fractional on both sides, so the writers' identically seeded Rands decide the
    extra rows) and every addRow column.  Two documented differences: the Q targets are listed in position order here and in child
    creation order there, so their stochastic rounding may differ by one unit; and the three "raw net statistics" columns come from a
    separate evaluation in the reference.  The driver's log and rows are stored (tests/reference_runs.py)."""
    from reference_runs import reference_run
    from test_npz_writer import _parse_text_dump
    log, rows = tmp_path / "slot.log", tmp_path / "rows.txt"
    reference_run("kgref_driver", ["rungame", os.path.join(GOLDEN, "models", "torchref_b2c16.bin.gz"), size, visits, max_moves, seed, psw, vsw, 0, log, rows])
    want = _parse_text_dump(rows.read_text())
    assert len(want) == 1
    sp = ReplaySlots(str(log), 1, size, visits)
    got = []
    writer = W.TrainingDataWriter(None, 100000, 1.0, size, "chain-test", on_flush=lambda b: got.append({k: v[:b.cur_rows].copy() for k, v in b.arrays.items()}))
    rec = R.GameRecorder(sp, writer, 6.5, policy_surprise_data_weight=psw, value_surprise_data_weight=vsw,
                         game_hash_fn=lambda slot, index: tuple(sp.last[slot]["game_hash"]))
    while rec.games_written < 1:
        rec.step()
    writer.flush_if_nonempty()
    fw, fg = want[0], got[0]
    n = len(fw["globalTargetsNC"])
    assert n == fg["globalTargetsNC"].shape[0] > 0
    assert [bytes.fromhex(x) for x in fw["binaryInputNCHWPacked"]] == [fg["binaryInputNCHWPacked"][i].tobytes() for i in range(n)]
    for name in ("policyTargetsNCMove", "scoreDistrN", "valueTargetsNCHW"):
        a = np.stack(fw[name]).astype(np.int64)
        b = fg[name].reshape(n, -1).astype(np.int64)
        assert np.array_equal(a, b), (name, np.argwhere(a != b)[:5])
    qa = np.stack(fw["qValueTargetsNCMove"]).astype(np.int64).reshape(n, 3, -1)
    qb = fg["qValueTargetsNCMove"].astype(np.int64)
    assert np.array_equal(qa[:, 2], qb[:, 2])                               # visits: exact
    assert np.abs(qa[:, :2] - qb[:, :2]).max() <= 1                         # stochastically rounded win/loss and score: same value up to the rounding draw
    assert (qa[:, :2] != qb[:, :2]).mean() < 0.5
    for name in ("globalInputNC", "globalTargetsNC"):
        a = np.stack(fw[name])
        b = fg[name].reshape(n, -1).astype(np.float64)
        if name == "globalTargetsNC":
            a, b = np.delete(a, [57, 58, 59], axis=1), np.delete(b, [57, 58, 59], axis=1)
        assert np.allclose(a, b, rtol=2e-5, atol=1e-30), (name, np.argwhere(~np.isclose(a, b, rtol=2e-5, atol=1e-30))[:8])


# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ko_rule,graph,mode", [(0, True, "step"), (1, False, "step"), (0, True, "pump"), (1, True, "pump")])
def test_recorder_turns_device_games_into_training_rows(tmp_path, tmp_models, ko_rule, graph, mode):
    """Games of the device loop (9x9, deterministic fake net, selfplay8mainb18-style search) recorded move by move in hold mode:
    the recorded moves replay to the recorded boards (device board replay), the final area / score / outcome targets agree with
    each other, and the written .npz rows carry the positions, policy targets and outcome of the games they came from.
    mode "pump" = per-game release (every game is recorded and released as soon as ITS search is finished, the others keep searching),
    with a ladder budget per wave on: the root's input row comes from the device-kept copy, not from the last wave."""
    from katago_b200.nn_backend import NeuralNet, SelfPlay, board_replay
    lm = NeuralNet.loadModelFile(tmp_models["tiny_reg"])
    L, G, V = 9, 6, 48
    ctx = NeuralNet.createComputeContext([0], L, L, True, lm)
    h = NeuralNet.createComputeHandle(ctx, lm, G, False, True, 0)
    komi = 7.0 if ko_rule else 6.5
    sp = SelfPlay(h, G, V, komi=komi, seed=11, max_moves=70, debug_fake_nn=True, debug_hold_at_max_visits=True, use_graph_search=graph,
                  value_weight_exponent=0.5, static_score_utility_factor=0.05, dynamic_score_utility_factor=0.3,
                  dynamic_score_center_zero_weight=0.25, dynamic_score_center_scale=0.5, use_play_selection=True, use_lcb_for_selection=True,
                  use_non_buggy_lcb=True, lcb_stdevs=5.0, min_visit_prop_for_lcb=0.15, chosen_move_temperature=0.15,
                  chosen_move_temperature_early=0.75, root_noise_enabled=True, root_dirichlet_noise_total_concentration=10.83,
                  root_dirichlet_noise_weight=0.25, ko_rule=ko_rule, full_history_rules=True,
                  ladder_nodes_per_wave=(6 if mode == "pump" else 0))
    games = []
    writer = W.TrainingDataWriter(str(tmp_path), 4096, 1.0, L, "recorder-test")    # one file: rows stay in write order
    rec = R.GameRecorder(sp, writer, komi, on_game=lambda g, data: games.append((g, data)))
    steps = 0
    if mode == "step":
        while len(games) < G and steps < 80:
            rec.step()
            steps += 1
        st = sp.stats()
        assert st["total_moves"] == steps * G            # hold / release: exactly one move per game and step
    else:
        if ko_rule == 0:
            sp.random_openings(12)                       # games at different stages: their searches finish in different waves
            rec = R.GameRecorder(sp, writer, komi, on_game=lambda g, data: games.append((g, data)))
        fresh = lambda: sum(1 for _, d in games if (d.boards_by_turn[0] == 0).all())
        while (len(games) < G or fresh() < 2) and steps < 6000:
            rec.pump(5)
            steps += 1
        assert sp.stats()["total_moves"] == rec.moves_recorded + (sp.stats()["total_moves"] - rec.moves_recorded)   # bookkeeping only
    all_games = list(games)                              # in write order
    if mode == "pump" and ko_rule == 0:
        games = [(g, d) for g, d in games if (d.boards_by_turn[0] == 0).all()]     # games that began inside the recording (not from an opening)
    assert len(games) >= (G if mode == "step" else 2), (len(games), steps)
    writer.flush_if_nonempty()

    total_rows = sum(len(d.moves) for _, d in all_games)
    for g, data in games:
        n = len(data.moves)
        assert n == len(data.target_weight_by_turn) and len(data.boards_by_turn) == n + 1 and len(data.white_value_targets_by_turn) == n + 1
        # the recorded moves reproduce the recorded boards, final position included
        mv = np.array([[(x, y, data.next_player_by_turn[t]) for t, (x, y) in enumerate(data.moves)]], np.int8)
        rep = board_replay(L, L, mv, True)
        for t in range(n):
            assert np.array_equal(rep["colors"][0, t].reshape(-1), data.boards_by_turn[t + 1]), (g, t)
        assert (data.boards_by_turn[0] == 0).all()
        assert [p for p in data.next_player_by_turn] == [1 + (t % 2) for t in range(n)]
        # outcome: area of the final position (every flag on) as replayed == the area the loop scored
        if not data.end_no_result:
            area = rep["area"][0, n - 1].reshape(-1)
            assert np.array_equal(area, data.final_ownership)
            score = float((area == 2).sum()) - float((area == 1).sum()) + komi
            last = data.white_value_targets_by_turn[-1]
            adj = (data.draw_equivalent_wins_for_white - 0.5) if float(int(komi)) == komi else 0.0
            assert last[3] == np.float32(score + adj) and last[0] == (1.0 if score > 0 else 0.0 if score < 0 else 0.5)
        assert data.hit_turn_limit == (n >= 70 and not data.end_finished) and (data.end_finished or data.hit_turn_limit)
        for t in range(n):
            win, loss, nores, score = data.white_value_targets_by_turn[t][:4]
            assert 0 <= win <= 1 and 0 <= loss <= 1 and abs(win + loss + nores - 1) < 1e-6 and abs(score) < 200
            moves, visits = data.policy_targets_by_turn[t]
            assert visits >= V and max(v for _, _, v in moves) >= 10
            # the move played is one of the searched moves
            assert tuple(data.moves[t]) in {(x, y) for x, y, v in moves}
            q = data.white_q_value_targets_by_turn[t]
            assert len(q) > 0 and all(abs(wl) <= 1 and v >= 1 for _, _, wl, _, v in q)

    files = sorted(os.listdir(tmp_path))
    rows = {k: np.concatenate([np.load(os.path.join(tmp_path, f))[k] for f in files]) for k in W.schema(L)}
    assert rows["globalTargetsNC"].shape[0] == total_rows == writer.row_count
    # rows come game by game, turn by turn: check positions, side to move and policy targets of the first recorded game
    g0, d0 = games[0]
    n0 = len(d0.moves)
    first = 0
    for _, d in all_games:                               # rows of the games written before it
        if d is d0:
            break
        first += len(d.moves)
    rows = {k: v[first:] for k, v in rows.items()}
    planes = np.unpackbits(rows["binaryInputNCHWPacked"][:n0], axis=2)[:, :, :L * L]
    for t in range(n0):
        own, opp = d0.next_player_by_turn[t], 3 - d0.next_player_by_turn[t]
        assert np.array_equal(planes[t, 1], (d0.boards_by_turn[t] == own).astype(np.uint8))
        assert np.array_equal(planes[t, 2], (d0.boards_by_turn[t] == opp).astype(np.uint8))
        assert rows["globalTargetsNC"][t, 51] == t
        dense = np.zeros(L * L + 1, np.int16)
        for x, y, v in d0.policy_targets_by_turn[t][0]:
            dense[L * L if x < 0 else y * L + x] = v
        assert np.array_equal(rows["policyTargetsNCMove"][t, 0], dense)
        if t + 1 < n0:
            assert rows["globalTargetsNC"][t, 28] == 1.0
    assert rows["globalTargetsNC"][n0 - 1, 28] == 0.0          # the last turn has no next-turn policy
    if not d0.end_no_result:
        own_area = np.where(d0.final_ownership == d0.next_player_by_turn[0], 1, np.where(d0.final_ownership == 0, 0, -1))
        assert np.array_equal(rows["valueTargetsNCHW"][0, 0].reshape(-1), own_area)
    sp.free(); h.free(); ctx.free()


@pytest.mark.gpu
@pytest.mark.parametrize("ko_rule", [0, 1])
def test_recorded_games_through_the_reference_writer(tmp_path, tmp_models, ko_rule):
    """The integrated configuration (INTEGRATION.md §6): oracle/_ref/kgref_record plays games on the device loop, fills the REFERENCE's
    FinishedGameData (integration/b200record.h) and lets the reference's own TrainingDataWriter write them - every input plane
    recomputed by the reference's fillRowV7 on its own Board / BoardHistory, every move re-checked by its isLegal, game end and
    final score by its BoardHistory.  The same configuration recorded by katago_b200/game_recorder.py + npz_writer.py must give the
    same rows: input planes bit for bit (the device's featurization of whole games vs the reference's), integer targets exactly,
    float columns to the 6 digits of the reference's text sink.  The reference's rows are stored (tests/reference_runs.py)."""
    import ctypes
    from katago_b200.nn_backend import NeuralNet, SelfPlay
    from reference_runs import reference_run
    from test_npz_writer import _parse_text_dump
    L, G, V, NUM = 9, 6, 40, 6
    komi = 7.0 if ko_rule else 6.5
    lm = NeuralNet.loadModelFile(tmp_models["tiny_reg"])
    ctx = NeuralNet.createComputeContext([0], L, L, True, lm)
    h = NeuralNet.createComputeHandle(ctx, lm, G, False, True, 0)
    sp = SelfPlay(h, G, V, komi=komi, seed=23, max_moves=60, debug_fake_nn=True, debug_hold_at_max_visits=True, use_graph_search=(ko_rule == 0),
                  value_weight_exponent=0.5, static_score_utility_factor=0.05, dynamic_score_utility_factor=0.3,
                  dynamic_score_center_zero_weight=0.25, dynamic_score_center_scale=0.5, use_play_selection=True, use_lcb_for_selection=True,
                  use_non_buggy_lcb=True, lcb_stdevs=5.0, min_visit_prop_for_lcb=0.15, chosen_move_temperature=0.15,
                  chosen_move_temperature_early=0.75, root_noise_enabled=True, root_dirichlet_noise_total_concentration=10.83,
                  root_dirichlet_noise_weight=0.25, ko_rule=ko_rule, full_history_rules=True)
    cfg_path = tmp_path / "config.bin"
    cfg_path.write_bytes(ctypes.string_at(ctypes.addressof(sp.cfg), ctypes.sizeof(sp.cfg)))
    out_path = tmp_path / "reference_rows.txt"
    reference_run("kgref_record", [tmp_models["tiny_reg"], L, cfg_path, NUM, out_path])
    want = _parse_text_dump(out_path.read_text())
    assert len(want) == 1

    got = []
    writer = W.TrainingDataWriter(None, 4096, 1.0, L, "recorder-test", on_flush=lambda b: got.append({k: v[:b.cur_rows].copy() for k, v in b.arrays.items()}))
    games = []

    class FirstGames:                      # the driver writes the first NUM finished games, in the order they finish
        def write_game(self, data):
            if len(games) < NUM:
                writer.write_game(data)
            games.append(data)
    rec = R.GameRecorder(sp, FirstGames(), komi)
    steps = 0
    while len(games) < NUM and steps < 2000:
        rec.step()
        steps += 1
    writer.flush_if_nonempty()
    assert len(got) == 1
    fw, fg = want[0], got[0]
    n = len(fw["globalTargetsNC"])
    assert n == fg["globalTargetsNC"].shape[0] == sum(len(d.moves) for d in games[:NUM]) > 0
    ref_planes = [bytes.fromhex(r) for r in fw["binaryInputNCHWPacked"]]
    for i in range(n):
        if ref_planes[i] != fg["binaryInputNCHWPacked"][i].tobytes():
            a = np.unpackbits(np.frombuffer(ref_planes[i], np.uint8).reshape(22, -1), axis=1)[:, :L * L]
            b = np.unpackbits(fg["binaryInputNCHWPacked"][i], axis=1)[:, :L * L]
            raise AssertionError(("input planes differ", i, sorted(set(np.argwhere(a != b)[:, 0].tolist()))))
    for name in ("policyTargetsNCMove", "scoreDistrN", "valueTargetsNCHW", "qValueTargetsNCMove"):
        a = np.stack(fw[name]).astype(np.int64)
        b = fg[name].reshape(n, -1).astype(np.int64)
        assert np.array_equal(a, b), (name, np.argwhere(a != b)[:5])
    for name in ("globalInputNC", "globalTargetsNC"):
        a = np.stack(fw[name])
        b = fg[name].reshape(n, -1).astype(np.float64)
        assert np.allclose(a, b, rtol=2e-5, atol=1e-30), (name, np.argwhere(~np.isclose(a, b, rtol=2e-5, atol=1e-30))[:5])
    sp.free(); h.free(); ctx.free()


def test_search_limits_this_move_restates_the_reference_rules():
    """getSearchLimitsThisMove (program/play.cpp:1093-1223): cheap searches with their probability, visit count and target weight (root noise
    off when they are not recorded), otherwise visits reduced quadratically once the recent root values are decided beyond the threshold."""
    import random
    from katago_b200.game_recorder import search_limits_this_move as L
    ps = dict(cheap_search_prob=0.75, cheap_search_visits=100, cheap_search_target_weight=0.0, reduce_visits=True, reduce_visits_threshold=0.9,
              reduce_visits_threshold_lookback=3, reduced_visits_min=50, reduced_visits_weight=0.1)
    r = random.Random(1)
    draws = [L(600, ps, r, []) for _ in range(4000)]
    cheap = [d for d in draws if d[3]]
    assert abs(len(cheap) / 4000 - 0.75) < 0.03 and all(d == (100, True, 0.0, True) for d in cheap)
    assert all(d == (600, False, 1.0, False) for d in draws if not d[3])           # no history: nothing to reduce
    full = dict(ps, cheap_search_prob=0.0)
    assert L(600, full, r, [0.95, 0.2, 0.97]) == (600, False, 1.0, False)           # one undecided value among the last three
    assert L(600, full, r, [0.1, 0.95, 0.96, 0.97])[0] == round(600 + ((0.95 - 0.9) / 0.1) ** 2 * (50 - 600))      # min over the lookback, white ahead
    v, plain, w, ch = L(600, full, r, [-0.99, -0.98, -1.0])                         # black ahead: max of the values, sign flipped
    assert (v, plain, ch) == (round(600 + 0.8 ** 2 * (50 - 600)), False, False) and abs(float(w) - (1.0 + 0.64 * (0.1 - 1.0))) < 1e-6
    assert L(600, full, r, [1.0, 1.0, 1.0])[0] == 50 and abs(float(L(600, full, r, [1.0, 1.0, 1.0])[2]) - 0.1) < 1e-6
    recorded = dict(ps, cheap_search_prob=1.0, cheap_search_target_weight=0.25)
    assert L(600, recorded, r, []) == (100, False, 0.25, True)                      # recorded cheap searches keep their root noise
    with pytest.raises(ValueError):
        L(80, dict(ps, cheap_search_prob=1.0), random.Random(2), [])        # cheapSearchVisits above maxVisits


@pytest.mark.gpu
def test_device_applies_per_move_search_limits(golden_dir, tmp_models):
    """kgb_selfplay_set_next_search_limits: a root with a reduced budget is held at that budget, and a "plain" root searches exactly like a
    loop whose root parameters are the tree's (runBotWithLimits removeRootNoise: no noise, temperature 1, tree FPU, no visit floor, one
    symmetry) - identical visit counts; the limits handed over for the following root take effect after the move."""
    from katago_b200 import NeuralNet, SelfPlay
    d = np.load(os.path.join(golden_dir, "searchfake.npz"))
    moves = [None if m[0] < 0 else (int(m[0]), int(m[1])) for m in d["c1_moves"]]
    lm = NeuralNet.loadModelFile(tmp_models["tiny_reg"])
    ctx = NeuralNet.createComputeContext([0], 9, 9, True, lm)
    h = NeuralNet.createComputeHandle(ctx, lm, 4, False, True, 0)
    common = dict(komi=7.5, seed=1, debug_fake_nn=True, debug_hold_at_max_visits=True, use_graph_search=True, value_weight_exponent=0.5,
                  fpu_reduction_max=0.2, fpu_loss_prop=0.1, static_score_utility_factor=0.05, dynamic_score_utility_factor=0.3,
                  dynamic_score_center_zero_weight=0.25, dynamic_score_center_scale=0.5, use_play_selection=True)
    a = SelfPlay(h, 3, 64, root_noise_enabled=True, root_policy_temperature=1.1, root_policy_temperature_early=1.5, root_fpu_reduction_max=0.0,
                 root_fpu_loss_prop=0.3, root_desired_per_child_visits_coeff=2.0, root_num_symmetries_to_sample=4, **common)
    b = SelfPlay(h, 3, 40, root_noise_enabled=False, root_fpu_reduction_max=0.2, root_fpu_loss_prop=0.1, **common)
    with pytest.raises(Exception, match="between 2 and max_visits"):
        a.set_next_search_limits(np.full((3, 2), 65, np.int32))
    for sp in (a, b):
        sp.play_moves(moves)
    a.set_next_search_limits(np.array([[40, 40], [40, 40], [64, 64]], np.int32), np.array([[1, 1], [1, 1], [0, 0]], np.uint8), also_current_roots=True)
    assert np.array_equal(a.search_limits()[0], [40, 40, 64]) and np.array_equal(a.search_limits()[1], [1, 1, 0])
    for sp in (a, b):
        for _ in range(60):
            sp.run(8)
    va, vb = a.root_visits(), b.root_visits()
    assert list(va) == [40, 40, 64] and list(vb) == [40, 40, 40]
    for g in (0, 1):
        ca, pa, ua = a.root_children(g); cb, pb, ub = b.root_children(g)
        assert np.array_equal(ca, cb) and np.array_equal(pa, pb) and np.abs(ua - ub)[ca > 0].max() < 1e-12
    assert not np.array_equal(a.root_children(2)[1], b.root_children(2)[1])            # the ordinary root of game 2 carries noise and temperature
    # NNRawStats::policyEntropy: the entropy of the policy as evaluated, before temperature and noise - for a plain root that IS the searched policy
    ent = a.root_raw_policy_entropy()
    H = lambda p: float(-(p[p > 0].astype(np.float64) * np.log(p[p > 0].astype(np.float64))).sum())
    assert abs(ent[0] - H(a.root_children(0)[1])) < 1e-6 and abs(ent[2] - H(a.root_children(2)[1])) > 1e-3
    with pytest.raises(Exception, match="already been searched"):
        a.set_next_search_limits(np.full((3, 2), 30, np.int32), also_current_roots=True)
    a.set_next_search_limits(np.array([[24, 50], [16, 50], [64, 50]], np.int32), np.array([[0, 0], [1, 0], [0, 0]], np.uint8))
    a.release()
    for _ in range(40):
        a.run(8)
    assert list(a.root_visits()) == [24, 16, 64] and np.array_equal(a.search_limits()[1], [0, 1, 0])
    a.free(); b.free(); h.free(); ctx.free()


def test_search_limits_equal_the_reference_games(tmp_path):
    """Whole games of the reference's Play::runGame with reduceVisits and recorded cheap searches on (tests/golden/make_searchlimits_fixture.py): the
    budget (root visits) and target weight of every turn equal what search_limits_this_move derives from the root win/loss values of the turns
    before it - exactly for reduced searches; a cheap turn has the cheap budget and weight, and cheap turns occur with cheapSearchProb."""
    import gzip, json, random
    from katago_b200.game_recorder import search_limits_this_move as L
    games = json.loads(gzip.open(os.path.join(GOLDEN, "searchlimits.json.gz")).read())
    checked = reduced = cheap_turns = cheap_games_turns = 0
    for g in games:
        ps = {}
        if g["reduce"]:
            thr, look, mn, w = g["reduce"].split(",")
            ps.update(reduce_visits=True, reduce_visits_threshold=float(thr), reduce_visits_threshold_lookback=int(look), reduced_visits_min=int(mn), reduced_visits_weight=float(w))
        cheap = None
        if g["cheap"]:
            pr, v, w = g["cheap"].split(",")
            cheap = (int(v), float(w))
        for t, (visits, weight) in enumerate(zip(g["rootVisits"], g["targetWeight"])):
            want_v, _, want_w, _ = L(g["maxVisits"], ps, random.Random(0), g["rootWinLoss"][:t])       # the non-cheap branch (no cheap_search_prob in ps)
            if cheap is not None and visits == cheap[0] and abs(weight - cheap[1]) < 1e-6:
                cheap_turns += 1
            else:
                assert visits == want_v and abs(weight - float(want_w)) < 1e-6, (g["size"], t, visits, want_v, weight, want_w)
                reduced += int(visits < g["maxVisits"])
            checked += 1
        if cheap is not None:
            cheap_games_turns += len(g["rootVisits"])
    assert checked > 250 and reduced > 20, (checked, reduced)
    assert 0.35 < cheap_turns / cheap_games_turns < 0.65, (cheap_turns, cheap_games_turns)      # games with cheapSearchProb 0.4 and 0.6
