"""The C++-only host (integration/b200_selfplay_main.cpp + b200_recorder.h + b200_npz.h) end to end on the CPU: linked against the mock of the
recording ABI (tests/mock/kgb200_mock.cpp: random legal games on the reference's Board, made-up search statistics, the reference's fillRowV7 rows
and Rand), it must write the same files as the Python host's recorder and writer do from the mock's log - whole .npz files array by array,
bit for bit, under the same names, and the same .sgfs records.  The Python writer is pinned to the reference's own addRow / writeGame / writeSgf
(tests/test_npz_writer.py), the Python recorder to whole reference games (tests/test_game_recorder.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
MOCK = os.path.join(ROOT, "oracle", "_ref", "kgb200_mock.o")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libkgref.a")

pytestmark = pytest.mark.skipif(not (os.path.exists(MOCK) and os.path.exists(REF_LIB)),
                                reason="oracle/_ref/kgb200_mock.o is not built (oracle/Makefile.drivers compiles the mock against the reference's sources)")


def _host_on_mock(main_src, exe):
    """A C++ host - repository sources only - linked against the mock of the recording ABI and the reference objects the mock plays on."""
    subprocess.run(["g++", "-O1", "-std=c++17", "-mfpmath=sse", "-DNDEBUG", "-w", "-I" + ROOT, "-o", str(exe), os.path.join(ROOT, "integration", main_src), MOCK,
                    "-Wl,--start-group", REF_LIB, "-Wl,--end-group", "-lz", "-lpthread"], check=True, cwd=ROOT)
    return str(exe)


@pytest.fixture(scope="module")
def host_on_mock(tmp_path_factory):
    return _host_on_mock("b200_selfplay_main.cpp", tmp_path_factory.mktemp("cpphost_mock") / "b200_selfplay_mock")


def _replay_slots_with_limits(log, G, size, V, uneven=0):
    """ReplaySlots plus the device's per-root search limits as the mock keeps them: a root's budget and plain flag are the ones handed over for "after
    this slot's next move" (entry 0 the game goes on, entry 1 a new game starts); searches finish instantly, root visits = budget (+ slot in the info)."""
    from test_game_recorder import ReplaySlots

    class Slots(ReplaySlots):
        def __init__(self):
            super().__init__(log, G, size, V)
            self.budget, self.plain = np.full(G, V, np.int32), np.zeros(G, np.uint8)
            self.next_budget, self.next_plain = np.full((G, 2), V, np.int32), np.zeros((G, 2), np.uint8)
            self.waves_run = [0] * G
            # KGB_MOCK_UNEVEN: a game's opening takes one wave per move; the slot has no root meanwhile (and reports its budget as visits, like stale device state)
            self.opening_left = [len(self.root[g].get("init_moves", [])) if uneven else 0 for g in range(G)]
            self.cur_setup = np.tile(np.array([size, size, 0, 1], np.int32), (G, 1))
            self.next_setup, self.last_setup = self.cur_setup.copy(), self.cur_setup.copy()
            self.cur_komi = np.full(G, 7.5, np.float32)
            self.next_komi, self.last_komi = self.cur_komi.copy(), self.cur_komi.copy()

        def set_next_search_limits(self, visits2, plain2=None, also_current_roots=False):
            self.next_budget = np.array(visits2, np.int32).reshape(G, 2)
            self.next_plain = np.zeros((G, 2), np.uint8) if plain2 is None else np.array(plain2, np.uint8).reshape(G, 2)
            if also_current_roots:
                self.budget, self.plain = self.next_budget[:, 0].copy(), self.next_plain[:, 0].copy()

        def search_limits(self):
            return self.budget.copy(), self.plain.copy()

        def release(self, mask=None):
            self.released = [True] * G if mask is None else [bool(m) for m in mask]

        # per-game board, rules and komi: of the games in progress, of each slot's next game and of its last finished one
        def set_game_setup(self, setups, also_current_games=False):
            self.next_setup = np.array(setups, np.int32).reshape(G, 4).copy()
            if also_current_games:
                self.cur_setup = self.next_setup.copy()

        def set_komi(self, komis, also_current_games=False):
            self.next_komi = np.array(komis, np.float32).copy()
            if also_current_games:
                self.cur_komi = self.next_komi.copy()

        def game_setups(self):
            return self.cur_setup.copy(), self.last_setup.copy()

        # a side loop's position: the host ends the slot's game with passes and replays the position's moves (komi_search.KomiSearcher._load)
        def play_moves_game(self, slot, moves):
            ev = self.queues[slot].pop(0)
            assert ev["ev"] == "playmoves" and [tuple(m) for m in ev["moves"]] == [(-1, -1) if m is None else (int(m[0]), int(m[1])) for m in moves], (ev, moves)
            before = self.root[slot]["move_num"]
            self.root[slot] = self.queues[slot].pop(0)
            self.waves_run[slot] = 0
            assert self.root[slot]["ev"] == "root"
            if moves and self.root[slot]["move_num"] < before + len(moves):        # a move ended the game: the slot took the setup and komi handed over
                self.last_setup[slot], self.cur_setup[slot] = self.cur_setup[slot].copy(), self.next_setup[slot].copy()
                self.last_komi[slot], self.cur_komi[slot] = self.cur_komi[slot], self.next_komi[slot]

        # policy-initialised openings: the mock plays a whole opening when the game starts and lists it with every root of the game
        def set_policy_init(self, num_moves, temperature=1.0, also_current_games=False):
            pass

        def policy_init(self, max_moves=0):
            n = self.x * self.y
            moves = [[(-1, -1) if p == n else (p % self.x, p // self.x) for p in self.root[g]["init_moves"]] for g in range(G)]
            return np.array(self.opening_left, np.int32), np.array([len(m) for m in moves], np.int32), (moves if max_moves > 0 else None)

        def komi_values(self):
            return self.cur_komi.copy(), self.last_komi.copy()

        def root_visits(self):          # the budget once the root's search has had the waves it needs (KGB_MOCK_UNEVEN), one less before
            return self.budget - np.array([1 if self.waves_left(g) > 0 else 0 for g in range(G)], np.int32)

        def waves_left(self, g):
            return 0 if self.opening_left[g] > 0 else max(0, self.root[g].get("waves_needed", 0) - self.waves_run[g])

        def game(self, g):
            colors, info = super().game(g)
            info["root_visits"] = int(self.budget[g]) + g
            return colors, info

        def run(self, n):
            moving = [g for g in range(G) if self.released[g] and self.queues[g]]
            for g in range(G):
                if self.released[g]:
                    continue
                if self.opening_left[g] > 0:
                    self.opening_left[g] -= min(n, self.opening_left[g])
                    self.waves_run[g] = 0
                else:
                    self.waves_run[g] += n
            assert all(self.waves_left(g) == 0 and self.opening_left[g] == 0 for g in moving), "a slot was released before its search had finished"
            super().run(n)
            for g in moving:
                self.waves_run[g] = 0
                if uneven and self.last[g]["flags"] & 1:
                    self.opening_left[g] = len(self.root[g].get("init_moves", []))
            for g in moving:
                k = 1 if self.last[g]["flags"] & 1 else 0
                self.budget[g], self.plain[g] = self.next_budget[g, k], self.next_plain[g, k]
                if k:
                    self.last_setup[g], self.cur_setup[g] = self.cur_setup[g].copy(), self.next_setup[g].copy()
                    self.last_komi[g], self.cur_komi[g] = self.cur_komi[g], self.next_komi[g]
    return Slots()


FORKS = ("earlyForkGameProb = 0.4\nearlyForkGameExpectedMoveProp = 0.15\nforkGameProb = 0.5\nforkGameMinChoices = 2\nearlyForkGameMaxChoices = 4\nforkGameMaxChoices = 3\n"
         "forkCompensateKomiProb = 0.5\n")
SIDE = "forkSidePositionProb = 0.25\n"
LIMITS = {"none": "", "side_positions": SIDE + "estimateLeadProb = 0.1\nestimateLeadVisits = 6\nmaxMovesPerGame = 30\n",
          "everything": SIDE + FORKS + "komiAuto = true\ncompensateKomiVisits = 10\nestimateLeadProb = 0.15\nestimateLeadVisits = 6\nmaxMovesPerGame = 30\ninitGamesWithPolicy = true\n"
                        "policyInitAreaProp = 0.05\ncheapSearchProb = 0.25\ncheapSearchVisits = 5\ncheapSearchTargetWeight = 0.0\nreduceVisits = true\nreduceVisitsThreshold = 0.3\n"
                        "reduceVisitsThresholdLookback = 2\nreducedVisitsMin = 6\nreducedVisitsWeight = 0.2\n", "forks": FORKS + "estimateLeadProb = 0.15\nestimateLeadVisits = 6\nmaxMovesPerGame = 30\ninitGamesWithPolicy = true\npolicyInitAreaProp = 0.05\n", "forks_only": FORKS, "komi_searches": "komiAuto = true\ncompensateKomiVisits = 10\nestimateLeadProb = 0.3\nestimateLeadVisits = 6\nmaxMovesPerGame = 30\n", "openings": "initGamesWithPolicy = true\npolicyInitAreaProp = 0.08\npolicyInitAreaTemperature = 0.7\ncheapSearchProb = 0.2\ncheapSearchVisits = 8\ncheapSearchTargetWeight = 0.25\n", "cheap": "cheapSearchProb = 0.3\ncheapSearchVisits = 8\ncheapSearchTargetWeight = 0.25\n",
          "cheap_unrecorded_and_reduced": "cheapSearchProb = 0.25\ncheapSearchVisits = 5\ncheapSearchTargetWeight = 0.0\nreduceVisits = true\nreduceVisitsThreshold = 0.3\n"
                                          "reduceVisitsThresholdLookback = 2\nreducedVisitsMin = 6\nreducedVisitsWeight = 0.2\n"}


MIXED = ("bSizes = 5,7,9\nbSizeRelProbs = 1,2,1\nallowRectangleProb = 0.3\nkoRules = SIMPLE,POSITIONAL,SITUATIONAL\nmultiStoneSuicideLegals = false,true\n"
         "komiStdev = 1.0\nkomiBigStdevProb = 0.2\nkomiBigStdev = 8.0\nkomiBiggerStdevProb = 0.05\nkomiAllowIntegerProb = 0.5\n")


@pytest.mark.parametrize("size,ko,komi,max_moves,psw,vsw,search_surprise,games,seed,limits", [
    (9, "SIMPLE", 6.5, 40, 0.5, 0.1, False, 7, 3, "none"),          # stock-like surprise weighting, games stopped by the move limit, several files
    (5, "POSITIONAL", 7.0, 60, 0.0, 0.0, False, 9, 11, "none"),     # integer komi (draws), games ended by passes, every weight 1
    (7, "SITUATIONAL", -2.5, 30, 0.3, 0.2, True, 5, 5, "none"),     # search-value surprise
    (9, "SIMPLE", 7.5, 40, 0.5, 0.1, False, 7, 21, "cheap"),        # recorded cheap searches (weight 0.25) under the surprise weighting
    (7, "POSITIONAL", 6.5, 50, 0.5, 0.1, False, 8, 8, "cheap_unrecorded_and_reduced"),   # unrecorded cheap searches (plain roots) and reduced visits
    (9, "MIXED", 6.5, 0, 0.5, 0.1, False, 12, 4, "cheap"),         # board size (rectangles), ko / suicide rule and komi noise drawn per game, inside a 9x9 data frame
    (9, "MIXED", 7.0, 0, 0.5, 0.1, False, 12, 9, "openings"),      # the same with policy-initialised openings: a start history before the recorded turns
    (9, "MIXED", 6.0, 0, 0.5, 0.1, False, 10, 13, "komi_searches"),  # komiAuto and lead targets: komi bisections as jobs on two side loops, games written when their jobs are back
    (9, "MIXED", 6.5, 0, 0.5, 0.1, False, 24, 17, "forks"),          # forked games: positions of finished games, a forking move chosen by the net's score, komi compensation, the fork pool
    (7, "SIMPLE", 7.5, 30, 0.0, 0.0, False, 15, 2, "forks_only"),    # forks without any other side-loop feature: the fork evaluations get a side loop of their own
    (9, "MIXED", 7.0, 0, 0.5, 0.1, False, 14, 19, "side_positions"), # side positions: forking moves off the main line searched on a third side loop, their rows written with the game
    (9, "MIXED", 6.5, 0, 0.5, 0.1, False, 20, 23, "everything"),     # every option this host has, together
    (19, "STOCK", 7.5, 40, 0.5, 0.1, False, 12, 29, "none"),         # the reference's stock b18 training configuration (what neither host has is left out and named)
])
@pytest.mark.parametrize("uneven", [0, 9], ids=["instant_searches", "uneven_searches"])       # searches that finish at once / after 1..9 waves, each slot on its own (KGB_MOCK_UNEVEN)
def test_cpp_host_writes_the_files_the_python_host_writes(tmp_path, host_on_mock, size, ko, komi, max_moves, psw, vsw, search_surprise, games, seed, limits, uneven):
    from katago_b200 import game_recorder as R, npz_writer as W, selfplay_cli as C
    G, V, ROWS_PER_FILE = 3, 20, 60
    cfg = tmp_path / "c.cfg"
    if ko == "STOCK":
        from test_selfplay_cli import STOCK_B18_SETTINGS
        V = int(STOCK_B18_SETTINGS["maxVisits"])
        stock = dict(STOCK_B18_SETTINGS, numGameThreads=G, maxMovesPerGame=max_moves, maxRowsPerTrainFile=ROWS_PER_FILE, firstFileRandMinProp=0.3, b200WavesPerPoll=4)
        psw, vsw = float(stock["policySurpriseDataWeight"]), float(stock["valueSurpriseDataWeight"])
        cfg.write_text("".join(f"{k} = {v}\n" for k, v in stock.items()))
    else:
        cfg.write_text(f"maxVisits = {V}\nnumGameThreads = {G}\nkomiMean = {komi}\n" + (f"maxMovesPerGame = {max_moves}\n" if max_moves else "") +
                       (MIXED + f"dataBoardLen = {size}\n" if ko == "MIXED" else f"bSizes = {size}\nkoRules = {ko}\n") +
                       f"policySurpriseDataWeight = {psw}\nvalueSurpriseDataWeight = {vsw}\nuseSearchValueSurprise = {'true' if search_surprise else 'false'}\n"
                       f"maxRowsPerTrainFile = {ROWS_PER_FILE}\nfirstFileRandMinProp = 0.3\nb200WavesPerPoll = 4\n" + LIMITS[limits])
    out, log = tmp_path / "cpp", tmp_path / "log.jsonl"
    if size == 5:      # `katago selfplay -models-dir`: the newest net of the directory, its files under <output-dir>/<net name>/
        os.makedirs(tmp_path / "nets" / "b6c96-s100-d200")
        (tmp_path / "nets" / "older.bin.gz").write_bytes(b"unused")
        os.utime(tmp_path / "nets" / "older.bin.gz", (1, 1))
        (tmp_path / "nets" / "b6c96-s100-d200" / "model.bin.gz").write_bytes(b"unused")
        model_args, net_name, out_dir = ["-models-dir", str(tmp_path / "nets")], "b6c96-s100-d200", out / "b6c96-s100-d200"
    else:
        (tmp_path / "model.bin").write_bytes(b"unused")
        model_args, net_name, out_dir = ["-model", str(tmp_path / "model.bin")], "mocknet", out
    r = subprocess.run([host_on_mock] + model_args + ["-config", str(cfg), "-output-dir", str(out), "-max-games-total", str(games), "-seed", str(seed)],
                       env=dict(os.environ, KGB_MOCK_LOG=str(log), **({"KGB_MOCK_UNEVEN": str(uneven)} if uneven else {})), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    out = out_dir

    # the Python host's recorder and writer on the same slots (the mock's log replayed), seeded like selfplay_cli.py seeds them
    _, loop_seed, writer_seed = C.shard_plan(0, 1, games, seed)
    sp = _replay_slots_with_limits(str(log), G, size, V, uneven)
    sp.max_visits = V
    kw, data, _ = C.selfplay_kwargs_from_cfg(C.parse_cfg(str(cfg)))
    py = tmp_path / "py"
    os.makedirs(py / "tdata")
    writer = W.TrainingDataWriter(str(py / "tdata"), ROWS_PER_FILE, 0.3, size, writer_seed)
    sink = C.SgfSink(str(py / "sgfs"), writer_seed + ":sgfs", net_name, net_name)
    done = []

    def on_game(slot, finished):
        if len(done) < games:
            writer.write_game(finished)
            sink.add(slot, finished)
            done.append(finished)
            if forks.enabled and fork_searcher is not None and not finished.end_no_result:        # Play::maybeForkGame on the finished game (as the command's on_game)
                all_moves = list(finished.start_moves) + list(finished.moves)
                ko_idx = {"SIMPLE": 0, "POSITIONAL": 1, "SITUATIONAL": 2, "SPIGHT": 3}[finished.ko_rule]
                setup = (finished.x_size, finished.y_size, ko_idx, int(finished.multi_stone_suicide_legal))
                job = forks.job(all_moves, setup, finished.komi, size)
                if job is not None:
                    cap = int(kw.get("max_moves", 0) or 2 * finished.x_size * finished.y_size)
                    fork_searcher.submit(job, setup, [], lambda moves, setup=setup, komi=finished.komi, cap=cap: forks.add(moves, setup, komi) if moves and len(moves) < cap else None)

    from katago_b200.game_initializer import GameInitializer
    # the side loops of the command (selfplay_cli.py make_aux): the mock's second and third loop, replayed from their own logs
    from katago_b200.komi_search import KomiSearcher
    from katago_b200.fork_play import ForkManager
    ks = data["komi_search"]
    forks = ForkManager(data["forks"], __import__("random").Random(loop_seed ^ 0x466F726B))
    fork_needs_loop = forks.enabled and not (ks["komi_auto"] or ks["estimate_lead_prob"] > 0)
    aux, instance = {"fair": None, "lead": None}, 1
    for name, want, visits in (("fair", ks["komi_auto"] or fork_needs_loop, ks["compensate_komi_visits"]), ("lead", ks["estimate_lead_prob"] > 0, ks["estimate_lead_visits"])):
        if want:
            instance += 1
            lp = _replay_slots_with_limits(f"{log}.{instance}", 4, size, max(2, visits))
            lp.max_visits = max(2, visits)
            aux[name] = KomiSearcher(lp)
    side = None
    if data["side_position_prob"] > 0:       # side positions are searched on a loop with the game's own parameters and full visits
        instance += 1
        lp = _replay_slots_with_limits(f"{log}.{instance}", 4, size, V)
        lp.max_visits = V
        side = KomiSearcher(lp)
    fair, lead = aux["fair"], aux["lead"]
    fork_searcher = lead or fair
    setups = C.SlotSetups(GameInitializer(seed=loop_seed ^ 0x47616D65, **data["game_init"]), G, policy_init=data["policy_init"], fair_komi=fair if ks["komi_auto"] else None,
                          forks=forks if forks.enabled else None, searcher=fork_searcher)      # the command's own per-game draws
    setups.start(sp)
    rec = R.GameRecorder(sp, None, komi, on_game=on_game, on_game_start=lambda slot: setups.game_started(sp, rec, slot), lead_estimator=lead,
                         estimate_lead_prob=data["komi_search"]["estimate_lead_prob"], side_searcher=side, side_position_prob=data["side_position_prob"], game_hash_fn=lambda slot, index: C._game_hash(loop_seed, slot, index),
                         policy_surprise_data_weight=psw, value_surprise_data_weight=vsw, use_search_value_surprise=search_surprise,
                         weight_rand=W.RowRand(writer_seed + ":weights"), play_settings=data["play_settings"],
                         limits_rand=__import__("random").Random(loop_seed ^ 0x4C696D69), policy_init=data["policy_init"]["enabled"])
    while len(done) < games:
        rec.pump(4)
        for searcher in (fair, lead, side):
            if searcher is not None:
                searcher.step(8)
    writer.flush_if_nonempty()

    cpp_files, py_files = sorted(os.listdir(out / "tdata")), sorted(os.listdir(py / "tdata"))
    assert cpp_files == py_files and len(cpp_files) >= 2 and all(len(f) == 20 and f.endswith(".npz") for f in cpp_files)
    rows = 0
    for f in cpp_files:
        a, b = np.load(out / "tdata" / f), np.load(py / "tdata" / f)
        assert sorted(a.files) == sorted(b.files) == sorted(W.schema(size))
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (f, k)
            assert a[k].tobytes() == b[k].tobytes(), (f, k, np.argwhere(a[k] != b[k])[:5])
        rows += a["globalTargetsNC"].shape[0]
    assert rows == writer.row_count > 0
    if psw == 0 and vsw == 0:
        assert rows == sum(len(d.moves) for d in done)
    weights = [float(w) for d in done for w in (d.target_weight_by_turn_unrounded or d.target_weight_by_turn)]
    if ko == "STOCK":
        assert "NOT BUILT (the loop runs WITHOUT it): handicapProb" in r.stderr and "TERRITORY not built" in r.stderr
        assert any(d.start_hist_moves > 0 for d in done) and len({d.komi for d in done}) >= 3 and any(len(d.side_positions) for d in done)
    if ko == "MIXED":
        assert len({(d.x_size, d.y_size) for d in done}) >= 3 and len({d.ko_rule for d in done}) >= 2
        assert limits in ("forks", "everything") or any(d.x_size != d.y_size for d in done)
        assert len({d.komi for d in done}) >= 3 and {d.multi_stone_suicide_legal for d in done} == {False, True}
    if limits in ("side_positions", "everything"):
        n_side = sum(len(d.side_positions) for d in done)
        assert n_side >= 10 and rows >= sum(1 for d in done for w in d.target_weight_by_turn if float(w) >= 1) + n_side - 5
    if limits in ("forks", "forks_only"):
        forked = [d for d in done if d.mode == 2]
        assert len(forked) >= 4 and all(d.start_hist_moves >= 1 for d in forked) and forks.forks_made >= forks.forks_used >= len(forked)
        openings = {tuple(d.start_moves + d.moves)[:len(f.start_moves) - 1] for d in done for f in forked}
        assert all(tuple(f.start_moves[:-1]) in openings for f in forked)          # a fork's start is another game's opening plus one move
    if limits == "komi_searches":
        with_lead = [sum(1 for v in d.white_value_targets_by_turn[:-1] if len(v) > 4 and v[4]) for d in done]
        assert sum(with_lead) >= 20 and fair.searches > 30 and lead.searches > 100 and rec.games_waiting_for_lead >= 0
        assert len({d.komi for d in done}) >= 5            # komis drawn around the searched fair komi of each board
    if limits == "openings":
        assert sum(1 for d in done if d.start_hist_moves > 0) >= 4 and max(d.start_hist_moves for d in done) >= 3
        assert all(len(d.start_moves) == d.start_hist_moves for d in done)
    if limits == "cheap_unrecorded_and_reduced":       # turns that are not recorded at all, and visit counts between the minimum and the full budget
        visits = [v - g for d in done for (_, v), g in zip(d.policy_targets_by_turn, [0] * len(d.moves))]
        assert any(w == 0.0 for w in weights) and any(6 + 0 <= v <= V + 2 and v not in (V, V + 1, V + 2) for v in visits)
    cpp_sgfs = os.listdir(out / "sgfs")
    assert cpp_sgfs == [os.path.basename(sink.path)]
    assert open(out / "sgfs" / cpp_sgfs[0]).read() == open(sink.path).read() and sink.count == games
    summary = __import__("json").loads(r.stdout.strip().splitlines()[-1])
    assert summary["games_written"] == games and summary["rows"] == rows and summary["files"] == len(cpp_files)


def _same_tree(a_dir, b_dir, size):
    """Both <dir>/tdata hold the same .npz files (every array byte for byte) and both <dir>/sgfs the same records.  Returns rows."""
    from katago_b200 import npz_writer as W
    fa, fb = sorted(os.listdir(os.path.join(a_dir, "tdata"))), sorted(os.listdir(os.path.join(b_dir, "tdata")))
    assert fa == fb and fa
    rows = 0
    for f in fa:
        a, b = np.load(os.path.join(a_dir, "tdata", f)), np.load(os.path.join(b_dir, "tdata", f))
        assert sorted(a.files) == sorted(b.files) == sorted(W.schema(size))
        for k in a.files:
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), (f, k)
        rows += a["globalTargetsNC"].shape[0]
    sa, sb = sorted(os.listdir(os.path.join(a_dir, "sgfs"))), sorted(os.listdir(os.path.join(b_dir, "sgfs")))
    assert sa == sb and len(sa) == 1 and open(os.path.join(a_dir, "sgfs", sa[0])).read() == open(os.path.join(b_dir, "sgfs", sb[0])).read()
    return rows


@pytest.mark.parametrize("uneven", [0, 9], ids=["instant_searches", "uneven_searches"])
def test_cpp_host_follows_a_new_net_in_the_models_directory(tmp_path, host_on_mock, uneven):
    """`katago selfplay`'s model loop (command/selfplay.cpp:142-231, 336-352): a newer net appears in -models-dir while the host plays; between two
    pumps it stages and commits the new weights into the live handle, drops the evaluation cache, and the finished games' files move to
    <output-dir>/<new net>/ with a writer of their own - the same files, under both nets, as the Python host's ModelOutputs writes when it switches at
    the same point."""
    import re
    from katago_b200 import game_recorder as R, npz_writer as W, selfplay_cli as C
    from katago_b200.game_initializer import GameInitializer
    G, V, size, games, seed = 3, 20, 7, 10, 6
    cfg = tmp_path / "c.cfg"
    cfg.write_text(f"maxVisits = {V}\nnumGameThreads = {G}\nbSizes = {size}\nkomiMean = 6.5\nmaxMovesPerGame = 24\npolicySurpriseDataWeight = 0.5\nvalueSurpriseDataWeight = 0.1\n"
                   "maxRowsPerTrainFile = 50\nfirstFileRandMinProp = 0.5\nb200WavesPerPoll = 4\n")
    nets = tmp_path / "nets"
    os.makedirs(nets / "netA-s100"); os.makedirs(nets / "netB-s200")
    (nets / "netA-s100" / "model.bin.gz").write_bytes(b"unused")
    os.utime(nets / "netA-s100" / "model.bin.gz", (1000, 1000))
    out, log = tmp_path / "cpp", tmp_path / "log.jsonl"
    r = subprocess.run([host_on_mock, "-models-dir", str(nets), "-config", str(cfg), "-output-dir", str(out), "-max-games-total", str(games), "-seed", str(seed),
                        "-model-poll-seconds", "0"],
                       env=dict(os.environ, KGB_MOCK_LOG=str(log), KGB_MOCK_NEW_MODEL=f"{70 * (3 if uneven else 1)}:{nets / 'netB-s200' / 'model.bin.gz'}",
                                **({"KGB_MOCK_UNEVEN": str(uneven)} if uneven else {})), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"changing midgame to new neural net: netB-s200 \(swap 1, after pump (\d+)\)", r.stderr)
    assert m, r.stderr
    swap_after = int(m.group(1))
    summary = __import__("json").loads(r.stdout.strip().splitlines()[-1])
    assert summary["net_swaps"] == 1 and summary["games_written"] == games

    _, loop_seed, writer_seed = C.shard_plan(0, 1, games, seed)
    sp = _replay_slots_with_limits(str(log), G, size, V)
    sp.max_visits = V
    kw, data, _ = C.selfplay_kwargs_from_cfg(C.parse_cfg(str(cfg)))
    outputs = C.ModelOutputs(str(tmp_path / "py"), data, size, writer_seed, W.TrainingDataWriter)
    outputs.switch_to(str(nets / "netA-s100" / "model.bin.gz"))
    done = []

    def on_game(slot, d):
        if len(done) < games:
            outputs.add_game(slot, d)
            done.append(outputs.model_name)
    setups = C.SlotSetups(GameInitializer(seed=loop_seed ^ 0x47616D65, **data["game_init"]), G, policy_init=data["policy_init"])
    setups.start(sp)
    rec = R.GameRecorder(sp, None, 6.5, on_game=on_game, on_game_start=lambda slot: setups.game_started(sp, rec, slot),
                         game_hash_fn=lambda slot, index: C._game_hash(loop_seed, slot, index), policy_surprise_data_weight=0.5, value_surprise_data_weight=0.1,
                         weight_rand=W.RowRand(writer_seed + ":weights"))
    pumps = 0
    while len(done) < games:
        rec.pump(4)
        pumps += 1
        if pumps == swap_after:
            outputs.switch_to(str(nets / "netB-s200" / "model.bin.gz"))
    outputs.close()
    assert set(done) == {"netA-s100", "netB-s200"} and sorted(os.listdir(out)) == ["netA-s100", "netB-s200"]
    rows = sum(_same_tree(str(out / name), str(tmp_path / "py" / name), size) for name in ("netA-s100", "netB-s200"))
    assert rows == summary["rows"] == outputs.rows_total


def test_cpp_host_ranks_swap_nets_together_under_nccl_weights(tmp_path, host_on_mock):
    """-nccl-weights, two ranks of one node (one process per GPU): rank 0 alone polls the models directory, packs the new net and announces the swap; both
    ranks join the library's broadcast of the packed weights and commit, each keeps playing its share of the games with its own seeds and file names, and a
    rank that finishes early stays until every rank has.  (On the mock the collective calls only have to line up; the broadcast itself is the library's,
    measured on GPUs through the Python host: profiles/r02_*weight_broadcast*.)"""
    import json, re
    G, V, size = 3, 20, 7
    cfg = tmp_path / "c.cfg"
    cfg.write_text(f"maxVisits = {V}\nnumGameThreads = {G}\nbSizes = {size}\nkomiMean = 6.5\nmaxMovesPerGame = 20\nmaxRowsPerTrainFile = 40\nb200WavesPerPoll = 4\n")
    nets = tmp_path / "nets"
    os.makedirs(nets / "netA-s100"); os.makedirs(nets / "netB-s200")
    (nets / "netA-s100" / "model.bin.gz").write_bytes(b"unused")
    os.utime(nets / "netA-s100" / "model.bin.gz", (1000, 1000))
    out = tmp_path / "out"
    os.makedirs(out)
    procs = []
    for rank in (0, 1):
        env = dict(os.environ, KGB_MOCK_LOG=str(tmp_path / f"log{rank}.jsonl"))
        if rank == 0:
            env["KGB_MOCK_NEW_MODEL"] = f"60:{nets / 'netB-s200' / 'model.bin.gz'}"
        procs.append(subprocess.Popen([host_on_mock, "-models-dir", str(nets), "-config", str(cfg), "-output-dir", str(out), "-max-games-total", "25", "-seed", "4",
                                       "-model-poll-seconds", "0", "-rank", str(rank), "-world-size", "2", "-gpu", "0", "-nccl-weights"],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=300) for p in procs]
    assert [p.returncode for p in procs] == [0, 0], [o[1][-1500:] for o in outs]
    summaries = [json.loads(o[0].strip().splitlines()[-1]) for o in outs]
    assert [s["games_written"] for s in summaries] == [13, 12] and [s["net_swaps"] for s in summaries] == [1, 1]
    for o in outs:
        assert re.search(r"changing midgame to new neural net: netB-s200 \(swap 1, after pump \d+, ncclBroadcast", o[1]), o[1][-800:]
    files = {name: sorted(os.listdir(out / name / "tdata")) for name in ("netA-s100", "netB-s200")}
    assert len(files["netA-s100"]) >= 2 and len(files["netB-s200"]) >= 2 and len(set(files["netA-s100"]) | set(files["netB-s200"])) == sum(len(v) for v in files.values())
    rows = sum(np.load(out / name / "tdata" / f)["globalTargetsNC"].shape[0] for name, fs in files.items() for f in fs)
    assert rows == sum(s["rows"] for s in summaries)
    assert len(os.listdir(out / "netA-s100" / "sgfs")) == 2 and len(os.listdir(out / "netB-s200" / "sgfs")) == 2        # one record file per rank and net
    hashes = set()
    for name in files:
        for f in os.listdir(out / name / "sgfs"):
            hashes.update(re.findall(r"gameHash=([0-9A-F]{32})", open(out / name / "sgfs" / f).read()))
    assert len(hashes) == 25          # every rank its own games


@pytest.fixture(scope="module")
def gatekeeper_on_mock(tmp_path_factory):
    return _host_on_mock("b200_gatekeeper_main.cpp", tmp_path_factory.mktemp("cppgate_mock") / "b200_gatekeeper_mock")


@pytest.mark.parametrize("uneven", [0, 9], ids=["instant_searches", "uneven_searches"])
@pytest.mark.parametrize("resign,required,seed", [(False, 0.5, 3), (True, 0.5, 8), (False, 0.9, 5)])
def test_cpp_gatekeeper_plays_the_match_the_python_gatekeeper_plays(tmp_path, gatekeeper_on_mock, resign, required, seed, uneven):
    """`katago gatekeeper` as a C++-only host (integration/b200_gatekeeper_main.cpp + b200_match.h) on the mock's two loops against the Python match
    engine (katago_b200/match_play.py) on their logs: the same games move for move and colour for colour (the record file character for character), the
    same points, the same early stop, and the directory protocol's verdict - the candidate moved to the accepted or the rejected directory, the
    self-play directories of an accepted net created."""
    import re
    from katago_b200 import gatekeeper_cli as GK, selfplay_cli as C
    from katago_b200.game_initializer import GameInitializer
    from katago_b200.match_play import MatchPlay
    from katago_b200.npz_writer import write_sgf
    G, V, size, total = 4, 20, 9, 14
    cfg = tmp_path / "g.cfg"
    cfg.write_text(f"maxVisits = {V}\nnumGameThreads = {G}\nnumGamesPerGating = {total}\nbSizes = 7,9\nbSizeRelProbs = 1,1\nkoRules = SIMPLE,POSITIONAL\nkomiMean = 7.0\nkomiStdev = 1.0\n"
                   "maxMovesPerGame = 40\nb200WavesPerPoll = 4\n" + ("allowResignation = true\nresignThreshold = -0.2\nresignConsecTurns = 2\n" if resign else ""))
    dirs = {k: tmp_path / k for k in ("test", "accepted", "rejected", "sgfs", "selfplay")}
    os.makedirs(dirs["test"] / "cand-s300"); os.makedirs(dirs["accepted"] / "base-s200")
    (dirs["accepted"] / "base-s200" / "model.bin.gz").write_bytes(b"unused")
    os.utime(dirs["accepted"] / "base-s200", (1000, 1000))
    (dirs["test"] / "cand-s300" / "model.bin.gz").write_bytes(b"unused")
    log = tmp_path / "log.jsonl"
    r = subprocess.run([gatekeeper_on_mock, "-config", str(cfg), "-test-models-dir", str(dirs["test"]), "-sgf-output-dir", str(dirs["sgfs"]), "-accepted-models-dir", str(dirs["accepted"]),
                        "-rejected-models-dir", str(dirs["rejected"]), "-selfplay-dir", str(dirs["selfplay"]), "-required-candidate-win-prop", str(required), "-games-per-gpu", "8",
                        "-quit-if-no-nets-to-test", "-seed", str(seed)], env=dict(os.environ, KGB_MOCK_LOG=str(log), **({"KGB_MOCK_UNEVEN": str(uneven)} if uneven else {})),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]

    # the Python match engine on the two loops' logs
    kw, data, _ = C.selfplay_kwargs_from_cfg(C.parse_cfg(str(cfg)))
    loops = []
    for i in (1, 2):
        lp = _replay_slots_with_limits(str(log) if i == 1 else f"{log}.{i}", G, size, V)
        lp.max_visits = V
        loops.append(lp)
    records = []
    mp = MatchPlay(loops, ("base-s200", "cand-s300"), total, GameInitializer(seed=seed ^ 0x4761746B, **data["game_init"]),
                   on_game=lambda slot, game, b, w, result: records.append(write_sgf(game, b, w)), allow_resignation=resign, resign_threshold=-0.2, resign_consec_turns=2)
    mp.run(waves=4, stop=lambda m: GK.early_verdict(m.win_points[1], m.games_tallied, total, required) != 0)
    m = re.search(r"Candidate (won|lost) match, score ([0-9.]+) to ([0-9.]+) in (\d+) games", r.stderr)
    assert m, r.stderr[-1500:]
    assert (float(m.group(2)), float(m.group(3)), int(m.group(4))) == (round(mp.win_points[1], 3), round(mp.win_points[0], 3), mp.games_tallied)
    accepted = GK.candidate_is_accepted(mp.win_points[1], mp.games_tallied, required)
    assert (m.group(1) == "won") == accepted
    sgf_files = os.listdir(dirs["sgfs"] / "cand-s300")
    assert len(sgf_files) == 1 and open(dirs["sgfs"] / "cand-s300" / sgf_files[0]).read() == "".join(s + "\n" for s in records) and len(records) == mp.games_tallied
    assert os.path.isdir(dirs["accepted" if accepted else "rejected"] / "cand-s300") and not os.listdir(dirs["test"])
    assert os.path.isdir(dirs["selfplay"] / "cand-s300" / "tdata") == accepted
    if resign:
        assert any("+R]" in s for s in records)
    if required == 0.9:
        assert mp.games_tallied < total and "terminating remaning games" in r.stderr          # stopped as soon as the verdict could not change


@pytest.mark.parametrize("uneven", [0, 9], ids=["instant_searches", "uneven_searches"])
def test_cpp_match_plays_two_named_bots_like_the_python_match(tmp_path, uneven):
    """`katago match` for two named bots as a C++-only host (integration/b200_match_main.cpp): per-bot search keys (maxVisits0 / maxVisits1), alternating
    colours, per-game setups - against the Python match engine on the mock loops' logs: the record file character for character, the same wins and points."""
    import re
    exe = _host_on_mock("b200_match_main.cpp", tmp_path / "b200_match_mock")
    from katago_b200 import match_cli as MC, selfplay_cli as C
    from katago_b200.game_initializer import GameInitializer
    from katago_b200.match_play import MatchPlay
    from katago_b200.npz_writer import write_sgf
    G, size, total, seed = 4, 9, 11, 6
    (tmp_path / "a.bin").write_bytes(b"unused"); (tmp_path / "b.bin").write_bytes(b"unused")
    cfg = tmp_path / "m.cfg"
    cfg.write_text(f"numBots = 2\nbotName0 = deep\nbotName1 = shallow\nnnModelFile0 = {tmp_path / 'a.bin'}\nnnModelFile1 = {tmp_path / 'b.bin'}\nmaxVisits0 = 24\nmaxVisits1 = 8\n"
                   f"cpuctExploration1 = 1.3\nnumGameThreads = {G}\nnumGamesTotal = {total}\nbSizes = 7,9\nbSizeRelProbs = 1,2\nkomiMean = 6.5\nkomiStdev = 0.5\nmaxMovesPerGame = 36\n"
                   "b200WavesPerPoll = 4\nallowResignation = true\nresignThreshold = -0.3\nresignConsecTurns = 3\n")
    log = tmp_path / "log.jsonl"
    r = subprocess.run([str(exe), "-config", str(cfg), "-sgf-output-dir", str(tmp_path / "sgfs"), "-log-file", str(tmp_path / "match.log"), "-seed", str(seed)],
                       env=dict(os.environ, KGB_MOCK_LOG=str(log), **({"KGB_MOCK_UNEVEN": str(uneven)} if uneven else {})), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "for bot deep (maxVisits 24)" in r.stderr and "for bot shallow (maxVisits 8)" in r.stderr

    full = C.parse_cfg(str(cfg))
    assert MC.bot_cfg(full, 1)["cpuctExploration"] == "1.3" and "cpuctExploration" not in MC.bot_cfg(full, 0)
    _, data0, _ = C.selfplay_kwargs_from_cfg({k: v for k, v in MC.bot_cfg(full, 0).items() if k not in ("numBots", "numGamesTotal")})
    loops = []
    for i, visits in ((1, 24), (2, 8)):
        lp = _replay_slots_with_limits(str(log) if i == 1 else f"{log}.{i}", G, size, visits)
        lp.max_visits = visits
        loops.append(lp)
    records, wins = [], {"deep": 0, "shallow": 0, "none": 0}

    def on_game(slot, game, b, w, result):
        records.append(write_sgf(game, b, w))
        wins[b if result.startswith("B") else w if result.startswith("W") else "none"] += 1
    mp = MatchPlay(loops, ["deep", "shallow"], total, GameInitializer(seed=seed ^ 0x4D617463, **data0["game_init"]), on_game=on_game, draw_equivalent_wins_for_white=0.5,
                   no_result_utility_for_white=0.0, allow_resignation=True, resign_threshold=-0.3, resign_consec_turns=3)
    mp.run(waves=4)
    files = os.listdir(tmp_path / "sgfs")
    assert len(files) == 1 and open(tmp_path / "sgfs" / files[0]).read() == "".join(s + "\n" for s in records) and len(records) == total == mp.games_tallied
    m = re.search(r"Match finished: deep (\d+) wins, shallow (\d+) wins, (\d+) draws or void; points ([0-9.]+) - ([0-9.]+) in (\d+) games", r.stderr)
    assert m and (int(m.group(1)), int(m.group(2)), int(m.group(3))) == (wins["deep"], wins["shallow"], wins["none"]), r.stderr[-600:]
    assert (float(m.group(4)), float(m.group(5)), int(m.group(6))) == (round(mp.win_points[0], 1), round(mp.win_points[1], 1), total)
    assert open(tmp_path / "match.log").read().count("\n") >= total + 3


def test_cpp_host_rebuilds_its_evaluator_for_a_net_of_another_architecture(tmp_path, host_on_mock):
    """A new net that the live handle cannot take (another architecture: kgb_handle_stage_weights refuses it) makes the host start afresh on it - a
    new evaluator, the games in flight dropped, the games still to play, the next output generation and loop seeds of its own - like
    selfplay_cli.py rebuilds its evaluator in place (the reference builds a new NNEvaluator for every net)."""
    import json, re
    G, V, size, games = 3, 20, 7, 14
    cfg = tmp_path / "c.cfg"
    cfg.write_text(f"maxVisits = {V}\nnumGameThreads = {G}\nbSizes = {size}\nkomiMean = 6.5\nmaxMovesPerGame = 16\nmaxRowsPerTrainFile = 50\nb200WavesPerPoll = 4\n")
    nets = tmp_path / "nets"
    os.makedirs(nets / "netA-s100"); os.makedirs(nets / "netB-otherarch-s200")
    (nets / "netA-s100" / "model.bin.gz").write_bytes(b"unused")
    os.utime(nets / "netA-s100" / "model.bin.gz", (1000, 1000))
    out = tmp_path / "out"
    r = subprocess.run([host_on_mock, "-models-dir", str(nets), "-config", str(cfg), "-output-dir", str(out), "-max-games-total", str(games), "-seed", "5", "-model-poll-seconds", "0"],
                       env=dict(os.environ, KGB_MOCK_LOG=str(tmp_path / "log.jsonl"), KGB_MOCK_NEW_MODEL=f"50:{nets / 'netB-otherarch-s200' / 'model.bin.gz'}"),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "rebuilding the evaluator (games in progress are abandoned)" in r.stderr and "Loaded latest neural net netB-otherarch-s200" in r.stderr
    summary = json.loads(r.stdout.strip().splitlines()[-1])          # the re-started run's own count
    records = {name: open(out / name / "sgfs" / os.listdir(out / name / "sgfs")[0]).read() for name in ("netA-s100", "netB-otherarch-s200")}
    played = {name: text.count("\n") for name, text in records.items()}
    assert played["netA-s100"] >= 3 and played["netB-otherarch-s200"] == summary["games_written"] and sum(played.values()) == games
    hashes = [h for text in records.values() for h in re.findall(r"gameHash=([0-9A-F]{32})", text)]
    assert len(set(hashes)) == games                                   # the re-started run has loop seeds of its own
    files = [f for name in records for f in os.listdir(out / name / "tdata")]
    assert len(set(files)) == len(files) >= 2
