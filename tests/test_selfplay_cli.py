"""CPU tests of the `selfplay` command's configuration layer (SURVEY §8f row 3): the reference's .cfg syntax and key names."""
import inspect, os, sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from katago_b200 import selfplay_cli as C

STOCK_B18_SETTINGS = {   # the settings of the reference's stock b18 self-play training configuration, as key -> value strings
    "allowRectangleProb": "0.10", "bSizeRelProbs": "75,1,4,10", "bSizes": "19,7,9,13", "cheapSearchProb": "0.75", "cheapSearchTargetWeight": "0.0",
    "cheapSearchVisits": "350", "chosenMovePrune": "1", "chosenMoveSubtract": "0", "chosenMoveTemperature": "0.15",
    "chosenMoveTemperatureEarly": "0.75", "chosenMoveTemperatureHalflife": "19", "cpuctExploration": "1.05", "cpuctExplorationLog": "0.28",
    "cudaDeviceToUseModel0Thread0": "0", "cudaUseFP16": "true", "dataBoardLen": "19", "drawEquivalentWinsForWhite": "0.5", "drawRandRadius": "0.5",
    "dynamicScoreCenterScale": "0.50", "dynamicScoreCenterZeroWeight": "0.25", "dynamicScoreUtilityFactor": "0.30", "earlyForkGameProb": "0.04",
    "estimateLeadProb": "0.50", "fancyKomiVarying": "true", "firstFileRandMinProp": "0.15", "forkGameProb": "0.01", "forkSidePositionProb": "0.020",
    "fpuParentWeightByVisitedPolicy": "true", "fpuParentWeightByVisitedPolicyPow": "2.0", "fpuReductionMax": "0.2",
    "handicapAsymmetricPlayoutProb": "0.5", "handicapProb": "0.10", "hasButtons": "false,false,true", "initGamesWithPolicy": "true",
    "koRules": "SIMPLE,POSITIONAL,SITUATIONAL", "komiAuto": "True", "komiStdev": "1.0", "lcbStdevs": "5.0", "logSearchInfo": "false",
    "logToStdout": "true", "maxMovesPerGame": "1600", "maxRowsPerTrainFile": "20000", "maxVisits": "2000", "minVisitPropForLCB": "0.15",
    "multiStoneSuicideLegals": "false,true", "nnCacheSizePowerOfTwo": "24", "nnMaxBatchSize": "192", "nnRandomize": "true",
    "noResultStdev": "0.166666666", "noResultUtilityForWhite": "0.0", "normalAsymmetricPlayoutProb": "0.01", "numGameThreads": "800",
    "numSearchThreads": "1", "numVirtualLossesPerThread": "1", "policyInitAreaProp": "0.08", "policySurpriseDataWeight": "0.5",
    "reduceVisits": "true", "reducedVisitsMin": "350", "rootDesiredPerChildVisitsCoeff": "2", "rootDirichletNoiseTotalConcentration": "10.83",
    "rootDirichletNoiseWeight": "0.25", "rootEndingBonusPoints": "0.5", "rootFpuReductionMax": "0.0", "rootNoiseEnabled": "true",
    "rootNumSymmetriesToSample": "4", "rootPolicyTemperature": "1.1", "rootPolicyTemperatureEarly": "1.5", "rootPruneUselessMoves": "true",
    "scoringRules": "AREA,TERRITORY", "sekiForkHackProb": "0.01", "staticScoreUtilityFactor": "0.05", "subtreeValueBiasFactor": "0.30",
    "subtreeValueBiasWeightExponent": "0.8", "switchNetsMidGame": "true", "taxRules": "NONE,NONE,SEKI,SEKI,ALL", "useGraphSearch": "true",
    "useLcbForSelection": "true", "useNonBuggyLcb": "true", "valueSurpriseDataWeight": "0.1", "valueWeightExponent": "0.5",
    "winLossUtilityFactor": "1.0",
}


@pytest.fixture(scope="module")
def stock_cfg(tmp_path_factory):
    """A .cfg file in the reference's syntax holding those settings."""
    path = tmp_path_factory.mktemp("cfg") / "selfplay.cfg"
    path.write_text("# written by the test\n" + "".join(f"{k} = {v}\n" for k, v in STOCK_B18_SETTINGS.items()))
    return str(path)


def test_stock_training_config_maps_onto_the_loop(stock_cfg):
    cfg = C.parse_cfg(stock_cfg)
    kw, data, report = C.selfplay_kwargs_from_cfg(cfg)
    # the search block of the stock configuration arrives under the loop's parameter names
    assert kw["max_visits"] == 2000 and kw["cpuct_exploration"] == 1.05 and kw["cpuct_exploration_log"] == 0.28
    assert kw["root_fpu_reduction_max"] == 0.0 and kw["value_weight_exponent"] == 0.5 and kw["use_graph_search"] is True
    assert kw["subtree_value_bias_factor"] == 0.30 and kw["root_num_symmetries_to_sample"] == 4 and kw["use_lcb_for_selection"] is True
    assert kw["root_policy_temperature_early"] == 1.5 and kw["chosen_move_temperature_halflife"] == 19.0 and kw["nn_cache_size_power_of_two"] == 24
    assert kw["max_moves"] == 1600 and kw["ko_rule"] == 0 and kw["full_history_rules"] is True and kw["multi_stone_suicide_legal"] is False
    gi = data.pop("game_init")
    ks = data.pop("komi_search")
    fk = data.pop("forks")
    assert data.pop("side_position_prob") == 0.02
    assert fk["early_fork_game_prob"] == 0.04 and fk["fork_game_prob"] == 0.01 and fk["fork_game_min_choices"] == 1
    ps = data.pop("play_settings")
    assert data.pop("policy_init") == {"enabled": True, "area_prop": 0.08, "temperature": 1.0}
    assert ps["cheap_search_prob"] == 0.75 and ps["cheap_search_visits"] == 350 and ps["cheap_search_target_weight"] == 0.0 and ps["reduce_visits"] is True
    assert ps["reduced_visits_min"] == 350
    assert data == {"board_size": 19, "komi": 7.5, "data_board_len": 19, "max_rows_per_train_file": 20000, "first_file_rand_min_prop": 0.15, "num_game_threads": 800,
                    "policy_surprise_data_weight": 0.5, "value_surprise_data_weight": 0.1, "use_search_value_surprise": False}
    # rules, board size and komi are drawn per game from the file's lists like GameInitializer does (bSizes 19,7,9,13 with weights
    # 75,1,4,10 and allowRectangleProb 0.10: every ordered pair of edges, play.cpp:152-172; komiStdev 1.0)
    assert gi["ko_rules"] == [0, 1, 2] and gi["multi_stone_suicide_legals"] == [False, True] and gi["komi_stdev"] == 1.0
    assert len(gi["sizes"]) == 16 and abs(sum(gi["size_probs"]) - 1.0) < 1e-12
    p = dict(zip(gi["sizes"], gi["size_probs"]))
    assert abs(p[(19, 19)] - (0.9 * 75 / 90 + 0.1 * 75 * 75 / 8100)) < 1e-12 and abs(p[(9, 13)] - 0.1 * 4 * 10 / 8100) < 1e-12
    # every keyword exists on the loop
    from katago_b200.nn_backend import SelfPlay
    params = set(inspect.signature(SelfPlay.__init__).parameters)
    assert set(kw) <= params, set(kw) - params
    # per-game randomisation the loop does not have is reported, as are the data-distribution options that are not built
    assert any(s.startswith("scoringRules") and "TERRITORY" in s for s in report["fixed"])      # left out of the draw, and said so
    assert not any(s.startswith(("koRules", "bSizes")) for s in report["fixed"])
    nb = " ".join(report["not_built"])
    assert "komiStdev" not in nb
    assert "cheapSearchProb" not in nb and "reduceVisits" not in nb        # built: drawn by the recorder, applied by the device
    assert "initGamesWithPolicy" not in nb and "policyInitAreaProp" not in nb
    assert "komiAuto" not in nb and "estimateLeadProb" not in nb             # built: komi-bisection searches on a side loop (komi_search.py)
    assert ks == {"komi_auto": True, "compensate_komi_visits": 20, "estimate_lead_prob": 0.5, "estimate_lead_visits": 6}
    assert "forkGameProb" not in nb and "earlyForkGameProb" not in nb           # built: fork_play.py
    assert "forkSidePositionProb" not in nb                                       # built: side positions searched on a side loop
    for key in ("sekiForkHackProb", "handicapProb"):
        assert key in nb, key
    assert "cudaUseFP16" in report["irrelevant"] and "logSearchInfo" in report["irrelevant"] and "numSearchThreads" in report["irrelevant"]
    assert not any(k in nb for k in ("maxVisits", "cpuctExploration", "koRules", "dataBoardLen"))
    with pytest.raises(ValueError, match="not built"):
        C.selfplay_kwargs_from_cfg(cfg, strict=True)


def test_list_valued_keys_are_drawn_per_game_like_the_reference():
    """bSizes with bSizeRelProbs as in the stock selfplay8mainb18.cfg: the evaluator's frame is the data frame, the per-game draw follows
    the weights; komi noise scales with the board (PlayUtils::chooseExtraBlackAndKomi) and stays a half-integer inside the clip range."""
    from katago_b200.game_initializer import GameInitializer, round_and_clip_komi
    kw, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg("bSizes = 7,9,11,13,15,17,19\nbSizeRelProbs = 1,4,2,10,3,4,35\ndataBoardLen = 19\nkomiMean = 7\nkomiStdev = 1.0\n"
                                                              "komiBigStdevProb = 0.06\nkomiBigStdev = 12.0\nkoRules = SIMPLE,POSITIONAL\nmultiStoneSuicideLegals = false,true\n", is_text=True))
    assert data["board_size"] == 19 and report["fixed"] == []
    init = GameInitializer(seed=5, **data["game_init"])
    setups, komis = init.draw_many(20000)
    assert setups.shape == (20000, 4) and (setups[:, 0] == setups[:, 1]).all()            # allowRectangleProb absent: squares only
    freq = {e: float((setups[:, 0] == e).mean()) for e in (7, 9, 11, 13, 15, 17, 19)}
    for e, w in zip((7, 9, 11, 13, 15, 17, 19), (1, 4, 2, 10, 3, 4, 35)):
        assert abs(freq[e] - w / 59) < 0.012, (e, freq[e])
    assert set(setups[:, 2]) == {0, 1} and set(setups[:, 3]) == {0, 1} and abs(float(setups[:, 2].mean()) - 0.5) < 0.02
    assert (komis * 2 == np.round(komis * 2)).all() and (np.abs(komis) <= 20 + setups[:, 0] * setups[:, 1]).all()
    small, big = komis[setups[:, 0] == 9], komis[setups[:, 0] == 19]
    assert abs(float(big.mean()) - 7.0) < 0.1 and float(small.std()) < float(big.std())           # noise scaled by sqrt(area) / 19
    assert 0.9 < float(np.std(big[np.abs(big - 7.0) < 3.5])) < 1.25                               # the common komiStdev = 1.0 part
    assert round_and_clip_komi(7.25, 19, 19) == 7.5 and round_and_clip_komi(-7.25, 19, 19) == -7.5 and round_and_clip_komi(500, 9, 9) == 101.0
    # the frame follows the largest board when dataBoardLen is absent
    kw, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg("bSizes = 9,13\nbSizeRelProbs = 1,1\n", is_text=True))
    assert data["board_size"] == 13 and data["data_board_len"] == 13 and [s_ for s_ in data["game_init"]["sizes"]] == [(9, 9), (13, 13)]
    with pytest.raises(ValueError, match="entries"):
        C.selfplay_kwargs_from_cfg(C.parse_cfg("bSizes = 9,13\nbSizeRelProbs = 1\n", is_text=True))
    # komiAuto: the komi noise is drawn around the fair komi of the empty board, found by search on the side loop; komiMean is where that search starts
    _, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg("komiAuto = true\n", is_text=True), strict=True)
    assert data["komi"] == 7.5 and data["komi_search"]["komi_auto"] is True and report["not_built"] == []
    _, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg("komiAuto = false\nkomiMean = 6.5\n", is_text=True))
    assert data["komi_search"]["komi_auto"] is False and data["komi"] == 6.5


def test_neutral_values_and_unsupported_rules():
    kw, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg("maxVisits = 100\ncheapSearchProb = 0\nreduceVisits = false\nkoRules = POSITIONAL\nbSizes = 9\nkomiMean = 7\nrootEndingBonusPoints = 0\nrootPruneUselessMoves = false\n", is_text=True), strict=True)
    assert kw["ko_rule"] == 1 and data["board_size"] == 9 and data["komi"] == 7.0 and report["not_built"] == [] and report["fixed"] == []
    assert data["policy_surprise_data_weight"] == 0.0
    assert kw["root_ending_bonus_points"] == 0.0 and kw["root_prune_useless_moves"] is False
    # the two root options the reference switches on by default are on when the file does not mention them (Setup::loadParams)
    kw2, _, rep = C.selfplay_kwargs_from_cfg(C.parse_cfg("maxVisits = 100\n", is_text=True), strict=True)
    assert kw2["root_ending_bonus_points"] == 0.5 and kw2["root_prune_useless_moves"] is True and rep["not_built"] == []
    with pytest.raises(ValueError, match="none of these is built"):
        C.selfplay_kwargs_from_cfg(C.parse_cfg("scoringRules = TERRITORY\n", is_text=True))
    with pytest.raises(ValueError, match="dataBoardLen"):
        C.selfplay_kwargs_from_cfg(C.parse_cfg("bSizes = 9,19\ndataBoardLen = 13\n", is_text=True))
    _, d9, _ = C.selfplay_kwargs_from_cfg(C.parse_cfg("bSizes = 9\ndataBoardLen = 19\n", is_text=True))      # small boards inside a 19x19 data frame
    assert d9["board_size"] == 19 and d9["game_init"]["sizes"] == [(9, 9)]
    with pytest.raises(ValueError, match="expected 'key = value'"):
        C.parse_cfg("maxVisits 100\n", is_text=True)
    assert C.parse_cfg("a = 1 # comment\n\n# only a comment\nb=x=y\n", is_text=True) == {"a": "1", "b": "x=y"}


def test_command_fails_loudly_without_a_gpu(tmp_path, stock_cfg):
    """No CPU fallback: on a machine without a B200 the command stops at the evaluator with the library's error."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "tiny.bin"), "tiny_reg", seed=3)
    with pytest.raises(Exception, match="no CUDA device|CUDA"):
        C.main(["-models-dir", str(models), "-output-dir", str(tmp_path / "out"), "-config", stock_cfg, "-max-games-total", "1", "-override-config", "bSizes=9,bSizeRelProbs=1,dataBoardLen=9"])


@pytest.mark.gpu
def test_command_writes_training_files(tmp_path, stock_cfg):
    """End to end on a B200: models dir + reference-style .cfg -> <output-dir>/<model>/tdata/<16 hex>.npz readable as training rows."""
    import numpy as np
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "tinynet.bin"), "tiny_reg", seed=3)
    out = tmp_path / "out"
    rc = C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", stock_cfg, "-max-games-total", "3", "-games-per-gpu", "4",
                 "-override-config", "bSizes=9,bSizeRelProbs=1,dataBoardLen=9,maxVisits=24,maxMovesPerGame=40,rootNumSymmetriesToSample=1,nnCacheSizePowerOfTwo=0,maxRowsPerTrainFile=50,firstFileRandMinProp=1.0,cheapSearchProb=0,reduceVisits=false"])
    assert rc == 0
    tdata = out / "tinynet" / "tdata"
    files = sorted(os.listdir(tdata))
    assert files and all(len(f) == 20 and f.endswith(".npz") for f in files)
    rows = 0
    for f in files:
        with np.load(tdata / f) as z:
            n = z["globalTargetsNC"].shape[0]
            rows += n
            assert n <= 50 and z["binaryInputNCHWPacked"].shape == (n, 22, 11) and z["policyTargetsNCMove"].shape == (n, 2, 82)
            assert (z["globalTargetsNC"][:, 63] == 3.0).all() and (z["globalTargetsNC"][:, 25] == 1.0).all()
    assert rows >= 3 * 2
    sgfs = os.listdir(out / "tinynet" / "sgfs")
    assert len(sgfs) == 1 and sum(1 for _ in open(out / "tinynet" / "sgfs" / sgfs[0])) >= 3


@pytest.mark.gpu
def test_command_plays_mixed_board_sizes_rules_and_komi(tmp_path):
    """BASELINE config 4 through the command: bSizes 5,7,9 (+ rectangles) inside a 9x9 data frame, two ko rules, both suicide rules and komi
    noise drawn per game; the training rows carry each game's own board (plane 0), rules (globals 6-8) and komi (global 5), the game
    records their own sizes."""
    import re
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "tinynet.bin"), "tiny_reg", seed=3)
    settings = dict(STOCK_B18_SETTINGS, bSizes="5,7,9", bSizeRelProbs="2,1,1", allowRectangleProb="0.3", dataBoardLen="9", koRules="SIMPLE,POSITIONAL",
                    multiStoneSuicideLegals="false,true", komiMean="6", komiStdev="2.0", maxVisits="16", maxMovesPerGame="50", rootNumSymmetriesToSample="2",
                    nnCacheSizePowerOfTwo="10", maxRowsPerTrainFile="100000", firstFileRandMinProp="1.0", cheapSearchProb="0", reduceVisits="false")
    settings.pop("komiAuto")
    cfg = tmp_path / "mixed.cfg"
    cfg.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    out = tmp_path / "out"
    rc = C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", str(cfg), "-max-games-total", "24", "-games-per-gpu", "8", "-per-game-release"])
    assert rc == 0
    tdata = out / "tinynet" / "tdata"
    areas, komis, ko_flags, suicide_flags = set(), set(), set(), set()
    for f in os.listdir(tdata):
        with np.load(tdata / f) as z:
            planes = np.unpackbits(z["binaryInputNCHWPacked"], axis=2)[:, :, :81].reshape(-1, 22, 9, 9)
            g = z["globalInputNC"]
            for on, row in zip(planes[:, 0], g):
                ys, xs = np.nonzero(on)
                by, bx = ys.max() + 1, xs.max() + 1
                assert on[:by, :bx].all() and on.sum() == by * bx and bx in (5, 7, 9) and by in (5, 7, 9)      # a full rectangle in the corner
                areas.add((int(bx), int(by)))
                komis.add(round(abs(float(row[5])) * 20.0, 1)); ko_flags.add(float(row[6])); suicide_flags.add(float(row[8]))
            assert ((planes[:, 1] + planes[:, 2]) <= planes[:, 0]).all()           # stones only on the game's own board
    assert len(areas) >= 3 and any(a[0] != a[1] for a in areas), areas
    assert len(komis) >= 3 and ko_flags == {0.0, 1.0} and suicide_flags == {0.0, 1.0}, (komis, ko_flags, suicide_flags)
    sgf_dir = out / "tinynet" / "sgfs"
    sizes = set()
    for f in os.listdir(sgf_dir):
        for line in open(sgf_dir / f):
            m = re.search(r"SZ\[(\d+)(?::(\d+))?\]", line)
            sizes.add((int(m.group(1)), int(m.group(2) or m.group(1))))
    assert sizes == areas or sizes >= {a for a in areas}, (sizes, areas)


@pytest.mark.gpu
def test_command_plays_cheap_and_reduced_searches(tmp_path, stock_cfg):
    """cheapSearchProb / cheapSearchVisits / cheapSearchTargetWeight and reduceVisits through the command: every move's search stops at ITS
    budget (the visit count in the game record), unrecorded cheap searches enter the training files only through the surprise weighting."""
    import re
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "tinynet.bin"), "tiny_reg", seed=3)
    out = tmp_path / "out"
    rc = C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", stock_cfg, "-max-games-total", "6", "-games-per-gpu", "6", "-per-game-release",
                 "-override-config", "bSizes=9,bSizeRelProbs=1,dataBoardLen=9,maxVisits=32,maxMovesPerGame=40,rootNumSymmetriesToSample=2,nnCacheSizePowerOfTwo=10,"
                 "maxRowsPerTrainFile=100000,firstFileRandMinProp=1.0,cheapSearchProb=0.5,cheapSearchVisits=8,cheapSearchTargetWeight=0.0,reduceVisits=true,"
                 "reduceVisitsThreshold=0.3,reduceVisitsThresholdLookback=2,reducedVisitsMin=12,reducedVisitsWeight=0.5,allowRectangleProb=0"])
    assert rc == 0
    visits, weights = [], []
    for f in os.listdir(out / "tinynet" / "sgfs"):
        for line in open(out / "tinynet" / "sgfs" / f):
            visits += [int(v) for v in re.findall(r" v=(\d+)", line)]
            weights += [float(w) for w in re.findall(r"weight=([0-9.]+)", line)]
    assert len(visits) >= 6 * 10 and set(visits) <= set(range(8, 33)), sorted(set(visits))
    # initGamesWithPolicy = true in the stock file: the games begin with policy-drawn moves that carry no search comment, and the record says how many
    openings = []
    for f in os.listdir(out / "tinynet" / "sgfs"):
        for line in open(out / "tinynet" / "sgfs" / f):
            start = int(re.search(r"startTurnIdx=(\d+)", line).group(1))
            body = line[line.index("C[startTurnIdx"):]
            nodes = body.split(";")[1:]
            assert all("C[" not in nd for nd in nodes[:start]) and (len(nodes) == start or "C[" in nodes[start])
            openings.append(start)
    assert max(openings) > 0, openings
    cheap = sum(v == 8 for v in visits)
    assert 0.3 < cheap / len(visits) < 0.7 and 32 in visits, (cheap, len(visits))
    assert set(visits) <= {8} | set(range(12, 33))       # a full search, a cheap one, or one reduced towards reducedVisitsMin (formula: CPU test)
    rows = 0
    for f in os.listdir(out / "tinynet" / "tdata"):
        with np.load(out / "tinynet" / "tdata" / f) as z:
            rows += z["globalTargetsNC"].shape[0]
    assert 0 < rows < len(visits)                  # unrecorded cheap searches are (mostly) not rows


@pytest.mark.gpu
def test_command_searches_fair_komi_and_lead_targets(tmp_path, stock_cfg, golden_dir):
    """komiAuto and estimateLeadProb through the command, with the trained g170 net on small boards: the komi of a game is drawn around the
    komi the net calls even for ITS empty board (found by the bisection searches of the side loop) instead of komiMean, and about half of the
    recorded rows carry a lead target (global target 21 with weight 29) from computeLead."""
    import shutil
    models = tmp_path / "models"; models.mkdir()
    shutil.copy(os.path.join(golden_dir, "models", "g170-b6c96-s175395328-d26788732.bin.gz"), models / "g170.bin.gz")
    settings = dict(STOCK_B18_SETTINGS, bSizes="7,9", bSizeRelProbs="1,1", allowRectangleProb="0", dataBoardLen="9", koRules="SIMPLE", multiStoneSuicideLegals="true",
                    komiAuto="true", komiStdev="0.0", maxVisits="20", maxMovesPerGame="30", rootNumSymmetriesToSample="2", nnCacheSizePowerOfTwo="10",
                    maxRowsPerTrainFile="100000", firstFileRandMinProp="1.0", cheapSearchProb="0", reduceVisits="false", initGamesWithPolicy="false",
                    estimateLeadProb="0.5", estimateLeadVisits="4", compensateKomiVisits="6", policySurpriseDataWeight="0", valueSurpriseDataWeight="0")
    cfg = tmp_path / "komi.cfg"
    cfg.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    out = tmp_path / "out"
    rc = C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", str(cfg), "-max-games-total", "16", "-games-per-gpu", "8", "-per-game-release"])
    assert rc == 0
    komi_by_size, lead_rows, rows = {}, 0, 0
    for f in os.listdir(out / "g170" / "tdata"):
        with np.load(out / "g170" / "tdata" / f) as z:
            planes = np.unpackbits(z["binaryInputNCHWPacked"], axis=2)[:, :, :81].reshape(-1, 22, 9, 9)
            gin, gt = z["globalInputNC"], z["globalTargetsNC"]
            for on, gi, g in zip(planes[:, 0], gin, gt):
                rows += 1
                lead_rows += int(g[29] > 0)
                komi_by_size.setdefault(int(on.sum()), set()).add(round(abs(float(gi[5])) * 20.0, 1))
    assert rows >= 16 * 10 and 0.25 < lead_rows / rows < 0.75, (lead_rows, rows)
    # the fair komi of the empty 7x7 board is not the fair komi of the empty 9x9 board (and neither is komiMean's 7.5 by construction)
    assert set(komi_by_size) == {49, 81} and komi_by_size[49] != komi_by_size[81], komi_by_size
    assert all(len(v) <= 6 for v in komi_by_size.values()), komi_by_size       # no komi noise configured: the few-visit estimates of one fair value, rounded (+ the first games' komiMean)


@pytest.mark.gpu
def test_command_forks_finished_games(tmp_path, stock_cfg):
    """earlyForkGameProb / forkGameProb through the command: finished games are forked (a position of theirs, replayed, plus one of a few random
    legal moves - the one the net scores best), forked games are marked gtype=fork, start from that position (startTurnIdx = its length) on the
    forked game's board, and their training rows carry the start-history length."""
    import re
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "tinynet.bin"), "tiny_reg", seed=3)
    settings = dict(STOCK_B18_SETTINGS, bSizes="7,9", bSizeRelProbs="1,1", allowRectangleProb="0", dataBoardLen="9", maxVisits="12", maxMovesPerGame="40",
                    rootNumSymmetriesToSample="2", nnCacheSizePowerOfTwo="10", maxRowsPerTrainFile="100000", firstFileRandMinProp="1.0", cheapSearchProb="0",
                    reduceVisits="false", initGamesWithPolicy="false", estimateLeadProb="0", komiAuto="false", komiMean="7", earlyForkGameProb="0.5",
                    earlyForkGameExpectedMoveProp="0.1", forkGameProb="0.9", forkGameMinChoices="2", earlyForkGameMaxChoices="4", forkGameMaxChoices="4",
                    forkCompensateKomiProb="0.5", policySurpriseDataWeight="0", valueSurpriseDataWeight="0")
    cfg = tmp_path / "forks.cfg"
    cfg.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    out = tmp_path / "out"
    assert C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", str(cfg), "-max-games-total", "40", "-games-per-gpu", "8", "-per-game-release"]) == 0
    games = []
    for f in os.listdir(out / "tinynet" / "sgfs"):
        for line in open(out / "tinynet" / "sgfs" / f):
            size = int(re.search(r"SZ\[(\d+)", line).group(1))
            start = int(re.search(r"startTurnIdx=(\d+)", line).group(1))
            gtype = re.search(r"gtype=(\w+)", line).group(1)
            moves = re.findall(r";([BW])\[([a-z]*)\]", line)
            games.append((size, start, gtype, moves))
    forked = [g for g in games if g[2] == "fork"]
    normal = [g for g in games if g[2] == "normal"]
    assert len(forked) >= 5 and len(normal) >= 8, (len(forked), len(normal))
    for size, start, _, moves in forked:
        assert start >= 1 and len(moves) > start
        # all but the last start move are the opening of some other game on the same board (the forked one); the last is the fork's own move
        assert any(g[0] == size and g[3][:start - 1] == moves[:start - 1] and g[3] is not moves for g in games), (size, start, moves[:start])
    assert all(g[1] == 0 for g in normal)
    rows_start = []
    for f in os.listdir(out / "tinynet" / "tdata"):
        with np.load(out / "tinynet" / "tdata" / f) as z:
            rows_start += list(z["globalTargetsNC"][:, 53])
    assert max(rows_start) >= 1 and min(rows_start) == 0


@pytest.mark.gpu
def test_command_records_side_positions(tmp_path, golden_dir):
    """forkSidePositionProb through the command (trained g170 net, 9x9): about that share of the turns gets a forking move off the main line whose
    position is searched on the side loop with the game's own search parameters; its row is written with the game - own policy / value targets,
    no outcome-dependent ones (global target 62 = 0 where the game's own rows have 1, ownership planes empty) - at the turn index after the fork."""
    import shutil
    models = tmp_path / "models"; models.mkdir()
    shutil.copy(os.path.join(golden_dir, "models", "g170-b6c96-s175395328-d26788732.bin.gz"), models / "g170.bin.gz")
    settings = dict(STOCK_B18_SETTINGS, bSizes="9", bSizeRelProbs="1", allowRectangleProb="0", dataBoardLen="9", koRules="SIMPLE", multiStoneSuicideLegals="true",
                    komiAuto="false", komiMean="7", komiStdev="0.0", maxVisits="16", maxMovesPerGame="300", rootNumSymmetriesToSample="2", nnCacheSizePowerOfTwo="10",
                    maxRowsPerTrainFile="100000", firstFileRandMinProp="1.0", cheapSearchProb="0", reduceVisits="false", initGamesWithPolicy="false",
                    estimateLeadProb="0", earlyForkGameProb="0", forkGameProb="0", forkSidePositionProb="0.25", policySurpriseDataWeight="0", valueSurpriseDataWeight="0")
    cfg = tmp_path / "side.cfg"
    cfg.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    out = tmp_path / "out"
    assert C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", str(cfg), "-max-games-total", "8", "-games-per-gpu", "8", "-per-game-release"]) == 0
    main_rows = side_rows = 0
    for f in os.listdir(out / "g170" / "tdata"):
        with np.load(out / "g170" / "tdata" / f) as z:
            g, own = z["globalTargetsNC"], z["valueTargetsNCHW"]
            side = (g[:, 62] == 0) & (g[:, 52] == 0)                    # not "game finished", and not because of the move limit
            main_rows += int((~side).sum()); side_rows += int(side.sum())
            assert (g[side, 60] == 16).all() and (g[side, 25] > 0).all()  # searched with the full budget, written with the game's weight
            assert not own[side][:, 0].any() and own[~side][:, 0].any()  # a side position has no final ownership
            assert (g[side, 51] >= 1).all()
    assert main_rows >= 8 * 20 and 0.1 * main_rows < side_rows < 0.4 * main_rows, (main_rows, side_rows)


@pytest.mark.gpu
@pytest.mark.parametrize("new_cfg", ["tiny_reg", "tiny_nbt"])
def test_command_moves_to_a_newer_net_while_games_run(tmp_path, stock_cfg, monkeypatch, new_cfg):
    """Model polling (command/selfplay.cpp:336-352): a newer file in the models directory is picked up while games are running.  Same
    architecture: the weights are swapped inside the live handle and the games go on (switchNetsMidGame); another architecture: the
    evaluator is rebuilt.  Either way the rows of games that end afterwards land in the new net's directory."""
    import time
    import numpy as np
    from katago_b200 import modelgen
    models = tmp_path / "models"; models.mkdir()
    modelgen.write_model(str(models / "net1.bin"), "tiny_reg", seed=3)
    calls = {"n": 0}
    orig = C.ModelPoller.poll

    def poll(self, force=False):
        calls["n"] += 1
        if calls["n"] == 4:
            path = modelgen.write_model(str(models / "net2.bin"), new_cfg, seed=4)
            os.utime(path, (time.time() + 60, time.time() + 60))
        return orig(self, force)
    monkeypatch.setattr(C.ModelPoller, "poll", poll)
    out = tmp_path / "out"
    rc = C.main(["-models-dir", str(models), "-output-dir", str(out), "-config", stock_cfg, "-max-games-total", "8", "-games-per-gpu", "4", "-per-game-release",
                 "-model-poll-seconds", "0", "-override-config",
                 "bSizes=9,bSizeRelProbs=1,dataBoardLen=9,maxVisits=16,maxMovesPerGame=30,rootNumSymmetriesToSample=2,nnCacheSizePowerOfTwo=10,maxRowsPerTrainFile=1000,firstFileRandMinProp=1.0,cheapSearchProb=0,reduceVisits=false"])
    assert rc == 0
    rows = {}
    for name in ("net1", "net2"):
        tdata = out / name / "tdata"
        rows[name] = sum(np.load(tdata / f)["globalTargetsNC"].shape[0] for f in os.listdir(tdata)) if tdata.exists() else 0
    assert rows["net2"] > 0, rows                 # games finished under the new net
    games = sum(sum(1 for _ in open(out / name / "sgfs" / f)) for name in ("net1", "net2") if (out / name / "sgfs").exists() for f in os.listdir(out / name / "sgfs"))
    assert games >= 8


def test_model_poller_reports_a_newer_file_once(tmp_path):
    import time
    a = tmp_path / "a.bin"; a.write_bytes(b"x")
    p = C.ModelPoller(str(tmp_path), str(a), 0.0)
    assert p.poll() is None
    b = tmp_path / "b.bin.gz"; b.write_bytes(b"y")
    os.utime(b, (time.time() + 5, time.time() + 5))
    assert p.poll() == str(b) and p.poll() is None
    older = tmp_path / "c.bin"; older.write_bytes(b"z")
    os.utime(older, (time.time() - 100, time.time() - 100))
    assert p.poll() is None
    slow = C.ModelPoller(str(tmp_path), str(a), 3600.0)
    assert slow.poll() is None and slow.poll(force=True) == str(b)
    assert C.model_name_of("/x/y/kata1-b18c384nbt-s123/model.bin.gz") == "kata1-b18c384nbt-s123" and C.model_name_of("/x/net7.bin.gz") == "net7"


def test_ranks_split_the_games_and_never_share_seeds_or_file_names():
    """One process per GPU: the ranks' game counts add up, their loop seeds, writer Rand streams (= file names) and game hashes differ."""
    from katago_b200.nn_backend import rand_uint32_stream
    for world in (1, 2, 8):
        plans = [C.shard_plan(r, world, 1001, 5) for r in range(world)]
        assert sum(p[0] for p in plans) == 1001 and max(p[0] for p in plans) - min(p[0] for p in plans) <= 1
        assert len({p[1] for p in plans}) == world and len({p[2] for p in plans}) == world
        streams = {tuple(rand_uint32_stream(p[2], 4).tolist()) for p in plans}
        assert len(streams) == world
    assert C.shard_plan(0, 4, 0, 1)[0] == 0                      # 0 = run until interrupted
    with pytest.raises(ValueError):
        C.shard_plan(4, 4, 10, 1)
    hashes = {C._game_hash(s, slot, i) for s in (1, 2) for slot in range(16) for i in range(16)}
    assert len(hashes) == 2 * 16 * 16 and all(0 <= a < 2 ** 64 and 0 <= b < 2 ** 64 for a, b in hashes)


def test_sgf_sink_appends_one_record_per_game(tmp_path):
    import gzip, json
    from test_npz_writer import _game_from_fixture, WRITEGAME_FIXTURES
    d = json.loads(gzip.open(WRITEGAME_FIXTURES[0], "rb").read())
    sink = C.SgfSink(str(tmp_path / "sgfs"), "seed:sgfs", "b200-black", "b200-white")
    sink.add(0, _game_from_fixture(d)); sink.add(3, _game_from_fixture(d))
    name = os.path.basename(sink.path)
    assert len(name) == 21 and name.endswith(".sgfs") and name[:16] == name[:16].upper()
    assert open(sink.path).read() == (d["sgf"] + "\n") * 2 and sink.count == 2


def _loader_case(which):
    """The .cfg variants both configuration loaders are compared on."""
    if which == "stock":
        settings = dict(STOCK_B18_SETTINGS)
    elif which == "almost_empty":       # every default comes from the loader
        settings = {"numSearchThreads": "1", "maxVisits": "500"}
    elif which == "dependent_defaults":  # defaults that follow other keys: rootPolicyTemperatureEarly, rootFpuLossProp, rootFpuReductionMax (setup.cpp:575-583)
        settings = {"numSearchThreads": "1", "maxVisits": "500", "rootNoiseEnabled": "true", "rootPolicyTemperature": "1.3", "fpuLossProp": "0.15"}
    elif which == "plain_fpu_weight":
        settings = {"numSearchThreads": "1", "maxVisits": "500", "fpuParentWeightByVisitedPolicy": "false", "fpuParentWeight": "0.4", "fpuParentWeightByVisitedPolicyPow": "3.0"}
    else:      # a value of its own for every key the loop implements
        settings = {"maxVisits": "777", "maxMovesPerGame": "321", "cpuctExploration": "0.93", "cpuctExplorationLog": "0.41", "cpuctExplorationBase": "350",
                    "fpuReductionMax": "0.13", "rootFpuReductionMax": "0.07", "fpuLossProp": "0.11", "rootFpuLossProp": "0.06", "fpuParentWeight": "0.3",
                    "fpuParentWeightByVisitedPolicy": "false", "fpuParentWeightByVisitedPolicyPow": "1.5", "valueWeightExponent": "0.35",
                    "cpuctUtilityStdevPrior": "0.33", "cpuctUtilityStdevPriorWeight": "1.7", "cpuctUtilityStdevScale": "0.85",
                    "rootDesiredPerChildVisitsCoeff": "3", "subtreeValueBiasFactor": "0.45", "subtreeValueBiasWeightExponent": "0.85",
                    "useGraphSearch": "false", "graphSearchRepBound": "9", "rootNoiseEnabled": "false", "rootDirichletNoiseTotalConcentration": "9.5",
                    "rootDirichletNoiseWeight": "0.2", "rootPolicyTemperature": "1.2", "rootPolicyTemperatureEarly": "1.4", "chosenMoveTemperature": "0.2",
                    "chosenMoveTemperatureEarly": "0.6", "chosenMoveTemperatureHalflife": "17", "chosenMoveTemperatureOnlyBelowProb": "0.9",
                    "chosenMoveSubtract": "1", "chosenMovePrune": "2", "useLcbForSelection": "false", "lcbStdevs": "4", "minVisitPropForLCB": "0.1",
                    "useNonBuggyLcb": "false", "winLossUtilityFactor": "0.9", "staticScoreUtilityFactor": "0.1", "dynamicScoreUtilityFactor": "0.2",
                    "dynamicScoreCenterZeroWeight": "0.3", "dynamicScoreCenterScale": "0.75", "noResultUtilityForWhite": "-0.1",
                    "drawEquivalentWinsForWhite": "0.6", "rootNumSymmetriesToSample": "2", "nnCacheSizePowerOfTwo": "18", "koRules": "POSITIONAL",
                    "multiStoneSuicideLegals": "false", "wideRootNoise": "0.04", "antiMirror": "true", "numSearchThreads": "1"}
    return settings


@pytest.mark.parametrize("which", ["stock", "every_key_changed", "almost_empty", "plain_fpu_weight", "dependent_defaults"])
def test_config_mapping_agrees_with_the_reference_loader(tmp_path, which):
    """The same .cfg through the reference's own ConfigParser + Setup::loadSingleParams and integration/b200params.h
    (`kgref_driver paramsmap`, answers stored by tests/reference_runs.py) and through selfplay_cli.py: every mapped field of
    kgb_selfplay_config agrees, defaults of absent keys included, and the C++ side reports the same search options as not implemented."""
    import json
    from katago_b200.nn_backend import SelfPlay
    from reference_runs import reference_run
    settings = _loader_case(which)
    path = tmp_path / "c.cfg"
    path.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    kw, data, report = C.selfplay_kwargs_from_cfg(C.parse_cfg(str(path)))
    ref = json.loads(reference_run("kgref_driver", ["paramsmap", path, kw["ko_rule"]]))
    sig = inspect.signature(SelfPlay.__init__)
    eff = {k: v.default for k, v in sig.parameters.items() if v.default is not inspect._empty}
    eff.update(kw)
    eff["komi"] = data["komi"]
    for k, v in ref.items():
        if k in ("unsupported", "komi", "multi_stone_suicide_legal"):      # rules come from the game initialiser, not from the search parameters
            continue
        assert k in eff, k
        assert abs(float(eff[k]) - float(v)) <= 1e-12, (k, eff[k], v)
    nb = " ".join(report["not_built"])
    for line in ref["unsupported"]:                   # search options the C++ side names must be named by the command too
        assert line.split(" = ")[0] in nb, (line, nb)


@pytest.fixture(scope="module")
def cpp_host(tmp_path_factory):
    """integration/b200_selfplay_main.cpp (the C++-only host of boundary 2) built against the library."""
    import subprocess
    exe = tmp_path_factory.mktemp("cpphost") / "b200_selfplay"
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", ROOT, os.path.join(ROOT, "integration", "b200_selfplay_main.cpp"), "-o", str(exe),
                    "-L", os.path.join(ROOT, "katago_b200"), "-lkgb200", "-lz", "-Wl,-rpath," + os.path.join(ROOT, "katago_b200")], check=True)
    return str(exe)


@pytest.mark.parametrize("which", ["stock", "every_key_changed", "almost_empty", "plain_fpu_weight", "dependent_defaults"])
def test_cpp_host_config_mapping_agrees_with_the_reference_loader(tmp_path, cpp_host, which):
    """The C++ host reads a .cfg by the reference's key names itself (no reference headers): its kgb_selfplay_config agrees field by field
    with the reference's own loader mapped by integration/b200params.h, defaults of absent keys included."""
    import json, subprocess
    from reference_runs import reference_run
    settings = {k: v.split(",")[0] for k, v in _loader_case(which).items() if k in C._SEARCH_KEYS or k in ("koRules", "multiStoneSuicideLegals", "numSearchThreads")}
    path = tmp_path / "c.cfg"
    path.write_text("".join(f"{k} = {v}\n" for k, v in settings.items()))
    mine = json.loads(subprocess.run([cpp_host, "-config", str(path), "-print-config"], capture_output=True, text=True, check=True).stdout)
    ref = json.loads(reference_run("kgref_driver", ["paramsmap", path, mine["ko_rule"]]))
    for k, v in ref.items():
        if k in ("unsupported", "komi", "multi_stone_suicide_legal"):      # rules are the game's, not the search parameters'
            continue
        assert abs(float(mine[k]) - float(v)) <= 1e-12, (k, mine[k], v)
    assert mine["debug_hold_at_max_visits"] == 1 and mine["num_games"] == 256


def test_cpp_host_refuses_what_it_does_not_play_and_needs_a_gpu(tmp_path, cpp_host, tmp_models):
    """Options this small host does not have are an error, not a silent difference; and without a CUDA device it stops with the library's
    error - there is no CPU path behind the C ABI."""
    import subprocess
    cfg = tmp_path / "c.cfg"
    cfg.write_text("maxVisits = 50\nnumGameThreads = 4\nbSizes = 9\nhandicapProb = 0.1\nscoringRules = AREA,TERRITORY\n")
    r = subprocess.run([cpp_host, "-config", str(cfg), "-model", tmp_models["tiny_reg"], "-output-dir", str(tmp_path), "-strict"], capture_output=True, text=True)
    assert r.returncode != 0 and "NOT BUILT (the loop runs WITHOUT it): handicapProb = 0.1" in r.stderr and "TERRITORY not built" in r.stderr and "-strict" in r.stderr
    cfg.write_text("maxVisits = 50\nnumGameThreads = 4\nbSizes = 9\nscoringRules = TERRITORY\n")
    r = subprocess.run([cpp_host, "-config", str(cfg), "-model", tmp_models["tiny_reg"], "-output-dir", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode != 0 and "none of these is built" in r.stderr
    cfg.write_text("maxVisits = 50\nnumGameThreads = 4\nbSizes = 9,13\ndataBoardLen = 9\n")
    r = subprocess.run([cpp_host, "-config", str(cfg), "-model", tmp_models["tiny_reg"], "-output-dir", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode != 0 and "dataBoardLen" in r.stderr          # the data frame must hold the largest board

    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the loud failure without one is checked on CPU boxes")
    cfg.write_text("maxVisits = 50\nnumGameThreads = 4\nbSizes = 9\n")
    r = subprocess.run([cpp_host, "-config", str(cfg), "-model", tmp_models["tiny_reg"], "-output-dir", str(tmp_path), "-max-games-total", "1"], capture_output=True, text=True)
    assert r.returncode != 0 and "b200_selfplay:" in r.stderr and not list(tmp_path.glob("*.sgf")), r.stderr


def test_slot_setups_hand_over_draws_forks_and_fair_komi():
    """The host side of the per-game setup (SlotSetups): every slot's NEXT game has its board, rules, komi and opening length on the device before it
    starts; a pooled fork replaces the draw (the forked game's setup, no opening, its moves played in when the game starts); komiAuto asks the side
    loop for the fair komi of the next game's empty board and redraws the komi around the answer - unless the game has started meanwhile."""
    from katago_b200.fork_play import ForkManager
    from katago_b200.game_initializer import GameInitializer
    import random

    class Loop:
        num_games = 4
        def __init__(self):
            self.calls = []
        def set_game_setup(self, s, also_current_games=False):
            self.calls.append(("setup", np.array(s).copy(), also_current_games))
        def set_komi(self, k, also_current_games=False):
            self.calls.append(("komi", np.array(k).copy(), also_current_games))
        def set_policy_init(self, n, t, also_current_games=False):
            self.calls.append(("init", np.array(n).copy(), t, also_current_games))
        def play_moves_game(self, g, moves):
            self.calls.append(("moves", g, list(moves)))

    class Searcher:
        def __init__(self):
            self.jobs = []
        def submit(self, gen, setup, moves, on_done):
            self.jobs.append((gen, setup, moves, on_done))

    class Rec:
        def __init__(self):
            self.started = []
        def start_from(self, g, moves, mode=2):
            self.started.append((g, list(moves), mode))

    init = GameInitializer([(9, 9), (13, 13)], [1, 1], ko_rules=(0, 1), multi_stone_suicide_legals=(True,), komi_mean=7.0, komi_stdev=0.0, seed=2)
    forks = ForkManager(dict(early_fork_game_prob=1.0, fork_compensate_komi_prob=0.0), random.Random(1))
    searcher, loop, rec = Searcher(), Loop(), Rec()
    slots = C.SlotSetups(init, 4, dict(enabled=True, area_prop=0.05, temperature=1.2), fair_komi=searcher, forks=forks, searcher=searcher)
    slots.start(loop)
    kinds = [c[0] for c in loop.calls]
    assert kinds[:3] == ["setup", "komi", "init"] and loop.calls[0][2] and loop.calls[1][2] and loop.calls[2][3]        # the games in progress ...
    assert kinds[3:6] == ["setup", "komi", "init"] and not loop.calls[3][2] and loop.calls[5][2] == 1.2                # ... and the ones after them
    assert len(searcher.jobs) == 4 and all(j[2] == [] for j in searcher.jobs)                                          # komiAuto: one empty-board job per slot
    # the fair-komi answer for slot 2 replaces its next game's komi (7.0 from komiMean) by a draw around it
    before = float(slots.komis[2])
    searcher.jobs[2][3](3.5)
    assert before == 7.0 and float(slots.komis[2]) == 3.5 and loop.calls[-1][0] == "komi"
    # slot 1's game ends: the new game is an ordinary one; the draw for the game after it pops the fork that is in the pool by then
    forks.add([(2, 2), (3, 3), (4, 4)], (13, 13, 1, 1), 5.5)
    n_jobs = len(searcher.jobs)
    slots.game_started(loop, rec, 1)
    assert rec.started == [] and tuple(slots.setups[1]) == (13, 13, 1, 1) and slots.openings[1] == 0 and float(slots.komis[1]) == 5.5
    assert slots.fork_next[1] is not None and len(searcher.jobs) == n_jobs                                             # no komiAuto job for a forked game
    # an answer that arrives for a slot whose draw has been replaced since is ignored
    searcher.jobs[1][3](1.0)
    assert float(slots.komis[1]) == 5.5
    # ... and when THAT game starts, the fork's moves are played into the slot and the recorder is told
    slots.game_started(loop, rec, 1)
    assert ("moves", 1, [(2, 2), (3, 3), (4, 4)]) in loop.calls and rec.started == [(1, [(2, 2), (3, 3), (4, 4)], 2)] and slots.fork_next[1] is None


def test_game_initializer_reproduces_the_reference_distributions(golden_dir):
    """200 000 games of the reference's GameInitializer::createGame (tests/golden/make_gameinit_fixture.py) against 200 000 draws of
    katago_b200/game_initializer.py from the same configuration: board sizes incl. rectangles, ko and suicide rules, and the komi histograms on
    9x9 and 19x19 (noise scaled by the board, big-stdev mixture, linear rounding, integers allowed half of the time) agree to sampling error."""
    import json
    from katago_b200.game_initializer import GameInitializer
    ref = json.load(open(os.path.join(golden_dir, "gameinit_hist.json")))
    cfg = C.parse_cfg("".join(f"{k} = {v}\n" for k, v in ref["cfg"].items()), is_text=True)
    _, data, report = C.selfplay_kwargs_from_cfg(cfg)
    assert report["fixed"] == []
    n = ref["n"]
    setups, komis = GameInitializer(seed=17, **data["game_init"]).draw_many(n)

    def tv(a, b):           # total variation distance of two histograms over the union of their keys
        keys = set(a) | set(b)
        return 0.5 * sum(abs(a.get(k, 0) / sum(a.values()) - b.get(k, 0) / sum(b.values())) for k in keys)
    mine_sizes = {}
    for x, y in setups[:, :2]:
        mine_sizes[f"{x}x{y}"] = mine_sizes.get(f"{x}x{y}", 0) + 1
    assert set(mine_sizes) == set(ref["sizes"]) and tv(mine_sizes, ref["sizes"]) < 0.005, (mine_sizes, ref["sizes"])
    assert tv({str(k): int((setups[:, 2] == k).sum()) for k in (0, 1, 2)}, ref["ko_rules"]) < 0.005
    assert tv({str(k): int((setups[:, 3] == k).sum()) for k in (0, 1)}, ref["multi_stone_suicide"]) < 0.005
    for size, edge in (("9x9", 9), ("19x19", 19)):
        sel = komis[(setups[:, 0] == edge) & (setups[:, 1] == edge)]
        mine = {}
        for k in sel:
            mine["%.1f" % k] = mine.get("%.1f" % k, 0) + 1
        d = tv(mine, ref["komi_by_size"][size])
        assert d < 0.012, (size, d)
        ints = sum(v for k, v in mine.items() if float(k) == int(float(k))) / len(sel)
        assert 0.2 < ints < 0.3, ints          # integers allowed half of the time: about a quarter of the komis
