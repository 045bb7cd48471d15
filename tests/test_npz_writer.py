"""CPU tests of the training-data container (SURVEY §8f row 1, container + schema layer)."""
import os, subprocess, sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from katago_b200 import npz_writer as W

GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_npy_headers_equal_the_reference_numpybuffer():
    """The 256-byte headers equal, byte for byte, what the reference's NumpyBuffer writes for the seven arrays (fixture:
    oracle/_ref/kgref_driver npyheader, tests/golden/make_npz_fixture.py) for 0, 1, 7 and 1024 rows."""
    d = np.load(os.path.join(GOLDEN, "npyheaders.npz"))
    sch = W.schema(19)
    for rows in (0, 1, 7, 1024):
        for name, (descr, rest) in sch.items():
            ref = bytes(d[f"r{rows}_{name}"])
            assert W.npy_header(descr, (rows,) + tuple(rest)) == ref, (rows, name)


def test_written_file_has_the_reference_schema_and_round_trips(tmp_path):
    rng = np.random.default_rng(0)
    n = 96
    sp = (rng.random((n, 361, 22)) < 0.2).astype(np.float32)
    gl = rng.standard_normal((n, 19)).astype(np.float32)
    visits = rng.integers(0, 50, (n, 362)).astype(np.float64)
    visits[visits < 25] = -1.0                      # no child there
    visits[:, 5] = 49.0
    rows = W.rows_from_root_observations(sp, gl, visits, turn_idx=np.arange(n), num_visits=np.maximum(visits, 0).sum(1))
    path = str(tmp_path / "rows.npz")
    assert W.write_npz(path, rows) == n
    with np.load(path) as z:
        # dtype and row shape of the reference's sample file python/testdata/benchmark_data_1024.npz (make_trainingdata_schema_fixture.py)
        ref = json.load(open(os.path.join(GOLDEN, "trainingdata_schema.json")))
        assert set(z.files) == set(W.schema()) == set(ref)
        for k, (descr, rest) in W.schema().items():
            assert z[k].dtype == np.dtype(descr) and z[k].shape == (n,) + tuple(rest)
            if k != "globalTargetsNC":          # the sample file is format version 2 (64 global targets)
                assert np.dtype(ref[k][0]) == z[k].dtype and tuple(ref[k][1]) == z[k].shape[1:], k
        # the reader's unpacking (python/katago/train/data_processing_pytorch.py:89-95) gives the planes back
        unpacked = np.unpackbits(z["binaryInputNCHWPacked"], axis=2)[:, :, :361]
        assert np.array_equal(unpacked, np.transpose(sp, (0, 2, 1)).astype(np.uint8))
        assert np.array_equal(z["policyTargetsNCMove"][:, 0], np.maximum(visits, 0).astype(np.int16))
        assert (z["policyTargetsNCMove"][:, 1] == 1).all()
        assert np.array_equal(z["globalInputNC"], gl)


@pytest.mark.skipif(not os.path.exists("/root/reference/python/katago/train/data_processing_pytorch.py"), reason="reference python not present")
def test_reference_training_reader_consumes_the_file(tmp_path):
    """Drop-in check: the reference's own training-data reader (python/katago/train/data_processing_pytorch.py) batches the file."""
    sys.path.insert(0, "/root/reference/python")
    import torch
    from katago.train import data_processing_pytorch as dp, modelconfigs
    rng = np.random.default_rng(1)
    n = 64
    sp = (rng.random((n, 361, 22)) < 0.2).astype(np.float32); sp[:, :, 0] = 1.0
    gl = np.zeros((n, 19), np.float32)
    visits = rng.integers(0, 30, (n, 362)).astype(np.float64)
    path = str(tmp_path / "rows.npz")
    W.write_npz(path, W.rows_from_root_observations(sp, gl, visits))
    cfg = modelconfigs.config_of_name["b2c16"]
    batches = list(dp.read_npz_training_data([path], batch_size=32, world_size=1, rank=0, pos_len=19, device=torch.device("cpu"),
                                             randomize_symmetries=False, include_meta=False, model_config=cfg))
    assert len(batches) == 2
    b = batches[0]
    assert tuple(b["binaryInputNCHW"].shape) == (32, 22, 19, 19) and tuple(b["policyTargetsNCMove"].shape)[0] == 32
    assert float(b["binaryInputNCHW"][:, 0].min()) == 1.0


def test_policy_target_follows_extract_policy_target():
    """Play::extractPolicyTarget: largest value scaled up to 10 when smaller, capped at 30000 when larger, rounded to int16."""
    t = W.policy_target_from_play_selection(np.array([[-1.0, 2.0, 0.5, -1.0], [-1.0, 60000.0, 15000.0, 1.0], [12.0, 3.4, -1.0, 7.5]]))
    assert t.tolist() == [[0, 10, 3, 0], [0, 30000, 7500, 1], [12, 3, 0, 8]]


# ---- TrainingWriteBuffers.add_row against the reference's own addRow (tests/golden/make_addrow_fixtures.py) -------------------------
import glob
import gzip
import json

ADDROW_FIXTURES = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "addrow_*.json.gz")))


def _replay_addrow_fixture(path):
    from katago_b200.npz_writer import RowRand, TrainingWriteBuffers
    d = json.loads(gzip.open(path, "rb").read())
    X, Y, L = d["X"], d["Y"], d["dataLen"]
    rows = d["rows"]
    buf = TrainingWriteBuffers(len(rows), L)
    rand = RowRand("addrow" + d["seed"])                 # one Rand for all rows of the file, like the reference's writer
    packed = (L * L + 7) // 8
    q_by_turn = [r["qTargets"] for r in rows]
    for r in rows:
        t = r["turnIdx"]
        buf.add_row(
            x_size=X, y_size=Y, next_player=r["nextPlayer"],
            packed_input=np.frombuffer(bytes.fromhex(r["out_binaryInputNCHWPacked"]), np.uint8).reshape(22, packed),
            global_input=np.asarray(r["out_globalInputNC"], np.float32),
            turn_idx=t, target_weight=r["targetWeight"], unreduced_num_visits=r["unreducedNumVisits"],
            policy_target0=r["policyTarget0"], policy_target1=r["policyTarget1"],
            policy_surprise=r["policySurprise"], policy_entropy=r["policyEntropy"], search_entropy=r["searchEntropy"],
            white_value_targets=d["valueTargets"], white_q_value_targets=q_by_turn[t], white_value_targets_idx=t,
            value_target_weight=r["valueTargetWeight"], td_value_target_weight=r["tdValueTargetWeight"],
            lead_target_weight_factor=r["leadTargetWeightFactor"], nn_raw_stats=r["nnRawStats"],
            final_full_area=d["finalFullArea"], final_ownership=d["finalOwnership"] if r["hasOwnership"] else None,
            final_white_scoring=d["finalWhiteScoring"] if r["hasScoring"] else None,
            pos_hist_for_future_boards=d["boards"] if r["hasFutureBoards"] else None,
            is_side_position=bool(r["isSidePosition"]), num_neural_nets_behind_latest=r["numNeuralNetsBehindLatest"],
            game_hash=d["gameHash"], num_changed_neural_nets=r["numChangedNeuralNets"], hit_turn_limit=bool(r["hitTurnLimit"]),
            num_extra_black=r["numExtraBlack"], mode=r["mode"], rand=rand, self_komi=r["selfKomi"],
            area_scoring_or_encore2=bool(r["areaScoringOrEncore2"]), start_hist_moves=d["startHistMoves"],
            initial_turn_number=r["initialTurnNumber"], white_bonus_now=r["whiteBonusScore"], white_bonus_end=d["endWhiteBonus"],
            end_finished=bool(d["endFinished"]), end_no_result=bool(d["endNoResult"]),
            always_pass_alive_under_suicide_rules=bool(r["alwaysComputePassAliveUnderSuicideRules"]), reanalysis=tuple(r["reanalysis"]))
    return d, buf


@pytest.mark.parametrize("path", ADDROW_FIXTURES, ids=[os.path.basename(p)[7:-8] for p in ADDROW_FIXTURES])
def test_add_row_matches_reference_add_row(path):
    """Every target array of every row equals what the reference's addRow wrote - bit for bit, including the stochastically
    rounded scoring plane and Q targets (same Rand, same draw order) and the float32 global targets."""
    d, buf = _replay_addrow_fixture(path)
    L = d["dataLen"]
    assert buf.cur_rows == len(d["rows"])
    for i, r in enumerate(d["rows"]):
        for name, key in (("policyTargetsNCMove", "out_policyTargetsNCMove"), ("scoreDistrN", "out_scoreDistrN"),
                          ("valueTargetsNCHW", "out_valueTargetsNCHW"), ("qValueTargetsNCMove", "out_qValueTargetsNCMove")):
            want = np.asarray(r[key], np.int64)
            got = buf.arrays[name][i].reshape(-1).astype(np.int64)
            assert np.array_equal(got, want), (i, name, np.flatnonzero(got != want)[:8])
        want = np.asarray(r["out_globalTargetsNC"], np.float32)
        got = buf.arrays["globalTargetsNC"][i]
        bad = np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))
        bad = [int(c) for c in bad if not (got[c] == 0 and want[c] == 0)]      # -0.0 vs 0.0 would still be reported by value below
        assert not bad, (i, bad, got[bad], want[bad])


def test_add_row_fixtures_cover_the_branches():
    """The fixtures exercise what addRow branches on: missing policy / ownership / future boards / scoring, no-result ending,
    bonus points, reanalysed rows, capped scores and leads, both colours, boards smaller than the data frame."""
    assert len(ADDROW_FIXTURES) >= 8
    seen = dict(p0_null=0, p1_null=0, own_null=0, fut_null=0, sc_null=0, rean=0, white=0, black=0, nores=0, bonus=0, small=0, capped=0, distr_low=0, distr_high=0,
                passalive=0, not_passalive=0)
    for path in ADDROW_FIXTURES:
        d = json.loads(gzip.open(path, "rb").read())
        seen["nores"] += d["endNoResult"]
        seen["bonus"] += d["endWhiteBonus"] != 0
        seen["small"] += d["X"] < d["dataLen"]
        for r in d["rows"]:
            seen["p0_null"] += r["policyTarget0"] is None
            seen["p1_null"] += r["policyTarget1"] is None
            seen["own_null"] += not r["hasOwnership"]
            seen["fut_null"] += not r["hasFutureBoards"]
            seen["sc_null"] += not r["hasScoring"]
            seen["rean"] += r["reanalysis"][0]
            seen["passalive"] += r["alwaysComputePassAliveUnderSuicideRules"] == 1 and r["out_globalTargetsNC"][68] == 1.0
            seen["not_passalive"] += r["alwaysComputePassAliveUnderSuicideRules"] == 0 and r["out_globalTargetsNC"][68] == 0.0
            seen["white"] += r["nextPlayer"] == 2
            seen["black"] += r["nextPlayer"] == 1
            seen["distr_low"] += r["out_scoreDistrN"][0] == 100
            seen["distr_high"] += r["out_scoreDistrN"][-1] == 100
            seen["capped"] += abs(r["out_globalTargetsNC"][21]) == 421.0 or abs(r["out_globalTargetsNC"][3]) == 421.0
    assert all(v > 0 for v in seen.values()), seen


def test_training_write_buffers_file_is_read_back(tmp_path):
    """write_to_zip_file: the rows of a replayed fixture survive the container (np.load) unchanged."""
    d, buf = _replay_addrow_fixture(ADDROW_FIXTURES[0])
    path = str(tmp_path / "rows.npz")
    assert buf.write_to_zip_file(path) == len(d["rows"])
    with np.load(path) as z:
        for k, v in buf.arrays.items():
            assert np.array_equal(z[k], v[:buf.cur_rows]) and z[k].dtype == v.dtype


# ---- TrainingDataWriter.write_game against the reference's own writeGame (tests/golden/make_writegame_fixtures.py) ------------------

WRITEGAME_FIXTURES = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "writegame_*.json.gz")))
ARRAY_NAMES = ["binaryInputNCHWPacked", "globalInputNC", "policyTargetsNCMove", "globalTargetsNC", "scoreDistrN", "valueTargetsNCHW", "qValueTargetsNCMove"]


def _parse_text_dump(text):
    """The writer's text sink (TrainingWriteBuffers::writeToTextOstream, trainingwrite.cpp:888-983): per flush, per array: name,
    header line, one line per row, blank line.  Returns a list of flushes, each {name: list of rows}."""
    flushes, cur, lines, i = [], None, text.split("\n"), 0
    while i < len(lines):
        ln = lines[i]
        if ln in ARRAY_NAMES:
            if ln == ARRAY_NAMES[0]:
                cur = {}
                flushes.append(cur)
            rows, i = [], i + 2                     # skip the header line
            while i < len(lines) and lines[i] != "":
                rows.append(lines[i])
                i += 1
            cur[ln] = rows if ln == ARRAY_NAMES[0] else [np.array(r.split(), np.float64) for r in rows]
        i += 1
    return flushes


def _game_from_fixture(d):
    from katago_b200.npz_writer import FinishedGameData, SidePosition
    L = d["dataLen"]
    packed = (L * L + 7) // 8
    g = FinishedGameData(d["X"], d["Y"], d["komi"])
    g.game_hash, g.mode, g.training_weight = d["gameHash"], d["mode"], d["trainingWeight"]
    g.draw_equivalent_wins_for_white = d["drawEquivalentWinsForWhite"]
    g.hit_turn_limit, g.num_extra_black = bool(d["hitTurnLimit"]), d["numExtraBlack"]
    g.end_finished, g.end_no_result = bool(d["endFinished"]), bool(d["endNoResult"])
    g.boards_by_turn = d["boards"]
    g.white_value_targets_by_turn = d["valueTargets"]
    g.changed_neural_net_turns = d["changedNeuralNetTurns"]
    g.final_full_area, g.final_ownership, g.final_white_scoring = d["finalFullArea"], d["finalOwnership"], d["finalWhiteScoring"]
    for t in d["turns"]:
        g.next_player_by_turn.append(t["nextPlayer"])
        g.packed_input_by_turn.append(np.frombuffer(bytes.fromhex(t["packedInput"]), np.uint8).reshape(22, packed))
        g.global_input_by_turn.append(np.asarray(t["globalInput"], np.float32))
        g.target_weight_by_turn.append(t["targetWeight"])
        g.policy_targets_by_turn.append((t["policyTarget"], t["unreducedNumVisits"]))
        g.white_q_value_targets_by_turn.append(t["qTargets"])
        g.policy_surprise_by_turn.append(t["policySurprise"]); g.policy_entropy_by_turn.append(t["policyEntropy"]); g.search_entropy_by_turn.append(t["searchEntropy"])
        g.nn_raw_stats_by_turn.append(t["nnRawStats"])
        if "reanalysis" in t:
            g.reanalysis_by_turn.append(tuple(t["reanalysis"]))
    g.moves = [tuple(m) for m in d["moves"]]
    g.start_moves = [tuple(m) for m in d.get("startMoves", [])]      # startHist: moves before the training period (KGREF_START_MOVES)
    g.start_hist_moves = len(g.start_moves)
    g.winner, g.final_white_minus_black_score = d["winner"], d["finalWhiteMinusBlackScore"]
    g.changed_neural_net_names = d.get("changedNeuralNetNames")
    for sp in d.get("sidePositions", []):
        g.side_positions.append(SidePosition(
            sp["nextPlayer"], sp["turnIdx"], np.frombuffer(bytes.fromhex(sp["packedInput"]), np.uint8).reshape(22, packed),
            np.asarray(sp["globalInput"], np.float32), sp["policyTarget"], sp["unreducedNumVisits"], sp["valueTargets"], sp["qTargets"],
            sp["policySurprise"], sp["policyEntropy"], sp["searchEntropy"], sp["nnRawStats"], target_weight=sp["targetWeight"],
            num_neural_net_changes_so_far=sp["numNeuralNetChangesSoFar"]))
    return g


@pytest.mark.parametrize("path", WRITEGAME_FIXTURES, ids=[os.path.basename(p)[10:-8] for p in WRITEGAME_FIXTURES])
def test_write_game_matches_reference_write_game(path):
    """Same files (row counts per flush, incl. the randomised first file), same rows in the same order, same integer targets
    (the scoring plane and Q targets depend on every earlier Rand draw, so the draw order is checked too); float arrays to the
    6 digits the reference's text sink prints."""
    from katago_b200.npz_writer import TrainingDataWriter
    d = json.loads(gzip.open(path, "rb").read())
    want = _parse_text_dump(d["dump"])
    got = []
    w = TrainingDataWriter(None, d["maxRows"], d["firstFileMinRandProp"], d["dataLen"], "writegame" + d["seed"],
                           on_flush=lambda b: got.append({k: v[:b.cur_rows].copy() for k, v in b.arrays.items()}))
    w.write_game(_game_from_fixture(d))
    w.flush_if_nonempty()
    assert [len(f["globalTargetsNC"]) for f in want] == [len(f["globalTargetsNC"]) for f in got]
    assert w.row_count == sum(len(f["globalTargetsNC"]) for f in want)
    for fw, fg in zip(want, got):
        n = len(fw["globalTargetsNC"])
        assert [bytes.fromhex(r) for r in fw["binaryInputNCHWPacked"]] == [fg["binaryInputNCHWPacked"][i].tobytes() for i in range(n)]
        for name in ("policyTargetsNCMove", "scoreDistrN", "valueTargetsNCHW", "qValueTargetsNCMove"):
            a = np.stack(fw[name]).astype(np.int64)
            b = fg[name].reshape(n, -1).astype(np.int64)
            assert np.array_equal(a, b), (name, np.argwhere(a != b)[:5])
        for name in ("globalInputNC", "globalTargetsNC"):
            a = np.stack(fw[name])
            b = fg[name].reshape(n, -1).astype(np.float64)
            assert np.allclose(a, b, rtol=2e-5, atol=1e-30), (name, np.argwhere(~np.isclose(a, b, rtol=2e-5))[:5])


def test_final_value_targets_and_scoring_match_the_reference_game_end():
    """final_value_targets / scoring_from_area against what the driver computed with the reference's game-end code
    (endAndScoreGameNow, ScoreValue::whiteWinsOfWinner / whiteScoreDrawAdjust, NNInputs::fillScoring)."""
    from katago_b200.npz_writer import final_value_targets, scoring_from_area
    for path in WRITEGAME_FIXTURES:
        d = json.loads(gzip.open(path, "rb").read())
        want = d["valueTargets"][-1]
        got = final_value_targets(d["winner"], d["finalWhiteMinusBlackScore"], d["drawEquivalentWinsForWhite"], d["komi"], bool(d["endNoResult"]))
        assert [float(np.float32(v)) for v in want[:4]] == [float(v) for v in got[:4]]
        if not d["endNoResult"]:
            assert want[4] == 1 and np.float32(want[5]) == got[5]
        assert np.array_equal(scoring_from_area(d["finalOwnership"]), np.asarray(d["finalWhiteScoring"], np.float32))


def test_writer_file_names_and_split(tmp_path):
    """Real files: <16 hex digits>.npz named by the writer's Rand, rows split at max_rows_per_file, all rows present."""
    from katago_b200.npz_writer import TrainingDataWriter
    d = json.loads(gzip.open(WRITEGAME_FIXTURES[0], "rb").read())
    w = TrainingDataWriter(str(tmp_path), 10, 1.0, d["dataLen"], "files")
    w.write_game(_game_from_fixture(d))
    w.flush_if_nonempty()
    files = sorted(os.listdir(tmp_path))
    assert all(len(f) == 20 and f.endswith(".npz") and f[:16] == f[:16].upper() for f in files)
    rows = [np.load(os.path.join(tmp_path, f))["globalTargetsNC"].shape[0] for f in files]
    assert sum(rows) == w.row_count and max(rows) <= 10 and len(files) == -(-w.row_count // 10)


@pytest.mark.parametrize("path", WRITEGAME_FIXTURES, ids=[os.path.basename(p)[10:-8] for p in WRITEGAME_FIXTURES])
def test_sgf_equals_the_reference_write_sgf(path):
    """The game record written next to the rows: character for character the reference's WriteSgf::writeSgf output for the same game."""
    from katago_b200.npz_writer import write_sgf
    d = json.loads(gzip.open(path, "rb").read())
    assert write_sgf(_game_from_fixture(d), "b200-black", "b200-white") == d["sgf"]


@pytest.mark.skipif(not os.path.exists("/root/reference/python/shuffle.py"), reason="reference python not present")
def test_files_go_through_the_reference_shuffler_into_its_training_reader(tmp_path):
    """SURVEY §8f row 1: "must drop straight into python/shuffle.py -> train.py".  Full rows (every target filled by add_row) written as
    .npz files, shuffled by the reference's own shuffle.py, read back by its training reader: no row is lost or altered."""
    import torch
    src = tmp_path / "selfplay"; out = tmp_path / "shuffled"; scratch = tmp_path / "scratch"
    for d in (src, out, scratch):
        d.mkdir()
    total = []
    for i, p in enumerate(p for p in ADDROW_FIXTURES if "_in_19" in p or "19x19" in p):
        _, buf = _replay_addrow_fixture(p)
        buf.write_to_zip_file(str(src / ("%016X.npz" % (i + 1))))
        total.append({k: v[:buf.cur_rows].copy() for k, v in buf.arrays.items()})
    n = sum(t["globalTargetsNC"].shape[0] for t in total)
    r = subprocess.run([sys.executable, "/root/reference/python/shuffle.py", str(src), "-min-rows", "10", "-keep-target-rows", "all", "-out-dir", str(out),
                        "-out-tmp-dir", str(scratch), "-num-processes", "1", "-approx-rows-per-out-file", "64"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    files = sorted(str(out / f) for f in os.listdir(out) if f.endswith(".npz"))
    shuffled = {k: np.concatenate([np.load(f)[k] for f in files]) for k in W.schema(19)}
    assert shuffled["globalTargetsNC"].shape[0] == n
    key = lambda a: sorted(map(bytes, np.ascontiguousarray(a).reshape(a.shape[0], -1)))      # rows as a multiset
    for k in W.schema(19):
        assert key(shuffled[k]) == key(np.concatenate([t[k] for t in total])), k
    sys.path.insert(0, "/root/reference/python")
    from katago.train import data_processing_pytorch as dp, modelconfigs
    batches = list(dp.read_npz_training_data(files, batch_size=16, world_size=1, rank=0, pos_len=19, device=torch.device("cpu"),
                                             randomize_symmetries=False, include_meta=False, model_config=modelconfigs.config_of_name["b2c16"]))
    assert len(batches) >= n // 16 - len(files) and all(tuple(b["globalTargetsNC"].shape) == (16, 80) for b in batches)


@pytest.mark.skipif(not os.path.exists("/root/reference/python/train.py"), reason="reference python not present")
def test_reference_trainer_trains_on_our_files(tmp_path):
    """The whole consumer side of SURVEY §8f row 1 with the reference's own, unmodified tools: games written by TrainingDataWriter ->
    python/shuffle.py -> python/train.py (one small epoch of its smallest net on the CPU) -> validation pass.  Every loss term the
    trainer computes from our targets (policy, value, TD values, ownership, scoring, future position, score distribution, ...) is finite."""
    d_in, d_out, d_tmp, d_data, d_tr = (tmp_path / n for n in ("in", "out", "tmp", "data", "tr"))
    for d in (d_in, d_out, d_tmp, d_data / "train", d_data / "val"):
        d.mkdir(parents=True)
    w = W.TrainingDataWriter(str(d_in), 64, 1.0, 9, "trainpipe")
    for p in WRITEGAME_FIXTURES:
        d = json.loads(gzip.open(p, "rb").read())
        if d["dataLen"] == 9:
            for _ in range(3):
                w.write_game(_game_from_fixture(d))
    w.flush_if_nonempty()
    r = subprocess.run([sys.executable, "/root/reference/python/shuffle.py", str(d_in), "-min-rows", "10", "-keep-target-rows", "all", "-out-dir", str(d_out),
                        "-out-tmp-dir", str(d_tmp), "-num-processes", "1", "-approx-rows-per-out-file", "128"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    files = sorted(f for f in os.listdir(d_out) if f.endswith(".npz"))
    assert len(files) >= 2
    for f in files:
        dst = d_data / ("val" if f == files[-1] else "train")
        os.replace(d_out / f, dst / f)
        os.replace(d_out / f.replace(".npz", ".json"), dst / f.replace(".npz", ".json"))
    (d_data / "train.json").write_text(json.dumps({"range": [0, w.row_count]}))
    r = subprocess.run([sys.executable, "train.py", "-traindir", str(d_tr), "-datadir", str(d_data), "-pos-len", "9", "-batch-size", "32", "-model-kind", "b2c16",
                        "-samples-per-epoch", "128", "-max-epochs-this-instance", "1", "-no-compile", "-no-export", "-quit-if-no-data", "-max-val-samples", "64"],
                       cwd="/root/reference/python", capture_output=True, text=True, timeout=900, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "Finished training subepoch" in r.stdout + r.stderr                 # the optimiser stepped through the training batches
    last = json.loads((d_tr / "metrics_val.json").read_text().strip().splitlines()[-1])
    losses = {k: v for k, v in last.items() if k.endswith("loss")}
    assert len(losses) >= 10 and all(np.isfinite(v) for v in losses.values()), losses
