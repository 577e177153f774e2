"""CPU checks of the measurement contract pieces that do not need a GPU: workloads cover BASELINE.json's configs, the committed
ncu capture feeds `roofline.traffic`, the reference arm answers for every workload, the default flags finish within minutes."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workloads_cover_baseline_configs():
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    text = " ".join(w[3] for w in bench.WORKLOADS.values())
    for key in ("TinyLlama", "MiniLM", "Mistral-7B", "Qwen2.5-7B", "Mixtral-8x7B"):
        assert any(key in c for c in base["configs"]) and key in text, key
    assert bench.WORKLOADS["mistral7b_b1"][1:3] == (1, 2048) and bench.WORKLOADS["mistral7b_b64"][1] == 64
    assert bench.WORKLOADS["minilm_256x128"][1:3] == (256, 128) and bench.WORKLOADS["mixtral8x7b_b32"][1] == 32


def test_ncu_traffic_matches_algorithmic_bytes():
    """profiles/rNN_persistent*_full_raw.csv (newest round): DRAM bytes per decode step of the persistent kernel == weights once +
    KV once (Mistral-7B b=1, KV 2048: 14.490 GB, SURVEY.md section 8d) within 1 %, and the line names the file it comes from."""
    import bench
    t, src = bench.ncu_traffic_per_step()
    assert t is not None and abs(t / 14.490e9 - 1.0) < 0.01, t
    assert "profiles/" in src


def test_reference_arm_answers_for_workloads_without_a_cpu_leg():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "mixtral8x7b_b32"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" in line


def test_peaks_come_from_measured_file_or_documented_fallback():
    import bench
    hbm, src = bench.peaks("hbm")
    tf, _ = bench.peaks("tensor")
    assert 5000 < hbm < 9000 and 1000 < tf < 2500 and ("measured" in src or "fallback" in src)


def test_reference_arm_times_whole_steps_with_every_core_under_a_launcher_that_pins_one_thread():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm (rank 0 alone) must still use every host core, and when the
    model fits the host it times WHOLE decode steps (TinyLlama: 4.1 GB f32), so ms_per_step x steps is time actually spent."""
    import time
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    t0 = time.time()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tinyllama_b1", "--gpus", "2",
                        "--steps", "6", "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env)
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["extrapolated"] is False and line["cpu_baseline"]["extrapolated"] is False
    assert line["cpu_baseline"]["cores"] == (os.cpu_count() or 1) or (os.cpu_count() or 1) == 1
    assert line["steps"] * line["ms_per_step"] / 1e3 < wall       # the claimed steps fit inside the run
    # the other ranks of the launch exit without work and without output
    env["RANK"] = "1"
    r1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tinyllama_b1", "--gpus", "2"],
                        capture_output=True, text=True, timeout=120, env=env)
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_dump_outputs_writes_exact_ids_and_refuses_more_than_64_mb(tmp_path):
    """--dump-outputs: one DIR/<name>.npy per output, token ids as float64 (every uint32 exactly), real values as float32; an
    output set above 64 MB is refused before anything is written."""
    import numpy as np
    import pytest
    import bench
    ids = np.array([5, 151935, 2**32 - 1], dtype=np.uint32)
    emb = np.linspace(-1, 1, 12, dtype=np.float32).reshape(3, 4)
    bench.dump_outputs(str(tmp_path / "out"), {"next_token_ids": ids, "embeddings": emb})
    got_ids, got_emb = np.load(tmp_path / "out" / "next_token_ids.npy"), np.load(tmp_path / "out" / "embeddings.npy")
    assert got_ids.dtype == np.float64 and np.array_equal(got_ids, ids)
    assert got_emb.dtype == np.float32 and np.array_equal(got_emb, emb)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros((8 << 20) + 1, dtype=np.float64)})
    assert not (tmp_path / "big").exists()


def test_compare_sharded_counts_rows_only_while_routing_agrees():
    """bench.compare_sharded with router records: a sequence rerouted on a near-tie leaves the comparison from that step on; a
    disagreement off a tie, or a large error in a row that was routed identically, fails the check."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(0)
    steps, b, L, k, V = 4, 3, 2, 2, 50
    want = rng.standard_normal((steps, b, V)).astype(np.float32)
    sel = [np.tile(np.array([1, 4], dtype=np.int32), (b, 1, L, 1)) for _ in range(steps)]
    mar = [np.full((b, 1, L), 0.2, dtype=np.float32) for _ in range(steps)]
    got = want + 1e-3
    ok = bench.compare_sharded(got, want, "x", routing=([x.copy() for x in sel], sel, mar))
    assert ok["greedy32"] and ok["router_disagreements"] == 0 and ok["rows_compared"] == steps * b
    # sequence 1 reroutes at step 2 on a near-tie: its rows 2.. may differ by anything, [4, 1] vs [1, 4] is the same set
    sel_g = [x.copy() for x in sel]
    sel_g[2][1, 0, 1] = [1, 6]
    sel_g[0][0, 0, 0] = [4, 1]
    mar2 = [x.copy() for x in mar]
    mar2[2][1, 0, 1] = 2e-5
    got2 = got.copy()
    got2[2:, 1] += 1.5
    r = bench.compare_sharded(got2, want, "x", routing=(sel_g, sel, mar2))
    assert r["greedy32"] and r["router_disagreements"] == 1 and r["rows_compared"] == steps * b - 2 and r["max_abs_all_rows"] > 1
    # the same disagreement with a wide margin is a defect
    assert not bench.compare_sharded(got2, want, "x", routing=(sel_g, sel, mar))["greedy32"]
    # consequences of a reroute are not defects: after the near-tie reroute of sequence 1 (step 2, layer 1) its picks in the following
    # calls -- and, inside one call, the picks of later layers at the same or later positions -- are made on different hidden states
    # and may differ at ANY margin; a wide-margin disagreement that nothing earlier can have caused (sequence 2, layer 0) stays a defect
    sel_c = [x.copy() for x in sel_g]
    sel_c[3][1, 0, 0] = [2, 7]
    r = bench.compare_sharded(got2, want, "x", routing=(sel_c, sel, mar2))
    assert r["greedy32"] and r["router_disagreements"] == 2 and r["consequences_of_an_earlier_reroute"] == 1 and r["disagreements_off_a_tie"] == 0
    sel_p = [np.tile(np.array([1, 4], dtype=np.int32), (b, 3, L, 1))] + [x.copy() for x in sel[1:]]      # a 3-token first call
    mar_p = [np.full((b, 3, L), 0.2, dtype=np.float32)] + [x.copy() for x in mar[1:]]
    sel_pg = [x.copy() for x in sel_p]
    sel_pg[0][0, 1, 0] = [1, 5]
    mar_p[0][0, 1, 0] = 1e-5            # root: position 1, layer 0, on a tie
    sel_pg[0][0, 2, 1] = [3, 4]         # later position, later layer, wide margin: a consequence
    got4 = got.copy()
    got4[:, 0] += 2.0
    r = bench.compare_sharded(got4, want, "x", routing=(sel_pg, sel_p, mar_p))
    assert r["greedy32"] and r["consequences_of_an_earlier_reroute"] == 1 and r["rows_compared"] == steps * (b - 1)
    sel_pg[0][2, 0, 1] = [3, 4]         # position 0 of another sequence at a wide margin: nothing precedes it
    assert not bench.compare_sharded(got4, want, "x", routing=(sel_pg, sel_p, mar_p))["greedy32"]
    # a large error where the routing agreed is a defect
    got3 = got.copy()
    got3[1, 0] += 0.5
    assert not bench.compare_sharded(got3, want, "x", routing=([x.copy() for x in sel], sel, mar))["greedy32"]
    assert not bench.compare_sharded(got3, want, "x")["greedy32"] and bench.compare_sharded(got, want, "x")["greedy32"]
