"""bench.py --impl reference: the reference arm's JSON line (one line on stdout, the keys the driver reads) on a small
instance of the workload, and the rule that under torchrun only rank 0 runs it.  CPU only: the arm times the reference's
own anneal() (oracle/_ref/libref.so when the reference build is present, else the oracle port)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--nodes", "20000", "--edges", "200000", "--k", "8", "--cpu-moves", "50000"]


def _run(env_extra):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"] + SMALL,
                          capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "vertex-moves/sec" and line["unit"] == "moves/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["vs_baseline"] is None
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_without_work():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_and_dump_outputs_are_checked(tmp_path):
    """No timed step, or --dump-outputs where it is not implemented (other workloads, several ranks): a usage error before
    any work, nothing written."""
    out = str(tmp_path / "out")
    two_ranks = {"RANK": "0", "LOCAL_RANK": "0", "WORLD_SIZE": "2"}
    for args, env in ((["--steps", "0"], {}), (["--impl", "reference", "--dump-outputs", out], {}),
                      (["--workload", "c4", "--dump-outputs", out], {}), (["--dump-outputs", out], two_ranks)):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=60,
                           cwd=ROOT, env=dict(os.environ, **env))
        assert r.returncode == 2 and r.stdout == "" and "error:" in r.stderr, (args, r.stderr)
    assert not os.path.exists(out)
