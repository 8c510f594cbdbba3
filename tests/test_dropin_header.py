"""The drop-in header scema_b200/host/strain2spline_b200.h against the reference header itself: one
caller (tests/helpers/dropin_driver.cc, written only against the MatHistPredict API and shaped like
FE_problem.h:1091-1270) is compiled against both; stdout and every result file must be identical.

The reference side runs live where oracle/_ref is built; elsewhere its recorded outputs are used
(tests/golden/reference_runs.json: exit code and SHA-256 of stdout, of stderr and of the set of result
files, written by tests/golden/make_golden_live.py)."""
import hashlib
import json
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "dropin_driver_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_runs.json")

# (key, driver arguments after the output directory, environment of both runs)
CASES = [(f"same_{n_qp}_{n_steps}_{P}_{thr!r}_{seed}", [str(n_qp), str(n_steps), str(P), repr(thr), str(seed)], {})
         for n_qp, n_steps, P, thr, seed in [(64, 12, 10, 1e-6, 5), (300, 21, 10, 4e-7, 9), (41, 7, 4, 1e-6, 2)]]
CASES += [(f"legacy_{legacy}", ["120", "12", "10", "1e-6", "4"], {"DROPIN_LEGACY": legacy}) for legacy in ("1", "2")]
CASES += [(f"error_{n_steps}", ["16", n_steps, "10", "1e-6", "1"], {}) for n_steps in ("2", "0")]
# what the drop-in header needs on top to write the reference's legacy outputs (the reference header always writes them),
# as test_legacy_outputs_on_request passes it
DROPIN_KNOBS = {"legacy_1": {"SCEMA_B200_ALL_SIMILAR": "1"}, "legacy_2": {"SCEMA_B200_NEAREST": "1"}}


def sha(data):
    return hashlib.sha256(data if isinstance(data, bytes) else data.encode()).hexdigest()


def run_driver(exe, d, args, env=None):
    """Runs the driver into the new directory d -> {returncode, stdout, stderr, files: {name: sha256}}."""
    os.makedirs(d)
    r = subprocess.run([exe, str(d)] + args, capture_output=True, text=True, timeout=600, env=dict(os.environ, **(env or {})))
    files = {}
    for f in sorted(os.listdir(d)):
        with open(os.path.join(d, f), "rb") as fh:
            files[f] = sha(fh.read())
    return {"returncode": r.returncode, "stdout": r.stdout, "stderr": r.stderr, "files": files}


def summary(run):
    """A run as it is recorded: exit code, digests of stdout and stderr, number and digest of the result files."""
    return {"returncode": run["returncode"], "stdout": sha(run["stdout"]), "stderr": sha(run["stderr"]), "files": len(run["files"]),
            "files_sha256": sha("".join(f"{f} {h}\n" for f, h in sorted(run["files"].items())))}


def same_run(ours, ref, stderr=False):
    """Our run gave the reference's exit code, stdout and result files (and stderr, when asked: successful runs of the
    two builds may log differently)."""
    got = summary(ours)
    keys = [k for k in got if stderr or k != "stderr"]
    return {k: got[k] for k in keys} == {k: ref[k] for k in keys}


def reference_run(key, tmp_path):
    """summary() of the reference header's run of a case: live where oracle/_ref is built, else the recorded one."""
    args, env = {k: (a, e) for k, a, e in CASES}[key]
    if os.path.exists(REF_BIN):
        return summary(run_driver(REF_BIN, tmp_path / ("ref_" + key), args, env))
    with open(GOLDEN) as f:
        return json.load(f)["dropin"][key]


def ours_run(exe, key, d):
    args, env = {k: (a, e) for k, a, e in CASES}[key]
    return run_driver(exe, d, args, dict(env, **DROPIN_KNOBS.get(key, {})))


def build_ours(tmp_path):
    exe = str(tmp_path / "dropin_driver_b200")
    subprocess.check_call(["g++", "-std=c++11", "-O2", "-ffp-contract=off", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "scema_b200", "host"),
                           os.path.join(ROOT, "tests", "helpers", "dropin_driver.cc"), "-o", exe,
                           "-L" + os.path.join(ROOT, "scema_b200"), "-lscema_hist",
                           "-Wl,-rpath," + os.path.join(ROOT, "scema_b200")])
    return exe


@pytest.mark.parametrize("n_qp,n_steps,P,thr,seed", [(64, 12, 10, 1e-6, 5), (300, 21, 10, 4e-7, 9), (41, 7, 4, 1e-6, 2)])
def test_same_caller_same_bytes(tmp_path, n_qp, n_steps, P, thr, seed):
    key = f"same_{n_qp}_{n_steps}_{P}_{thr!r}_{seed}"
    ref = reference_run(key, tmp_path)
    ours = ours_run(build_ours(tmp_path), key, tmp_path / "ours")
    assert ours["returncode"] == 0, ours["stderr"]
    assert same_run(ours, ref)
    assert "flagged" in ours["stdout"] and "run_new_md" in ours["stdout"] and len(ours["files"]) > n_qp
    assert any(h != sha(b"") for f, h in ours["files"].items() if f.endswith("similar_hist"))


def test_in_process_pattern_uploads_only_the_new_samples(tmp_path):
    """FE_problem.h's pattern (append a sample to every point, fit every point, compare the flagged subset) keeps the
    histories on the GPU: one store build, then 48 bytes per point and NEW timestep — same bytes out as the reference,
    and as the flat-upload path (SCEMA_B200_STORE=0)."""
    ours_exe = build_ours(tmp_path)
    n_qp, n_steps = 300, 21
    key = "same_300_21_10_4e-07_9"
    runs = {}
    for name, env in (("store", {"DROPIN_STATS": "1"}), ("flat", {"DROPIN_STATS": "1", "SCEMA_B200_STORE": "0"})):
        runs[name] = run_driver(ours_exe, tmp_path / name, {k: a for k, a, _ in CASES}[key], env)
        assert runs[name]["returncode"] == 0, (name, runs[name]["stderr"])
    ref = reference_run(key, tmp_path)
    assert runs["store"]["stdout"] == runs["flat"]["stdout"] and runs["store"]["files"] == runs["flat"]["files"]
    assert same_run(runs["store"], ref)
    errs = {name: r["stderr"] for name, r in runs.items()}
    stats = dict(kv.split("=") for kv in errs["store"].split("store:")[1].split())
    # comparisons at t = 3, 5, 10, 15, 20, 21: one build (3 samples), then exactly the samples added since: 21 in total
    assert int(stats["rebuilds"]) == 1 and int(stats["appended_steps"]) == n_steps and int(stats["flat_uploads"]) == 0, stats
    assert int(stats["h2d_bytes"]) == 48 * n_qp * n_steps, stats
    flat = dict(kv.split("=") for kv in errs["flat"].split("store:")[1].split())
    assert int(flat["appended_steps"]) == 0 and int(flat["rebuilds"]) == 0


@pytest.mark.parametrize("legacy,env", [("1", {"SCEMA_B200_ALL_SIMILAR": "1"}), ("2", {"SCEMA_B200_NEAREST": "1"})])
def test_legacy_outputs_on_request(tmp_path, legacy, env):
    """The reference's "theory-checking" outputs: all_similar_histories_to_file (every comparison of every history,
    FE_problem.h:1237-1238) with SCEMA_B200_ALL_SIMILAR=1, and the legacy global nearest neighbour
    (get_most_similar_history_ID / _diff, lowest ID on ties) with either knob — byte-identical to the reference header."""
    ref = reference_run(f"legacy_{legacy}", tmp_path)
    ours = run_driver(build_ours(tmp_path), tmp_path / "ours", ["120", "12", "10", "1e-6", "4"], dict(env, DROPIN_LEGACY=legacy))
    assert ours["returncode"] == 0, ours["stderr"]
    assert same_run(ours, ref) and ours["stdout"].count("nearest of") >= 40
    if legacy == "1":
        full = [f for f in ours["files"] if f.endswith("all_similar_hist")]
        assert full and all(os.path.getsize(tmp_path / "ours" / f) > 1000 for f in full)


def test_error_behaviour_matches(tmp_path):
    """< 3 samples: both print the reference's message and exit(1) (strain2spline.h:142-148)."""
    ours_exe = build_ours(tmp_path)
    for n_steps in ("2", "0"):
        key = f"error_{n_steps}"
        ours = ours_run(ours_exe, key, tmp_path / ("ours" + n_steps))
        assert same_run(ours, reference_run(key, tmp_path), stderr=True)
        assert ours["returncode"] == 1 and "splinify" in ours["stderr"]
