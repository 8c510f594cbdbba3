"""Generate tests/golden/reference_runs.json: what the reference's own programs print for the cases that
tests/test_dropin_header.py and tests/test_cli.py otherwise compare with live, where oracle/_ref is not built.

    python tests/golden/make_golden_live.py [SOURCE-NOTE]

  dropin: tests/helpers/dropin_driver.cc against the reference header (oracle/_ref/dropin_driver_ref), every case of
          test_dropin_header.CASES: exit code, SHA-256 of stdout, of stderr and of the set of result files;
  cli:    oracle/_ref/mpi_comparison_test and compare_all_histories on the directories test_cli.py writes, as line sets
          (SHA-256 of the sorted lines: another machine enumerates the directory in another order);
  oracle: the reference header behind oracle/_ref/libscema_ref.so on the randomized inputs of tests/test_oracle_vs_ref.py
          (SHA-256 of the bit patterns, 64 bits of it per history or file).

Where oracle/_ref is not built, this project's own drop-in header, command lines (needs a GPU) and CPU oracle are run
instead.
That is a faithful record only where they are known to print the reference's bytes for these cases; SOURCE-NOTE,
stored as "source", says why.
"""
import json
import os
import pathlib
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_cli  # noqa: E402
import test_dropin_header  # noqa: E402
import test_oracle_vs_ref  # noqa: E402
from oracle.pyoracle import Oracle, Reference  # noqa: E402


def main():
    live = os.path.exists(test_dropin_header.REF_BIN)
    out = {"source": "reference programs built by oracle/Makefile" if live else
           (sys.argv[1] if len(sys.argv) > 1 else "this project's drop-in header and command lines"),
           "dropin": {}, "cli": {}, "oracle": {}}
    with tempfile.TemporaryDirectory() as tmp:
        tmp = pathlib.Path(tmp)
        if live:
            for key, args, env in test_dropin_header.CASES:
                out["dropin"][key] = test_dropin_header.summary(test_dropin_header.run_driver(test_dropin_header.REF_BIN, tmp / key, args, env))
        else:
            exe = test_dropin_header.build_ours(tmp)
            for key, _, _ in test_dropin_header.CASES:
                out["dropin"][key] = test_dropin_header.summary(test_dropin_header.ours_run(exe, key, tmp / key))
        bin_dir = test_cli.REF if live else test_cli.BIN
        sdir = str(tmp / "strains") + "/"
        ids = test_cli.write_strain_dir(sdir)
        (tmp / "m" / "__results").mkdir(parents=True)
        r = subprocess.run([os.path.join(bin_dir, "mpi_comparison_test"), sdir, "10", repr(test_cli.THR)], cwd=tmp / "m",
                           capture_output=True, text=True, check=True)
        out["cli"]["mpi_comparison_test"] = test_cli.mpi_comparison_record(r.stdout, tmp / "m" / "__results", ids)
        sdir = str(tmp / "strains60") + "/"
        test_cli.write_strain_dir(sdir, n=60, seed=5)
        r = subprocess.run([os.path.join(bin_dir, "compare_all_histories"), sdir, "10"], cwd=tmp, capture_output=True,
                           text=True, check=True)
        out["cli"]["compare_all_histories"] = test_cli.compare_all_record(r.stdout)
        (tmp / "p").mkdir()
        lib = Reference() if live else Oracle()
        out["oracle"]["random"] = test_oracle_vs_ref.random_record(lib)
        make = test_oracle_vs_ref.reference_pipeline_record if live else test_oracle_vs_ref.oracle_pipeline_record
        out["oracle"]["pipeline"] = make(lib, str(tmp / "p"))
    with open(os.path.join(HERE, "reference_runs.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
