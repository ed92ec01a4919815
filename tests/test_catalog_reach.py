"""csrc/host/catalog_reach.hpp: the catalog's host-side rules, which inq_set_loci, inq_push_reads_routed and the CLI's
shard workers share -- the fetch predicate that routes reads to catalog shards, the running max of `end` the device join
reads, and the catalog checks with the error inq_set_loci reports. tests/catalog_reach_check.cpp compares all three
with brute force on seeded random catalogs, under AddressSanitizer and UndefinedBehaviorSanitizer."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_catalog_reach_equals_brute_force(tmp_path):
    exe = str(tmp_path / "catalog_reach_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-Wall", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", os.path.join(ROOT, "inquistr_b200", "csrc", "host"), "-o", exe,
                    os.path.join(ROOT, "tests", "catalog_reach_check.cpp")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    f = r.stdout.split()
    assert f[:2] == ["bad", "0"], r.stdout
    counts = dict(zip(f[0:10:2], map(int, f[1:10:2])))
    faults = list(map(int, f[11:]))
    # both answers of the predicate, slices that cut contigs, the top of the coordinate range, and each rule alone
    assert counts["reach"] > 0 and counts["miss"] > 0 and counts["cut"] > 0 and counts["top"] > 0, r.stdout
    assert faults[0] > 0 and faults[1] > 0 and faults[2] > 0 and faults[4] > 0, r.stdout
