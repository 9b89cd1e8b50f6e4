"""The PG_* switch table (tests/switch_table.py) names every switch the package reads, and only those.  No GPU."""
import glob
import os
import re
import subprocess
import sys

import pytest

from conftest import ROOT
import switch_table as T

_READ = re.compile(r"""(?:getenv|environ\.get)\(\s*["'](PG_[A-Z0-9_]+)["']""")


def switches_read(root):
    """every PG_* name passed to getenv() / os.environ.get() in pangenome_b200/csrc/*.cu* and pangenome_b200/*.py"""
    found = {}
    files = glob.glob(os.path.join(root, "pangenome_b200", "csrc", "*.cu*")) + glob.glob(os.path.join(root, "pangenome_b200", "*.py"))
    for path in sorted(files):
        with open(path, encoding="utf-8") as f:
            for name in _READ.findall(f.read()):
                found.setdefault(name, []).append(os.path.relpath(path, root))
    return found


def test_table_names_every_switch():
    found = switches_read(ROOT)
    missing = sorted(set(found) - set(T.SWITCHES))
    stale = sorted(set(T.SWITCHES) - set(found))
    assert not missing, "switches read by the sources but missing from tests/switch_table.py: %s" % {n: found[n] for n in missing}
    assert not stale, "tests/switch_table.py names switches no source reads any more: %s" % stale


def test_every_switch_has_a_disposition():
    """each entry is run by a child profile (values, launches, replaces), run in-process, inert or not run - with a reason"""
    in_profiles = {k for _, env, _, _, _ in T.PROFILES for k in env}
    for name, e in T.SWITCHES.items():
        kinds = [x for x in ("launches", "inert", "not_run", "in_process") if x in e]
        assert len(kinds) == 1, (name, kinds)
        if "launches" in e:
            assert e["values"] and "replaces" in e, name
            assert name in in_profiles, "%s has no child profile" % name
        elif "inert" in e:
            assert e["values"] and name in in_profiles, "an inert switch is still run once, to show its kernel list equals the default's"
        else:
            assert name not in in_profiles and (e.get("not_run") or e.get("in_process")), name


def test_profile_values_are_tabled():
    """a profile sets only switches of the table, to values the table lists"""
    for pname, env, groups, must, must_not in T.PROFILES:
        assert set(groups) <= set(T.ALL_GROUPS), pname
        assert must, pname
        for k, v in env.items():
            assert k in T.SWITCHES and v in T.SWITCHES[k]["values"], (pname, k, v)
    assert len({p[0] for p in T.PROFILES}) == len(T.PROFILES)


@pytest.mark.parametrize("raw,norm", [
    ("void <unnamed>::k2a_partition_c<(int)256, (bool)0, (int)27, (int)3, (bool)0>(<unnamed>::CPartArgs)", "k2a_partition_c<256,false,27,3,false>"),
    ("void (anonymous namespace)::k2a_partition_c<256, true, 0, 3, false>((anonymous namespace)::CPartArgs)", "k2a_partition_c<256,true,0,3,false>"),
    ("<unnamed>::k1x_pack(const unsigned char *, long, long, const <unnamed>::TileEntry *, unsigned int *)", "k1x_pack"),
    ("(anonymous namespace)::k_table_clear(uint4*, long, long*)", "k_table_clear"),
    ("void <unnamed>::k3_insert_records<(int)8, (bool)1>(TableView, const uint4 *)", "k3_insert_records<8,true>"),
    ("void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<long>>(int)", None),
])
def test_kernel_names_normalise(raw, norm):
    assert T.norm_kernel(raw) == norm


def test_scan_catches_a_new_switch(tmp_path):
    """A copy of the sources with one more getenv("PG_...") fails the completeness check and names the switch."""
    pkg = tmp_path / "pangenome_b200"
    (pkg / "csrc").mkdir(parents=True)
    for path in glob.glob(os.path.join(ROOT, "pangenome_b200", "csrc", "*.cu*")) + glob.glob(os.path.join(ROOT, "pangenome_b200", "*.py")):
        rel = os.path.relpath(path, os.path.join(ROOT, "pangenome_b200"))
        with open(path, encoding="utf-8") as f:
            (pkg / rel).write_text(f.read())
    with open(pkg / "csrc" / "common.cu", "a") as f:
        f.write('\nstatic int pg_new_switch() { const char *e = getenv("PG_NEW"); return e ? atoi(e) : 0; }\n')
    found = switches_read(str(tmp_path))
    assert sorted(set(found) - set(T.SWITCHES)) == ["PG_NEW"]
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_switch_inventory as t, conftest; conftest.ROOT = t.ROOT = %r; "
            "t.test_table_names_every_switch()" % (os.path.join(ROOT, "tests"), ROOT, str(tmp_path)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "PG_NEW" in r.stderr, r.stderr[-2000:]
