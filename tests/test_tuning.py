"""The SMM_* switches are read in one module, smm_tuning.cpp, and documented in smm_tuning.h (host
only, from the sources).

The planner, the plan cache key and the isolation lists of the variant tests all depend on which
switches shape a plan and which are read once per process.  These checks keep the four from
drifting apart: a plan switch left out of the cache key would let a cached file serve a plan built
under other settings, and a switch missing from the tests' lists would leak between tests.
"""
import os
import re

from test_gpu_variants import CREATE_ENV, PROCESS_ENV, ROOT

CSRC = os.path.join(ROOT, "smmregrid_b200", "csrc")


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _struct(name):
    m = re.search(r"struct %s \{(.*?)\n\};" % name, _read("smm_tuning.h"), re.S)
    assert m, name
    return m.group(1)


def _documented(name):
    """Switches a settings struct documents: `SMM_NAME:` or `SMM_NAME="..."` in its comments."""
    return set(re.findall(r"\b(SMM_[A-Z0-9_]+)(?=[:=])", _struct(name)))


def _plan_fields():
    """PlanSettings field -> the switch its preceding comment documents."""
    fields, switch = {}, None
    for line in _struct("PlanSettings").splitlines():
        line = line.strip()
        if line.startswith("//"):
            m = re.match(r"// (SMM_[A-Z0-9_]+)(?=[:=])", line)
            switch = m.group(1) if m else switch
        elif line.endswith(";"):
            assert switch, line
            for decl in line.rstrip(";").split(","):
                fields[decl.split("=")[0].split()[-1]] = switch
            switch = None
    return fields


def test_only_the_settings_module_reads_the_environment():
    readers = sorted(n for n in os.listdir(CSRC) if re.search(r"\bgetenv\b", _read(n)))
    assert readers == ["smm_tuning.cpp"]


def test_every_switch_read_is_documented():
    read = set(re.findall(r'"(SMM_[A-Z0-9_]+)"', _read("smm_tuning.cpp")))
    documented = _documented("PlanSettings") | _documented("LaunchSettings") | _documented("HostCallSettings")
    assert read == documented
    assert len(read) == 21


def test_cache_key_hashes_exactly_the_plan_shaping_switches():
    fields = _plan_fields()
    body = re.search(r"PlanCacheKey plan_cache_key\(.*?\n\}", _read("smm_plan_cache.cpp"), re.S).group(0)
    hashed = set(re.findall(r"hs\.pod\(s\.(\w+)\)", body))
    # every field but the thread count, which spreads the work and leaves the plan as it is
    assert hashed == set(fields) - {"plan_threads"}
    assert {fields[f] for f in hashed} == set(CREATE_ENV)


def test_process_switches_are_launch_settings():
    assert set(PROCESS_ENV) <= _documented("LaunchSettings")
