"""The environment switches of the library are exactly the ones INTEGRATION.md documents.

* every `BTF_*` variable the package reads (getenv in the CUDA sources, os.environ in the Python) is in the switch
  table, and every name in the table is read somewhere: a switch cannot be retired in the code and left in the
  documents, or added without being documented;
* every `BTF_*` name that tests/ and tools/ use is in the table, so a test or a script cannot set a misspelt or
  retired switch and silently measure the default route.
"""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'functionalmf_b200')
NOT_SWITCHES = re.compile(r'BTF_(OK|E[A-Z]+|CFG\w*)$')     # return codes of the C ABI, tile-configuration macros
COMPILE_TIME = {'BTF_BAND_PROFILE'}                         # a -D flag of the instrumented band-kernel build


def _files(top, exts):
    for d, _, names in os.walk(top):
        for n in names:
            if n.endswith(exts):
                yield os.path.join(d, n)


def _documented():
    text = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    head = text.index('### Environment switches')
    table = text[head:text.index('\n\n', text.index('| Variable |', head))]
    rows = [line for line in table.splitlines() if line.startswith('| `')]
    names = set()
    for line in rows:
        names.update(re.findall(r'BTF_[A-Z0-9_]+', line.split('|')[1]))
    assert names, 'no switch table in INTEGRATION.md'
    return names


def _read_by_package():
    # the CUDA sources name a BTF_* string only to read it from the environment (read_env in engine.cu)
    names = set()
    for f in _files(PKG, ('.cu', '.cuh', '.h', '.cpp')):
        names.update(re.findall(r'"(BTF_[A-Z0-9_]+)"', open(f).read()))
    for f in _files(PKG, ('.py',)):
        names.update(re.findall(r'''os\.(?:environ(?:\.get)?|getenv)[\[(]\s*['"](BTF_[A-Z0-9_]+)''', open(f).read()))
    return names


def test_package_reads_exactly_the_documented_switches():
    documented, read = _documented(), _read_by_package()
    assert read - documented == set(), 'read but not in the INTEGRATION.md switch table'
    assert documented - read == set(), 'in the INTEGRATION.md switch table but read nowhere'


def test_cuda_switches_are_read_in_one_place():
    readers = sorted(os.path.basename(f) for f in _files(PKG, ('.cu', '.cuh', '.h', '.cpp'))
                     if re.search(r'"BTF_', open(f).read()))
    assert readers == ['engine.cu']


def test_tests_and_tools_name_only_documented_switches():
    documented = _documented()
    used = {}
    for top in ('tests', 'tools'):
        for f in _files(os.path.join(ROOT, top), ('.py', '.sh', '.md')):
            for nm in re.findall(r'BTF_[A-Z0-9_]+', open(f).read()):
                if not NOT_SWITCHES.match(nm) and nm not in COMPILE_TIME:
                    used.setdefault(nm, set()).add(os.path.relpath(f, ROOT))
    unknown = {nm: sorted(fs) for nm, fs in used.items() if nm not in documented}
    assert unknown == {}
