"""
Compiles the reference's Python package (dragonfly-opt 0.1.7) into oracle/_ref/dragonfly as sourceless bytecode,
for the tests that run the drop-in inside the reference's own classes and BO loop (tests/test_integration_*.py).
Called by __graft_entry__.build().  The reference source tree is $DRAGONFLY_SRC if set, else DEFAULT_SRC.  Where
neither holds a `dragonfly` package, nothing is built, an oracle/_ref/ built earlier is kept, and those tests skip.
oracle/_ref/ is a build product and stays out of git.
"""
import os
import py_compile
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '_ref')
DEFAULT_SRC = '/root/reference'


def source_tree():
  src = os.environ.get('DRAGONFLY_SRC') or DEFAULT_SRC
  return src if os.path.isdir(os.path.join(src, 'dragonfly')) else None


def build():
  """ Returns the package directory built, or None when the reference's sources are not there. """
  src = source_tree()
  if src is None:
    return None
  pkg_out = os.path.join(OUT, 'dragonfly')
  shutil.rmtree(pkg_out, ignore_errors=True)
  pkg_src = os.path.join(src, 'dragonfly')
  for dirpath, _, files in os.walk(pkg_src):
    rel = os.path.relpath(dirpath, pkg_src)
    for f in files:
      if f.endswith('.py'):
        name = os.path.normpath(os.path.join('dragonfly', rel, f))
        py_compile.compile(os.path.join(dirpath, f), cfile=os.path.join(OUT, name + 'c'), dfile=name, doraise=True)
  return pkg_out
