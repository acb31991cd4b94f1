"""Installs the unmodified reference package (google/uis-rnn, pure Python: nothing to compile) under oracle/_ref/,
where `bench.py --impl reference` and the `cpu_baseline` leg of `bench.py` import it from.  oracle/_ref/ is
git-ignored; without a reference checkout nothing is installed and those legs run the numpy port
(oracle/uis_oracle.py) instead.

The checkout is taken from $UISRNN_REFERENCE, else from a directory `reference` next to this repository.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, '_ref')
SOURCE = os.path.abspath(os.environ.get('UISRNN_REFERENCE') or
                         os.path.join(os.path.dirname(os.path.dirname(HERE)), 'reference'))


def installed():
  return os.path.exists(os.path.join(DST, 'uisrnn', 'uisrnn.py'))


def install():
  """Copies SOURCE/uisrnn to oracle/_ref/uisrnn unless it is there already or SOURCE holds no reference."""
  pkg = os.path.join(SOURCE, 'uisrnn')
  if installed() or not os.path.isfile(os.path.join(pkg, 'uisrnn.py')):
    return
  tmp = os.path.join(DST, 'uisrnn.tmp.%d' % os.getpid())   # renamed into place whole: no half-copied package
  try:
    os.makedirs(DST, exist_ok=True)
    shutil.copytree(pkg, tmp, ignore=shutil.ignore_patterns('__pycache__', '*.pyc'))
    os.replace(tmp, os.path.join(DST, 'uisrnn'))
  except OSError as err:   # the reference legs then run the numpy port; the product build is unaffected
    sys.stderr.write('oracle/_ref install failed: %s\n' % err)
  finally:
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
  install()
  print(DST if installed() else 'no reference found at %s' % SOURCE)
