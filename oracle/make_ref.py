#!/usr/bin/env python
"""Package the UNMODIFIED reference (dfm/emcee, pure Python) for the CPU arm of bench.py.

    python -m oracle.make_ref        # also run by __graft_entry__.build()

Writes ``oracle/_ref/emcee_reference.zip`` (git-ignored): the ``.py`` files of the reference's
``src/emcee`` byte for byte (the same checkout ``oracle/gen_golden.py`` reads), plus the one-line
``emcee/emcee_version.py`` that setuptools_scm would generate at install time
(``src/emcee/__init__.py:22`` imports it; ``setup.py:59-64``).  ``bench.py`` puts the archive on
``sys.path`` (zipimport) and drives the reference's own ``EnsembleSampler`` -- nothing of this
repository is on that path.  Copying the package directory is what ``pip install`` would do; the
reference's build backend needs setuptools_scm.

Where the reference checkout cannot be read, an archive already there is kept and nothing else
happens: the CPU arm of bench.py then times the numpy port and says so in its output.
"""
import os
import sys
import zipfile

from oracle.gen_golden import REF_SRC

REF = os.path.join(REF_SRC, "emcee")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "emcee_reference.zip")


def main():
    if not os.path.isdir(REF):
        print("make_ref: %s not readable -- %s" % (REF, "keeping " + OUT if os.path.exists(OUT) else "no archive"))
        return 0
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    tmp = OUT + ".tmp"
    n = 0
    with zipfile.ZipFile(tmp, "w", zipfile.ZIP_DEFLATED) as z:
        for root, dirs, files in os.walk(REF):
            dirs.sort()
            for f in sorted(files):
                if not f.endswith(".py"):
                    continue
                full = os.path.join(root, f)
                z.write(full, os.path.join("emcee", os.path.relpath(full, REF)))
                n += 1
        z.writestr("emcee/emcee_version.py", '__version__ = "3.1.6+reference.8ab6c0f"\n')
    os.replace(tmp, OUT)
    print("make_ref: %d files -> %s" % (n + 1, OUT))
    return 0


if __name__ == "__main__":
    sys.exit(main())
