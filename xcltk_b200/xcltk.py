"""Command-line dispatcher: the `xcltk <command> [options]` surface (xcltk/xcltk.py:40-53) for the
commands this package implements."""

import sys

from .config import APP, VERSION

_HELP = """
Program: {app} (Toolkit for XClone Preprocessing) -- B200 counting paths
Version: {version}

Usage:   {app} <command> [options]

Commands:
  -- RDR calculation
     basefc           Basic feature counting (GPU).

  -- BAF calculation
     pileup           SNP-level allele counting at candidate SNPs, or at sites discovered from the
                      reads when no -P is given (GPU): cellSNP.* output.
     (feature-level allele counting is a Python API: xcltk_b200.baf.fc.main.afc_wrapper;
      the `baf` pipeline around it -- genotyping, Eagle2 -- stays in the reference)

  -- Others
     -h, --help       Print this message and exit.
     -V, --version    Print version and exit.

"""

_ELSEWHERE = ("baf", "fixref", "convert")       # commands of the reference that are out of scope here


def _run_basefc(argv):
    from .rdr.fc.main import fc_main
    return fc_main(argv) or 0


def _run_pileup(argv):
    from .baf.pileup import pileup_main
    return pileup_main(argv) or 0


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    command = argv[1] if len(argv) > 1 else "--help"
    if command in ("-h", "--help"):
        sys.stdout.write(_HELP.format(app=APP, version=VERSION))
        sys.exit(0)
    if command in ("-V", "--version"):
        sys.stderr.write(VERSION + "\n")
        sys.exit(0)
    if command == "basefc":
        sys.exit(_run_basefc(argv))
    if command == "pileup":
        sys.exit(_run_pileup(argv))
    if command in _ELSEWHERE:
        sys.stderr.write("Error: command '%s' is outside the scope of xcltk_b200; use the reference.\n" % command)
    else:
        sys.stderr.write("Error: wrong command '%s'\n" % command)
    sys.exit(1)
