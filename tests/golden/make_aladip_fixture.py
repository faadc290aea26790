#!/usr/bin/env python
"""Parameter fixture of testsystems.AlanineDipeptideVacuum: the original project's own input files for that test system
(data/alanine-dipeptide-gbsa/alanine-dipeptide.{prmtop,crd}, read by testsystems.py:3375-3388; stored verbatim next to
this script) parsed by openmmtools_b200.amber and stored as plain numbers, so that the package needs no AMBER files at
run time.  Output: openmmtools_b200/data/alanine_dipeptide_vacuum.json"""
import json, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..', '..'))
from openmmtools_b200 import amber

SRC = os.path.join(HERE, 'alanine-dipeptide')


def build():
    d = amber.read_prmtop(SRC + '.prmtop')
    x = amber.read_inpcrd(SRC + '.crd')
    return dict(names=d['names'], mass=[float(v) for v in d['mass']], charge=[float(v) for v in d['charge']],
                sigma=[float(v) for v in d['sigma']], epsilon=[float(v) for v in d['epsilon']],
                bonds=[[int(b[0]), int(b[1]), float(b[2]), float(b[3]), bool(b[4])] for b in d['bonds']],
                angles=[[int(a[0]), int(a[1]), int(a[2]), float(a[3]), float(a[4])] for a in d['angles']],
                torsions=[[int(t[0]), int(t[1]), int(t[2]), int(t[3]), int(t[4]), float(t[5]), float(t[6])] for t in d['torsions']],
                exclusions=[[int(i), int(j)] for i, j in d['exclusions']],
                exceptions=[[int(e[0]), int(e[1]), float(e[2]), float(e[3]), float(e[4])] for e in d['exceptions']],
                positions=[[float(c) for c in r] for r in x])


if __name__ == '__main__':
    dst = os.path.join(HERE, '..', '..', 'openmmtools_b200', 'data', 'alanine_dipeptide_vacuum.json')
    json.dump(build(), open(dst, 'w'))
    print('wrote', os.path.abspath(dst), os.path.getsize(dst))
