"""Generate ``reference_run__*.npz``: outputs of the REFERENCE'S OWN ``estimators.py`` / ``reductor.py`` /
``online_enrichment.py`` (loaded unmodified from ``$LRBMS_REFERENCE_DIR``, see ``oracle/reference_run.py``) on the seeded
inputs of ``make_golden.py``.

    LRBMS_REFERENCE_DIR=<pylrbms checkout>/python/dune/pylrbms python tests/golden/make_reference_golden.py

The reference's third-party layers (pyMOR fork, dune-gdt, mpi4py) are not installable; they are replaced by the NumPy
stand-ins named in ``oracle/reference_run.py``.  So these vectors pin the arithmetic that lives in the reference's own
files -- estimator, image bases and reduced flux / Oswald operators, Doerfler marking, the enrichment loop -- and the tests
compare both the oracle (CPU, ``tests/test_oracle_golden.py``) and the CUDA path (``tests/test_gpu_golden.py``) with them.
The sha256 of each reference source file that was executed is stored alongside.
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
import make_golden  # noqa: E402

ENRICHMENT_CASES = {
    # name: (case, mu, enrichment steps, Doerfler theta, max age)
    'os2015_2x2_N5': (0.4, 2, 0.5, 2),
    'os2015_3x2_ragged': (0.7, 1, 0.33, 1),   # (a second step at the same mu re-marks a subdomain whose corrector is already in
                                              #  the basis: ExtensionError, which the reference does not catch)
}


def reference_file_digests():
    from oracle.reference_run import REFERENCE_DIR
    out = {}
    for name in ('estimators', 'reductor', 'online_enrichment'):
        with open(os.path.join(REFERENCE_DIR, name + '.py'), 'rb') as f:
            out['reference_sha256__' + name] = np.array(hashlib.sha256(f.read()).hexdigest())
    return out


def generate(name):
    from oracle.reference_run import reference_enrichment, reference_outputs
    data, bases = make_golden.build_case(name)
    out = reference_outputs(data, bases, make_golden.MUS)
    if name.startswith('synthetic3d'):
        out = {k: v for k, v in out.items() if not k.startswith('basis__')}     # keeps the file small
    if name in ENRICHMENT_CASES:
        mu, steps, theta, max_age = ENRICHMENT_CASES[name]
        enr = reference_enrichment(data, bases, mu, steps, theta=theta, max_age=max_age)
        out.update({'enrichment__' + k: v for k, v in enr.items()})
        out['enrichment__args'] = np.array([mu, steps, theta, max_age], dtype=float)
    out['input_sha256'] = np.array(make_golden.input_digest(data, bases))
    out.update(reference_file_digests())
    return out


SEQUENCE_CASES = {
    # name: (subdomains, cells, SPE10-like field seed, contrast, parameters): a field without symmetries -- on the symmetric
    # OS2015 example mirror-image subdomains have equal indicators and the marking hangs on the last bit of the estimator
    'enrichment_spe10like_2x2': ((2, 2), 4, 7, 50.0, (0.4, 0.9, 0.15)),
    'enrichment_spe10like_3x3': ((3, 3), 4, 7, 50.0, (0.4, 0.9, 0.15)),
}


def build_sequence_case(name):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, spe10_like_problem
    subdomains, cells, seed, contrast, mus = SEQUENCE_CASES[name]
    return assemble_block_swipdg(subdomains, cells, problem=spe10_like_problem(seed=seed, contrast=contrast)), mus


def generate_sequence(name):
    from oracle.reference_run import reference_enrichment_sequence
    data, mus = build_sequence_case(name)
    out = reference_enrichment_sequence(data, mus)
    out.update(reference_file_digests())
    return out


def main():
    for name in SEQUENCE_CASES:
        out = generate_sequence(name)
        path = os.path.join(HERE, 'reference_run__' + name + '.npz')
        np.savez_compressed(path, **out)
        print(name, '->', path, os.path.getsize(path), 'bytes', out['eta'], out['rb_size'])
    for name in make_golden.CASES:
        out = generate(name)
        path = os.path.join(HERE, 'reference_run__' + name + '.npz')
        np.savez_compressed(path, **out)
        print(name, '->', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
