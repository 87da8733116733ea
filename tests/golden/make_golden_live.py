#!/usr/bin/env python3
"""Write tests/golden/golden_live.json: the reference C++'s result strings for the seeded inputs of
tests/test_oracle.py::live_cases(), so that test compares the oracle with the reference without the reference present.

Needs oracle/_ref/cpp_functions.so (`make -C oracle ref REF=<Porechop checkout>`).
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from helpers import abi_string, ref_lib  # noqa: E402
from test_oracle import live_cases  # noqa: E402


def main():
    lib = ref_lib()
    if lib is None:
        sys.exit('oracle/_ref/cpp_functions.so is not built')
    results = [abi_string(lib, rd, ad, sc) for rd, ad, sc in live_cases()]
    with open(os.path.join(HERE, 'golden_live.json'), 'w') as f:
        json.dump({'generator': 'tests/test_oracle.py::live_cases', 'results': results}, f, indent=0)
    print('live', len(results))


if __name__ == '__main__':
    main()
