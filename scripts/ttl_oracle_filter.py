#!/usr/bin/env python3
"""Console entry point of the tractogram filter (tracktolearn_b200/runners/ttl_oracle_filter.py)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tracktolearn_b200.runners.ttl_oracle_filter import main  # noqa: E402

if __name__ == '__main__':
    main()
