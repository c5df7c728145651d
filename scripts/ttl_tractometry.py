#!/usr/bin/env python3
"""Console entry point of the tractometry command (tracktolearn_b200/runners/ttl_tractometry.py)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tracktolearn_b200.runners.ttl_tractometry import main  # noqa: E402

if __name__ == '__main__':
    main()
