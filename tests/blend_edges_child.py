"""Computes the outputs of one blend configuration for test_blend_edges_gpu.py in a fresh process (the library reads
B200GS_BLEND_WIDE and B200GS_BLEND_CTAS once per process) and writes them to the .npz named on the command line.
--sessions adds the persistent-session sequence."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402

import test_blend_edges_gpu as t  # noqa: E402

if __name__ == "__main__":
    np.savez(sys.argv[1], **t.config_outputs(sessions="--sessions" in sys.argv[2:]))
