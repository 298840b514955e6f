"""Seeded synthetic weights / inputs -- re-exported from the product's generator (tha4_b200/synthetic.py) so that the
oracle-side tests and the CUDA path are guaranteed to see the very same tensors.  TEST INFRASTRUCTURE."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tha4_b200.synthetic import (make_state_dict, random_poses, student_state_dicts, synthetic_image,  # noqa: E402,F401
                                 teacher_state_dicts)
from tha4_b200.nn.state_dict_spec import Spec, STUDENT_SPECS, TEACHER_SPECS  # noqa: E402,F401

# CPU threads the golden fixtures are recorded and checked with: the thread count decides how the CPU convolutions split
# their sums, which moves the outputs by ~1e-5
FIXTURE_THREADS = 8
