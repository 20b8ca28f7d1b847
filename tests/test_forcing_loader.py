"""CPU: forcing loader formats (SURVEY 8f N3)."""
import numpy as np

import lgar_b200
from lgar_b200 import forcing


def test_three_formats(tmp_path):
    a = tmp_path / "a.csv"
    a.write_text("Time,P(mm/h),PET(mm/h)\n2016-10-01 00:00:00,0.0,0.0\n2016-10-01 01:00:00,12.5,0.25\n")
    b = tmp_path / "b.txt"
    b.write_text("#Time,P(mm/h),PET(mm/h)\n2016-10-01 00:00:00,0.0,0.0\n2016-10-01 00:05:00,20.0,0.0\n")
    c = tmp_path / "c.txt"
    c.write_text("Time P(mm/h) PET(mm/h)\n2016-10-01 00:00:00 0.0 0.0\n2016-10-01 00:05:00 50.0 0.5\n")
    np.testing.assert_allclose(forcing.read_forcing(str(a)), [[0, 0], [1.25, 0.025]])
    np.testing.assert_allclose(forcing.read_forcing(str(b)), [[0, 0], [2.0, 0.0]])
    np.testing.assert_allclose(forcing.read_forcing(str(c)), [[0, 0], [5.0, 0.05]])
    s = forcing.stack_sites([forcing.read_forcing(str(a)), forcing.read_forcing(str(b))], pin=False)
    assert tuple(s.shape) == (2, 2, 2)
