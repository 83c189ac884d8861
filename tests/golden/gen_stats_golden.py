"""Generate tests/golden/stats_golden.json: the reference's own get_df_stats (mlrun/data_types/infer.py:104-149) on the
frames of tests/stats_frames.py.

Requires /root/reference (read-only), imported in place with its missing third-party dependencies mocked
(tests/golden/_refshim.py).  Run:  python -m tests.golden.gen_stats_golden.  Nothing here is imported by the test-suite or
the product; the JSON it writes is data only."""

import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests import stats_frames
    from tests.golden import _refshim

    _refshim.install()
    import numpy as np
    import pandas as pd

    from mlrun.data_types.infer import get_df_stats

    out = {"pandas": pd.__version__, "numpy": np.__version__, "frames": []}
    for name, df, options in stats_frames.frames():
        spec = stats_frames.to_spec(df)
        again = stats_frames.from_spec(spec)
        pd.testing.assert_frame_equal(again, df, check_index_type=False)  # the JSON form round-trips
        out["frames"].append({"name": name, "options": options, "frame": spec, "stats": get_df_stats(df, options)})
    with open(os.path.join(HERE, "stats_golden.json"), "w") as fh:
        json.dump(out, fh, indent=None, separators=(",", ":"))
        fh.write("\n")
    print(f"{len(out['frames'])} frames")


if __name__ == "__main__":
    main()
