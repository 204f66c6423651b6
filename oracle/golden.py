"""Size limits of the stored fixtures under tests/golden/ (each file stays below 1 MB).

Both generators (oracle/gen_golden.py, oracle/gen_golden_step.py) pass what they recorded through these functions, so a
regenerated fixture has the same layout as the committed one.  The samples are fixed (no random draw): a test that
reads a fixture compares exactly the entries it holds.
"""


def sample_grads(grads, every):
    """Every scalar entry (the `.v` gradients, the `#norm` entries), and every `every`-th of the other entries in sorted
    key order."""
    out, i = {}, 0
    for k in sorted(grads):
        g = grads[k]
        if g.numel() == 1:
            out[k] = g
        else:
            if i % every == 0:
                out[k] = g
            i += 1
    return out


def sample_rows(m, row_stride):
    """Every `row_stride`-th row of a matrix, with the stride the test needs to pick the same rows."""
    return dict(row_stride=row_stride, rows=m[::row_stride].contiguous())
