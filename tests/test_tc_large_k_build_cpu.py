"""Build guard for the K' = 16 instantiations of the tensor kNN kernel (6 <= k <= 12): the no-spill guard of
test_build_no_spill_cpu.py covers every k_knn_tc instantiation it finds in the ptxas report, so these four must be in
that report -- with and without bias, long sweep (pre-filter) and short sweep -- or nothing guards them."""
import re

from test_build_no_spill_cpu import ptxas_report  # noqa: F401  (module-scoped fixture: one compile here)


def test_large_list_instantiations_are_reported(ptxas_report):  # noqa: F811
    found = {}
    for name, v in ptxas_report.items():
        m = re.search(r"k_knn_tcILb([01])ELb([01])ELb([01])ELi16ELi1EE", name)
        if m:
            found[tuple(int(x) for x in m.groups())] = v
    # (BIAS, DUMP, PRE): no score-dump variant
    assert set(found) == {(0, 0, 0), (1, 0, 0), (0, 0, 1), (1, 0, 1)}, sorted(ptxas_report)
    for key, v in found.items():
        assert v["stack"] == 0 and v["spill_st"] == 0 and v["spill_ld"] == 0 and v["regs"] == 168, (key, v)
