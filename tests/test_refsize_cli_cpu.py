"""CPU: the command line's -refsize range (1..4096: the narrow search up to 384, the wide-refsize search above)."""
import pytest


@pytest.mark.parametrize("tool,head", [("newref", ["a.npz", "out.npz"]), ("newrefpart", ["p.npz", "part", "1", "3"]),
                                       ("newrefrank", ["p.npz", "out.npz"])])
def test_refsize_range(tool, head):
    import wisecondor
    p = wisecondor.buildParser()
    for k in (1, 384, 385, 4096):
        assert p.parse_args([tool] + head + ["-refsize", str(k)]).refsize == k
    for k in (0, 4097):
        with pytest.raises(SystemExit):
            p.parse_args([tool] + head + ["-refsize", str(k)])


def test_refsize_help_states_the_range():
    import wisecondor
    assert "1..4096" in wisecondor.buildParser()._subparsers._group_actions[0].choices["newref"].format_help()
