"""Drop-in for the reference's src/overflow_cli.py (D8 commands and single-cell pit breaching)."""
from overflow_b200.cli import (  # noqa: F401
    basins_cli,
    breach_single_cell_pits_cli,
    flow_accumulation_cli,
    flow_direction_cli,
    flow_routing_cli,
    main,
)

if __name__ == "__main__":
    main()  # pylint: disable=no-value-for-parameter
