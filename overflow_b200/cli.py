"""Command line interface -- mirror of the reference's src/overflow_cli.py for the D8 path.

`flow-direction` keeps the reference's options, messages and exit codes (overflow_cli.py:54-84);
`breach-single-cell-pits` likewise (overflow_cli.py:18-51); `flow-accumulation`, `flow-routing` (both steps, one
pass over the device) and `basins` (drainage basins or watersheds of a flow-direction raster) are added with the same
conventions (the reference snapshot has no such commands).
"""
import click

from .basins import basins, read_pour_points
from .breach_single_cell_pits import breach_single_cell_pits
from .constants import DEFAULT_CHUNK_SIZE
from .flow_accumulation import flow_accumulation
from .flow_direction import flow_direction
from .flow_routing import flow_routing


@click.group()
def main():
    """The main entry point for the command line interface."""


@main.command(name="breach-single-cell-pits")
@click.option("--input_file", help="path to the DEM file")
@click.option("--output_file", help="path to the output file")
@click.option("--chunk_size", help="chunk size", default=DEFAULT_CHUNK_SIZE)
def breach_single_cell_pits_cli(input_file: str, output_file: str, chunk_size: int):
    """Breach single cell pits in a DEM (reference overflow_cli.py:18-51)."""
    try:
        breach_single_cell_pits(input_file, output_file, chunk_size)
    except Exception as exc:
        print(f"breach_single_cell_pits failed with the following exception: {str(exc)}")
        raise click.Abort()


@main.command(name="flow-direction")
@click.option("--input_file", help="path to the DEM file")
@click.option("--output_file", help="path to the output file")
@click.option("--chunk_size", help="chunk size", default=DEFAULT_CHUNK_SIZE)
def flow_direction_cli(input_file: str, output_file: str, chunk_size: int):
    """Generate a D8 flow direction raster from a DEM."""
    try:
        flow_direction(input_file, output_file, chunk_size)
    except Exception as exc:
        print(f"flow_direction failed with the following exception: {str(exc)}")
        # non-zero exit code on failure, like the reference
        raise click.Abort()


@main.command(name="flow-accumulation")
@click.option("--input_file", help="path to the flow direction raster")
@click.option("--output_file", help="path to the output file")
@click.option("--chunk_size", help="chunk size", default=DEFAULT_CHUNK_SIZE)
@click.option("--tile_size", default=0, help="rasters beyond device memory: accumulate in square tiles of this many "
              "cells a side (two passes over the file, the tiles' perimeter graph solved on the host); 0 = whole raster")
def flow_accumulation_cli(input_file: str, output_file: str, chunk_size: int, tile_size: int = 0):
    """Generate a flow accumulation raster from a D8 flow direction raster."""
    try:
        if tile_size and int(tile_size) > 0:
            from .tiles import flow_accumulation_file_tiled

            flow_accumulation_file_tiled(input_file, output_file, int(tile_size), int(tile_size))
        else:
            flow_accumulation(input_file, output_file, chunk_size)
    except Exception as exc:
        print(f"flow_accumulation failed with the following exception: {str(exc)}")
        raise click.Abort()


@main.command(name="flow-routing")
@click.option("--input_file", help="path to the DEM file")
@click.option("--flow_direction_file", help="path to the flow direction output file")
@click.option("--flow_accumulation_file", help="path to the flow accumulation output file")
@click.option("--chunk_size", help="chunk size", default=DEFAULT_CHUNK_SIZE)
def flow_routing_cli(input_file: str, flow_direction_file: str, flow_accumulation_file: str, chunk_size: int):
    """Generate D8 flow direction and flow accumulation rasters from a DEM in one pass."""
    try:
        flow_routing(input_file, flow_direction_file, flow_accumulation_file, chunk_size)
    except Exception as exc:
        print(f"flow_routing failed with the following exception: {str(exc)}")
        raise click.Abort()


@main.command(name="basins")
@click.option("--input_file", help="path to the flow direction raster")
@click.option("--output_file", help="path to the output file")
@click.option("--chunk_size", help="chunk size", default=DEFAULT_CHUNK_SIZE)
@click.option("--pour_points", default=None, help="text file with one row,col pour point per line: label watersheds "
              "of these points instead of the basins of every outlet")
def basins_cli(input_file: str, output_file: str, chunk_size: int, pour_points: str = None):
    """Label every cell of a D8 flow direction raster with the outlet (or pour point) it drains to."""
    try:
        basins(input_file, output_file, chunk_size, read_pour_points(pour_points) if pour_points else None)
    except Exception as exc:
        print(f"basins failed with the following exception: {str(exc)}")
        raise click.Abort()


if __name__ == "__main__":
    main()  # pylint: disable=no-value-for-parameter
