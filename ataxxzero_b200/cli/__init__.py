"""Command-line twins of the reference's entry points (same flags, same file formats):

    python -m ataxxzero_b200.cli.accelerated_generate_games   (accelerated_generate_games.py)
    python -m ataxxzero_b200.cli.generate_games               (generate_games.py)
    python -m ataxxzero_b200.cli.looper                       (looper.py)
    python -m ataxxzero_b200.cli.perft                        (perft.py)
    python -m ataxxzero_b200.cli.uai_interface                (uai_interface.py)

and one the reference does not have:

    python -m ataxxzero_b200.cli.arena                        (two networks matched on the GPU)
"""
