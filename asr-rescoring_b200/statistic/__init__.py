"""statistic: error analysis of the reference's ``statistic/`` directory (U/S/I/D counts)."""
