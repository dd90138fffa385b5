"""RMBR: minimum-Bayes-risk decoding of N-best lists with a BERTScore-recall utility on the device
(``utility_functions.BertScoreFunction``, ``mbr.find_best_length``).  The 1 - CER utility of the
same reference directory is ``cer_clients.CerScoreFunction``; ``cer_clients.mbr_decode`` takes either."""
