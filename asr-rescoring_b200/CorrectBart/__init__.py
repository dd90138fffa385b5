"""CorrectBart (one_hyp): a BART model reads the 1-best hypothesis of every utterance and generates a
corrected sentence greedily on the device (``model.CorrectBart``); ``model.compute_cer`` takes the corpus
CER of the outputs through the Levenshtein kernel.  DESIGN.md §3.11."""
