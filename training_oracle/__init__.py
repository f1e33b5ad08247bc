"""CPU ORACLE for the reward / termination model's TRAINING row (test infrastructure, like oracle/).  It builds on
oracle/torch_oracle.py and oracle/fp16_oracle.py without changing them, so the oracle that the existing fixtures pin stays
the one they were recorded against."""
