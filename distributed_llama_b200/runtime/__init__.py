from .engine import Engine, ScoreResult
