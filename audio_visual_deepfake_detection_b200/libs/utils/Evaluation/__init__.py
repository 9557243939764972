from .eval_proposal import ANETproposal, average_recall_vs_avg_nr_proposals

__all__ = ["ANETproposal", "average_recall_vs_avg_nr_proposals"]
