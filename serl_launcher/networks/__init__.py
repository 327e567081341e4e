"""reference networks/ -> serl_b200.networks."""
