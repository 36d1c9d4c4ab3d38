"""Synthetic heavy-tailed-coverage mismatch matrices (SURVEY.md 8d, BASELINE.json configs 2-5).

Host-side numpy generator used by bench.py and the tests. It produces the SoA columns that
`mdg_counts_reduce` consumes (rows grouped by TaxID, 2*P rows per TaxID: z = +1..+P then
-1..-P) with damage injected in the C->T (forward) / G->A (reverse) substitutions:

    N_alignments = floor(10 * Pareto(alpha=1.1)) clipped to [10, 6e7]          (heavy tail)
    per row and reference base r:  N_r ~ Binomial(N_alignments, 0.2), floor 1
    30 % "ancient": A~U(0.05,0.5), q~U(0.2,0.7);  70 % "modern": A~U(0,0.01);  c~U(0.002,0.03)
    phi = 2 + Exp(mean 1000);   D(z) = A (1-q)^(|z|-1) + c
    k(z) ~ BetaBinomial(N_ref(z), D phi, (1-D) phi)   in CT (forward rows) / GA (reverse rows)
    every other mismatch ~ Binomial(N_r, 0.003); the diagonal takes the rest.

TaxIDs that fail the cuts (min_alignments, min_y_sum) stay in the input so the counts kernel's
cut + compaction path is exercised; `n_fit` asks for exactly that many TaxIDs to survive.
"""
import numpy as np

SEEDS = {"cfg2": 20240001, "cfg3": 20240002, "cfg4": 20240003, "cfg5": 20240004}


def _draw_taxa(rng, n_tax, P):
    n_al = np.floor(10.0 * (1.0 + rng.pareto(1.1, n_tax)))
    n_al = np.clip(n_al, 10, 6e7).astype(np.int64)
    ancient = rng.random(n_tax) < 0.3
    A = np.where(ancient, rng.uniform(0.05, 0.5, n_tax), rng.uniform(0.0, 0.01, n_tax))
    q = rng.uniform(0.2, 0.7, n_tax)
    c = rng.uniform(0.002, 0.03, n_tax)
    phi = 2.0 + rng.exponential(1000.0, n_tax)
    return n_al, A, q, c, phi


def make_mismatch_matrix(n_tax, max_position=15, seed=SEEDS["cfg2"], n_fit=None, min_alignments=10,
                         min_y_sum=10, fwd="CT", rev="GA", tax_id_start=1, jump=0):
    """Returns a dict with the SoA input columns, the dense k/N truth and the generator's
    parameters. If `n_fit` is given, `n_tax` is ignored and TaxIDs are generated until exactly
    `n_fit` of them pass the cuts (the failing ones stay in the input). `jump` selects the jump-th
    2^128-draw block of the seed's Philox stream: the shares of one seeded data set (BASELINE config 3:
    seed 20240002 partitioned by TaxID range over the GPUs) are generated independently, rank r with
    jump = r, without any rank generating the others' TaxIDs."""
    P = int(max_position)
    bitgen = np.random.Philox(seed)
    rng = np.random.Generator(bitgen.jumped(int(jump)) if jump else bitgen)
    bases = "ACGT"
    fr, fo = bases.index(fwd[0]), bases.index(fwd[1])
    rr, ro = bases.index(rev[0]), bases.index(rev[1])
    # damage is always injected in CT (forward rows) / GA (reverse rows): a control run that
    # looks at other substitutions must see no signal (BASELINE.json config 4)
    dmg = {False: (1, 3), True: (2, 0)}

    def generate(m):
        n_al, A, q, c, phi = _draw_taxa(rng, m, P)
        R = 2 * P
        rows = m * R
        pos0 = np.tile(np.concatenate([np.arange(P), np.arange(P)]), m).astype(np.uint8)
        is_rev = np.tile(np.concatenate([np.zeros(P, np.uint8), np.ones(P, np.uint8)]), m)
        n_al_row = np.repeat(n_al, R)
        counts = np.zeros((16, rows), dtype=np.int64)
        x = pos0.astype(np.float64)
        Dz = np.repeat(A, R) * (1.0 - np.repeat(q, R)) ** x + np.repeat(c, R)
        Dz = np.clip(Dz, 1e-6, 1 - 1e-6)
        phi_row = np.repeat(phi, R)
        for r in range(4):
            n_r = np.maximum(rng.binomial(n_al_row, 0.2), 1)
            off = 0
            for o in range(4):
                if o == r:
                    continue
                cnt = rng.binomial(n_r, 0.003)
                for strand_rev in (False, True):
                    if (r, o) == dmg[strand_rev]:
                        sel = is_rev == (1 if strand_rev else 0)
                        p = rng.beta(Dz[sel] * phi_row[sel], (1.0 - Dz[sel]) * phi_row[sel])
                        cnt[sel] = rng.binomial(n_r[sel], p)
                counts[r * 4 + o] = cnt
                off = off + cnt
            # diagonal takes the rest; if the three mismatches overshoot, grow the reference total
            counts[r * 4 + r] = np.maximum(n_r - off, 0)
        return dict(n_al=n_al, A=A, q=q, c=c, phi=phi, pos0=pos0, is_rev=is_rev, n_al_row=n_al_row, counts=counts)

    def passing(g):
        R = 2 * P
        kf = g["counts"][fr * 4 + fo].reshape(-1, R)[:, :P].sum(1)
        kr = g["counts"][rr * 4 + ro].reshape(-1, R)[:, P:].sum(1)
        return (g["n_al"] >= min_alignments) & (kf + kr >= min_y_sum)

    if n_fit is None:
        g = generate(int(n_tax))
        ok = passing(g)
    else:
        parts, oks, have = [], [], 0
        batch = max(1024, int(n_fit * 2))
        while have < n_fit:
            gp = generate(batch)
            okp = passing(gp)
            parts.append(gp)
            oks.append(okp)
            have += int(okp.sum())
        ok = np.concatenate(oks)
        cut = int(np.nonzero(np.cumsum(ok) == n_fit)[0][0]) + 1  # first index where n_fit have passed
        R = 2 * P
        g = {}
        for key in parts[0]:
            if key == "counts":
                g[key] = np.concatenate([p_[key] for p_ in parts], axis=1)[:, : cut * R]
            elif key in ("pos0", "is_rev", "n_al_row"):
                g[key] = np.concatenate([p_[key] for p_ in parts])[: cut * R]
            else:
                g[key] = np.concatenate([p_[key] for p_ in parts])[:cut]
        ok = ok[:cut]

    m = len(g["n_al"])
    R = 2 * P
    tax_id = np.arange(tax_id_start, tax_id_start + m, dtype=np.int64)
    counts16 = np.ascontiguousarray(g["counts"].astype(np.uint32))
    nf = counts16[fr * 4: fr * 4 + 4].sum(0, dtype=np.uint64)
    nr = counts16[rr * 4: rr * 4 + 4].sum(0, dtype=np.uint64)
    kf = counts16[fr * 4 + fo]
    kr = counts16[rr * 4 + ro]
    rev_mask = g["is_rev"].astype(bool)
    k_dense = np.where(rev_mask, kr, kf).reshape(m, R).astype(np.uint32)
    N_dense = np.where(rev_mask, nr, nf).reshape(m, R).astype(np.uint32)
    return dict(
        tax_id=np.repeat(tax_id, R), n_alignments=g["n_al_row"].astype(np.uint32),
        is_reverse=g["is_rev"], pos0=g["pos0"], counts16=counts16,
        tax_ids=tax_id, tax_n_alignments=g["n_al"].astype(np.uint32), passes=ok,
        k=k_dense, N=N_dense, truth=dict(A=g["A"], q=g["q"], c=g["c"], phi=g["phi"]),
        max_position=P,
    )


def write_tsv(g, path, legacy=False, tax_name="synthetic taxon", tax_rank="species"):
    """Write the SoA columns of `make_mismatch_matrix` as the mismatch-matrix text file the reference parses
    (counts.py:37-45, 229-235: 22 tab-separated columns, no header; `legacy`: the 20-column layout with a header
    that data/input/*.txt use). pyarrow's multi-threaded CSV writer: ~1 s per million rows."""
    import pyarrow as pa
    import pyarrow.csv as pacsv

    n = len(g["tax_id"])
    cols = {"tax_id": pa.array(g["tax_id"])}
    if not legacy:
        cols["tax_name"] = pa.repeat(tax_name, n)
        cols["tax_rank"] = pa.repeat(tax_rank, n)
    cols["N_alignments"] = pa.array(g["n_alignments"])
    cols["strand"] = pa.array(np.where(g["is_reverse"] == 1, "3'", "5'"))
    cols["position"] = pa.array(g["pos0"])
    for i, r in enumerate("ACGT"):
        for j, o in enumerate("ACGT"):
            cols[r + o] = pa.array(g["counts16"][4 * i + j])
    with open(path, "wb") as fh:
        if legacy:
            fh.write(("\t".join(["#taxid", "Nalignments", "Direction", "Pos"] + list(cols)[4:]) + "\n").encode())
        pacsv.write_csv(pa.table(cols), fh, write_options=pacsv.WriteOptions(include_header=False, delimiter="\t", quoting_style="none"))
    return path


def dense_fit_batch(n_fit, max_position=15, seed=SEEDS["cfg2"], **kw):
    """Dense (tax_id, k, N) of exactly `n_fit` TaxIDs that pass the cuts, in input order."""
    g = make_mismatch_matrix(0, max_position=max_position, seed=seed, n_fit=n_fit, **kw)
    sel = g["passes"]
    return g["tax_ids"][sel], np.ascontiguousarray(g["k"][sel]), np.ascontiguousarray(g["N"][sel]), g


def dense_fit_batch_shares(n_fit, parts, max_position=15, seed=SEEDS["cfg3"]):
    """Dense (tax_id, k, N) of `n_fit` passing TaxIDs generated as `parts` independent shares (share r = jumped block r,
    tax ids from 1 + r * 10^8), the way bench.py's multi-GPU workload cuts config 3; no share is held twice in memory."""
    tid, k, N = [], [], []
    for r in range(parts):
        g = make_mismatch_matrix(0, max_position=max_position, seed=seed, n_fit=n_fit // parts + (r < n_fit % parts), jump=r,
                                 tax_id_start=1 + r * 100_000_000)
        sel = g["passes"]
        tid.append(g["tax_ids"][sel])
        k.append(g["k"][sel])
        N.append(g["N"][sel])
    return np.concatenate(tid), np.ascontiguousarray(np.vstack(k)), np.ascontiguousarray(np.vstack(N))


def mism12_from_counts16(counts16, first_rows, max_position):
    """[n_tax][2P][12] off-diagonal raw counts (AC..TG) of complete 2P-row TaxIDs, for the noise estimate."""
    R = 2 * int(max_position)
    off = [r * 4 + o for r in range(4) for o in range(4) if r != o]
    idx = (np.asarray(first_rows)[:, None] + np.arange(R)[None, :]).ravel()
    return np.ascontiguousarray(counts16[off][:, idx].T.reshape(len(first_rows), R, 12))
