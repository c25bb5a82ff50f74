/*
 * orb_oracle_kfdb.h -- C interface of the CPU oracle for KeyFrameDatabase (liborb_oracle_kfdb.so).
 *
 * TEST INFRASTRUCTURE ONLY, like orb_oracle.h: a literal restatement of ORB-SLAM2's KeyFrameDatabase.cc, which
 * SwarmMap carries (code/src/KeyFrameDatabase.cc: add, erase, clear, DetectLoopCandidates,
 * DetectRelocalizationCandidates), and of DBoW2's L1Scoring::score (Thirdparty/DBoW2/DBoW2/ScoringObject.cpp).
 * It is built as its own library so that the extractor / matcher oracle stays as it is.  The rules and the three
 * definitions that freeze what the reference leaves open are in orb_oracle_kfdb.cpp's header comment and in
 * DESIGN.md section 2.
 */
#ifndef ORB_ORACLE_KFDB_H
#define ORB_ORACLE_KFDB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* DBoW2 L1Scoring::score of two BowVectors (word ids strictly ascending). */
double orc_l1_score(int na, const uint32_t* aw, const double* av, int nb, const uint32_t* bw, const double* bv);

typedef struct orc_kfdb orc_kfdb;
/* n_words: the vocabulary size (mvInvertedFile.resize(mpVoc->size())). */
orc_kfdb* orc_kfdb_create(int n_words);
void orc_kfdb_destroy(orc_kfdb* db);
/* KeyFrameDatabase::add.  -1 when `id` is live already or a word id is out of range (nothing is added). */
int orc_kfdb_add(orc_kfdb* db, uint64_t id, int n, const uint32_t* words, const double* values);
/* KeyFrameDatabase::erase: an id that is not live is a no-op. */
void orc_kfdb_erase(orc_kfdb* db, uint64_t id);
void orc_kfdb_clear(orc_kfdb* db);
int orc_kfdb_size(const orc_kfdb* db);
/* The covisibility graph the queries read: GetBestCovisibilityKeyFrames(10) of keyframe ids[i] is
 * neigh[offsets[i] .. offsets[i+1]) in that order.  Ids without an entry have no neighbours.  Replaces the table. */
void orc_kfdb_set_neighbours(orc_kfdb* db, int n, const uint64_t* ids, const int32_t* offsets, const uint64_t* neigh);

/* One query.  mode 0: DetectRelocalizationCandidates; mode 1: DetectLoopCandidates(pKF, min_score) with
 * GetConnectedKeyFrames() = conn[0 .. n_conn).  Writes lScoreAndMatch (list order) to scored_ids / scored_scores
 * (*n_scored entries, at most scored_cap written) and the candidates to cand_ids (at most cand_cap written).
 * Returns the candidate count. */
int orc_kfdb_query(orc_kfdb* db, int mode, int n, const uint32_t* words, const double* values, float min_score,
                   int n_conn, const uint64_t* conn, uint64_t* scored_ids, float* scored_scores, int scored_cap,
                   int* n_scored, uint64_t* cand_ids, int cand_cap);
/* Host time of `iters` repetitions of queries 0 .. nq-1 (CSR q_off / q_words / q_values) in mode 0 or 1 (loop mode:
 * min_score per query, no connected keyframes), in seconds. */
double orc_kfdb_time_queries(orc_kfdb* db, int mode, int nq, const int32_t* q_off, const uint32_t* q_words,
                             const double* q_values, const float* min_score, int iters);

#ifdef __cplusplus
}
#endif
#endif /* ORB_ORACLE_KFDB_H */
