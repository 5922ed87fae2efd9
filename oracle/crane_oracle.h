/*
 * crane_oracle.h — C interface of the CPU oracle (TEST INFRASTRUCTURE ONLY).
 *
 * The oracle is a CPU restatement of the reference's scheduling hot path
 * (SchedulerAlgo::NodeSelect and callees). Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it. The product
 * path (cranesched_b200/) never links, imports or calls anything in oracle/.
 *
 * Parity status: UNPINNED by the reference (the reference ships no test of the
 * scheduler, SURVEY.md §4/§8c, and cannot be compiled here). The only
 * known-answer vectors the reference holds for this path —
 * test/Utilities/dedicated_resource_test.cpp:27-171 — are ported in
 * crane_oracle_selftest().
 */
#ifndef CRANE_ORACLE_H_
#define CRANE_ORACLE_H_

#include "../include/crane_sched.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Restates SchedulerAlgo::NodeSelect (JobScheduler.cpp:5543-5868). Writes the
 * same crane_placements_t the GPU path writes. elapsed_ms (optional) brackets
 * what the reference brackets as "NodeSelect costed {} ms"
 * (JobScheduler.cpp:1139-1147): everything after the job/node objects exist.
 * max_jobs > 0 stops the job loop after that many jobs of the priority order
 * (bounded CPU-baseline sample); the rest keep reason NONE/unset and
 * *jobs_done tells how many were processed. */
int crane_oracle_node_select(const crane_sched_config_t* cfg,
                             const crane_cluster_t* cluster, int64_t now,
                             const crane_running_t* running,
                             const crane_pending_t* pending,
                             crane_placements_t* out, double* elapsed_ms,
                             uint32_t max_jobs, uint32_t* jobs_done);

/* Reservations for the next crane_oracle_node_select calls (JobScheduler.cpp:5655-5713);
 * the pointer must stay valid; NULL = none. pending->reservation / running->reservation
 * refer to it. */
void crane_oracle_set_reservations(const crane_reservations_t* resv);

/* ResourceView::GetFeasibleResourceInNode (PublicHeader.cpp:519-599) on one
 * (request, availability) pair. Returns 1 feasible / 0 not; *alloc written when
 * feasible. */
int crane_oracle_feasible(const crane_cluster_t* dict,
                          const crane_res_view_t* req,
                          const crane_res_in_node_t* avail,
                          crane_res_in_node_t* alloc);

/* ResourceInNodeV3::Ckmin (PublicHeader.cpp:815-827): a = Ckmin(a, b). */
void crane_oracle_ckmin(const crane_cluster_t* dict, crane_res_in_node_t* a,
                        const crane_res_in_node_t* b);

/* operator<=(ResourceInNodeV3, ResourceInNodeV3) (PublicHeader.cpp:886-890). */
int crane_oracle_res_le(const crane_cluster_t* dict,
                        const crane_res_in_node_t* a,
                        const crane_res_in_node_t* b);

/* NodeState::UpdateResourceInNode (JobScheduler.h:334-453) on a timeline given
 * as parallel arrays (times ascending, last may be INT64_MAX sentinel).
 * In/out: *n_seg entries, capacity cap. Returns 0, or -1 if cap exceeded. */
int crane_oracle_timeline_update(const crane_cluster_t* dict, int64_t* times,
                                 crane_res_in_node_t* rows, uint32_t* n_seg,
                                 uint32_t cap, int64_t start, int64_t end,
                                 const crane_res_in_node_t* res);

/* EarliestStartSubsetSelector::CalcEarliestStartTime (JobScheduler.h:786-859)
 * for one job of node_num nodes and time_limit seconds over n_nodes timelines
 * (node k: times/rows[off[k] .. off[k+1]), ascending), asking alloc[k] of
 * node k. Returns 1 and writes *start, or 0 when no start lies within
 * max_window seconds of now. */
int crane_oracle_earliest_start(const crane_cluster_t* dict, uint32_t n_nodes,
                                uint32_t node_num, const uint32_t* off,
                                const int64_t* times,
                                const crane_res_in_node_t* rows,
                                const crane_res_in_node_t* alloc, int64_t now,
                                int64_t time_limit, int64_t max_window,
                                int64_t* start);

/* Restates the CheckAndMallocQosResource pass of the commit loop
 * (JobScheduler.cpp:1262; Accounting/AccountMetaContainer.cpp:164-191,
 * 382-531, 546-587) over the placements NodeSelect produced: job-id order,
 * jobs with reason NONE only; updates placements->reason and the usage tables
 * of `qos` in place. */
int crane_oracle_qos_filter(const crane_cluster_t* dict,
                            const crane_pending_t* pending,
                            crane_placements_t* placements,
                            const crane_qos_table_t* qos);

/* Ports test/Utilities/dedicated_resource_test.cpp:27-171 (14 cases) plus
 * hand-derived micro-cases. Returns the number of failed cases; fills `log`
 * (if non-NULL) with one line per failure. */
int crane_oracle_selftest(char* log, size_t log_cap);

#ifdef __cplusplus
}
#endif
#endif
