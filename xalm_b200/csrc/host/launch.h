// launch.h — tensor-parallel ranks for xalm_main (`-g P`) without torch, MPI or a launcher: the process forks P workers,
// worker r drives CUDA device r as tensor-parallel rank r of P, and the parent only relays the two rendezvous messages
// (rank 0's NCCL id, then every rank's CUDA IPC handle), forwards stderr and reaps.
#pragma once
#include <functional>

#include "model.h"

// Where one worker sits in the group.  The default is the one-GPU model.cuda(): device 0, rank 0 of 1, no communicator.
struct TpRank {
	int device = 0, rank = 0, size = 1;
	const void* comm_id = nullptr; // XALM_COMM_ID_BYTES from rank 0 (size > 1)
	IpcExchange ipc_exchange;      // size > 1: this rank's IPC handle in, every rank's out (rank order)
};

// Runs fn on P worker processes and returns the exit code for main: 0 when every worker returned 0, else 1.
//   * The calling process (the supervisor) makes no CUDA or NCCL call, before or after the fork: a child forked after cuInit
//     cannot use CUDA, and the threads NCCL starts do not survive fork.
//   * Each worker first checks that the box has P visible devices, then takes part in the id exchange, then runs fn.
//   * Only rank 0 writes stdout (the others' goes to /dev/null); every rank's stderr comes out line by line as "rank r: ...".
//   * When one worker fails (non-zero exit or a signal) the others are killed, since they may be blocked in a collective that
//     will never complete; a worker dies with the supervisor (PR_SET_PDEATHSIG).  No worker outlives the call.
int run_tp_ranks(int P, const std::function<int(const TpRank&)>& fn);
