// launch.cpp — the `-g P` supervisor and its workers (launch.h).
//
// Rendezvous, the same two steps tp.broadcast_comm_id / tp.make_ipc_exchange take through torch.distributed on the Python side,
// over one SOCK_SEQPACKET socketpair per worker (message boundaries are kept, so every recv is one whole message):
//   1. worker 0 sends its XALM_COMM_ID_BYTES NCCL id; the supervisor sends it on to every worker;
//   2. inside model.cuda() every worker sends its XALM_IPC_HANDLE_BYTES handle; once all P have arrived the supervisor sends the
//      rank-ordered table to every worker.
// The workers inherit the environment (XALM_NO_PREFILL, the XALM_<knob> tuning overrides, ...), so it is the same on every rank.
#include "launch.h"

#include <fcntl.h>
#include <poll.h>
#include <signal.h>
#include <sys/prctl.h>
#include <sys/socket.h>
#include <sys/wait.h>
#include <unistd.h>

#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {

bool send_msg(int fd, const void* p, size_t n) { return send(fd, p, n, MSG_NOSIGNAL) == (ssize_t) n; }

// One whole message of exactly n bytes (anything else, or the peer gone, is a failure).
bool recv_msg(int fd, void* p, size_t n) {
	ssize_t r;
	do r = recv(fd, p, n, MSG_TRUNC); while (r < 0 && errno == EINTR);
	return r == (ssize_t) n;
}

[[noreturn]] void worker(int r, int P, int sock, const std::function<int(const TpRank&)>& fn) {
	// Checked before any CUDA call: a worker on a box with fewer devices fails at once instead of waiting for peers.
	int n = 0;
	std::string why;
	if (xalm_cuda_device_count(&n) != XALM_OK) {
		n = 0;
		why = std::string(" (") + xalm_cuda_last_error() + ")";
	}
	if (n < P) {
		fprintf(stderr, "error: -g %d needs %d visible CUDA devices, %d found%s\n", P, P, n, why.c_str());
		exit(1);
	}
	unsigned char comm_id[XALM_COMM_ID_BYTES];
	if (r == 0) {
		if (xalm_cuda_comm_unique_id(comm_id) != XALM_OK) {
			fprintf(stderr, "error: NCCL id: %s\n", xalm_cuda_last_error());
			exit(1);
		}
		if (!send_msg(sock, comm_id, sizeof comm_id)) exit(1);
	}
	if (!recv_msg(sock, comm_id, sizeof comm_id)) exit(1); // the supervisor is gone or another rank failed
	TpRank tp;
	tp.device = r;
	tp.rank = r;
	tp.size = P;
	tp.comm_id = comm_id;
	tp.ipc_exchange = [sock, P](const std::vector<uint8_t>& mine) {
		std::vector<uint8_t> table((size_t) P * XALM_IPC_HANDLE_BYTES);
		if (!send_msg(sock, mine.data(), mine.size()) || !recv_msg(sock, table.data(), table.size()))
			throw std::runtime_error("model.cuda(): IPC handle exchange with the other ranks failed");
		return table;
	};
	exit(fn(tp)); // exit, not _exit: stdout is flushed as on one GPU
}

struct Worker {
	pid_t pid = -1;
	int sock = -1, err = -1; // supervisor ends: the rendezvous socket, the read end of the worker's stderr
	std::string line;        // stderr bytes after the last newline
	bool running = false, sent_handle = false;
};

void write_all(int fd, const char* p, size_t n) {
	while (n) {
		const ssize_t w = write(fd, p, n);
		if (w < 0 && errno == EINTR) continue;
		if (w <= 0) return;
		p += w;
		n -= (size_t) w;
	}
}

// Moves what the worker's stderr holds to ours, one "rank r: " prefix per line; at EOF (or flush) the tail too.
void pump_stderr(Worker& w, int r, bool flush) {
	char buf[4096];
	for (;;) {
		const ssize_t k = w.err >= 0 ? read(w.err, buf, sizeof buf) : 0;
		if (k < 0 && errno == EINTR) continue;
		if (k > 0) w.line.append(buf, (size_t) k);
		size_t nl;
		while ((nl = w.line.find('\n')) != std::string::npos) {
			const std::string out = "rank " + std::to_string(r) + ": " + w.line.substr(0, nl + 1);
			write_all(2, out.data(), out.size());
			w.line.erase(0, nl + 1);
		}
		if (k > 0) continue;
		if (k == 0 && w.err >= 0) { close(w.err); w.err = -1; } // EOF: the worker and everything it forked are done with it
		if ((k == 0 || flush) && !w.line.empty()) {
			const std::string out = "rank " + std::to_string(r) + ": " + w.line + "\n";
			write_all(2, out.data(), out.size());
			w.line.clear();
		}
		return; // EOF, or nothing more to read now (EAGAIN)
	}
}

} // namespace

int run_tp_ranks(const int P, const std::function<int(const TpRank&)>& fn) {
	fflush(stdout);
	fflush(stderr);
	const pid_t supervisor = getpid();
	std::vector<Worker> w((size_t) P);
	bool failed = false;
	for (int r = 0; r < P && !failed; r++) {
		int sv[2], pe[2];
		if (socketpair(AF_UNIX, SOCK_SEQPACKET, 0, sv) != 0) { perror("socketpair"); failed = true; break; }
		if (pipe(pe) != 0) { perror("pipe"); close(sv[0]); close(sv[1]); failed = true; break; }
		const pid_t pid = fork();
		if (pid < 0) { perror("fork"); close(sv[0]); close(sv[1]); close(pe[0]); close(pe[1]); failed = true; break; }
		if (pid == 0) {
			prctl(PR_SET_PDEATHSIG, SIGKILL);
			if (getppid() != supervisor) _exit(1); // the supervisor died before prctl took effect
			for (int j = 0; j < r; j++) { close(w[j].sock); close(w[j].err); } // the earlier workers' supervisor ends
			close(sv[0]);
			close(pe[0]);
			dup2(pe[1], 2);
			close(pe[1]);
			if (r > 0) {
				const int null = open("/dev/null", O_WRONLY);
				if (null >= 0) { dup2(null, 1); close(null); }
			}
			worker(r, P, sv[1], fn);
		}
		close(sv[1]);
		close(pe[1]);
		fcntl(pe[0], F_SETFL, fcntl(pe[0], F_GETFL) | O_NONBLOCK);
		w[r].pid = pid;
		w[r].sock = sv[0];
		w[r].err = pe[0];
		w[r].running = true;
	}

	std::vector<uint8_t> table((size_t) P * XALM_IPC_HANDLE_BYTES);
	int handles = 0, running = 0;
	bool have_id = false;
	for (const Worker& x : w) running += x.running;
	while (!failed && running > 0) {
		std::vector<pollfd> fds;
		std::vector<std::pair<int, bool>> who; // (rank, is the socket)
		for (int r = 0; r < P; r++) {
			if (w[r].sock >= 0) { fds.push_back({w[r].sock, POLLIN, 0}); who.push_back({r, true}); }
			if (w[r].err >= 0) { fds.push_back({w[r].err, POLLIN, 0}); who.push_back({r, false}); }
		}
		// the timeout bounds how late a worker's exit is noticed when it left its descriptors to a child of its own
		if (poll(fds.data(), fds.size(), 100) < 0 && errno != EINTR) { perror("poll"); failed = true; break; }
		for (size_t i = 0; i < fds.size(); i++) {
			if (!fds[i].revents) continue;
			Worker& x = w[(size_t) who[i].first];
			const int r = who[i].first;
			if (!who[i].second) { pump_stderr(x, r, false); continue; }
			unsigned char msg[XALM_COMM_ID_BYTES];
			const ssize_t k = recv(x.sock, msg, sizeof msg, MSG_DONTWAIT | MSG_TRUNC);
			if (k < 0 && (errno == EAGAIN || errno == EINTR)) continue;
			if (k <= 0) { close(x.sock); x.sock = -1; continue; } // the worker exited: its status decides
			if (r == 0 && !have_id && k == XALM_COMM_ID_BYTES) {
				have_id = true;
				for (Worker& y : w)
					if (y.sock >= 0) send_msg(y.sock, msg, (size_t) k);
			} else if (have_id && !x.sent_handle && k == XALM_IPC_HANDLE_BYTES) {
				x.sent_handle = true;
				std::memcpy(table.data() + (size_t) r * XALM_IPC_HANDLE_BYTES, msg, XALM_IPC_HANDLE_BYTES);
				if (++handles == P)
					for (Worker& y : w)
						if (y.sock >= 0) send_msg(y.sock, table.data(), table.size());
			} else {
				fprintf(stderr, "rank %d: unexpected %zd-byte rendezvous message\n", r, k);
				failed = true;
			}
		}
		for (int r = 0; r < P; r++) {
			int st = 0;
			if (!w[r].running || waitpid(w[r].pid, &st, WNOHANG) != w[r].pid) continue;
			w[r].running = false;
			running--;
			if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) {
				failed = true;
				if (WIFSIGNALED(st)) fprintf(stderr, "rank %d: killed by signal %d\n", r, WTERMSIG(st));
			}
		}
	}
	// On a failure the other ranks may be blocked in a collective that will never complete: kill them.
	for (Worker& x : w)
		if (x.running) kill(x.pid, SIGKILL);
	for (int r = 0; r < P; r++) {
		if (w[r].running) {
			while (waitpid(w[r].pid, nullptr, 0) < 0 && errno == EINTR) {}
			w[r].running = false;
		}
		pump_stderr(w[r], r, true);
		if (w[r].err >= 0) close(w[r].err);
		if (w[r].sock >= 0) close(w[r].sock);
	}
	return failed ? 1 : 0;
}
