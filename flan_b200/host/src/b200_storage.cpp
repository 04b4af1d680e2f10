// Device mirror, recycled host vectors and the process-wide engine context of the B200 build (see flan/b200_storage.h).
#include "flan/b200_storage.h"
#include "flan/defines.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <map>
#include <mutex>

#include "flan_b200.h"

namespace flan::b200 {

namespace {

// The process-wide engine: one device, or every visible one behind a multi handle whose device 0 is the primary context.
struct Engine { flan_b200_ctx * ctx = nullptr; flan_b200_multi * multi = nullptr; };

Engine & engine()
	{
	static std::once_flag once;
	static Engine e;
	std::call_once( once, []
		{
		const char * one = std::getenv( "FLAN_B200_DEVICE" );
		const char * many = std::getenv( "FLAN_B200_DEVICES" );
		if( !one && ( many || flan_b200_device_count() > 1 ) )
			{
			std::vector<int> ids;
			if( many )
				for( const char * p = many; *p; )
					{
					char * end = nullptr;
					const long v = std::strtol( p, &end, 10 );
					if( end == p ) break;
					ids.push_back( int( v ) );
					p = ( *end == ',' ) ? end + 1 : end;
					}
			if( flan_b200_multi_create( ids.empty() ? nullptr : ids.data(), int( ids.size() ), &e.multi ) == FLAN_B200_OK )
				{
				e.ctx = flan_b200_multi_ctx( e.multi, 0 );
				if( flan_b200_multi_device_count( e.multi ) < 2 ) { /* one device after all: keep the handle for its context only */ }
				return;
				}
			std::cout << "flan_b200: cannot create the multi-GPU engine (" << flan_b200_multi_last_error( nullptr ) << "), using one device" << std::endl;
			e.multi = nullptr;
			}
		const int device = one ? std::atoi( one ) : 0;
		if( flan_b200_create( device, &e.ctx ) != FLAN_B200_OK )
			{
			std::cout << "flan_b200: cannot create the GPU engine: " << flan_b200_last_error( nullptr ) << std::endl;
			e.ctx = nullptr;
			}
		} );
	return e;
	}

}

flan_b200_ctx * context() { return engine().ctx; }

// For tools and bench.py: the process-wide engine of the C++ layer, reachable from C (per-kernel timing, launch counts).
extern "C" flan_b200_ctx * flan_b200_host_context( void ) { return engine().ctx; }

flan_b200_multi * multi()
	{
	Engine & e = engine();
	return ( e.multi && flan_b200_multi_device_count( e.multi ) > 1 ) ? e.multi : nullptr;
	}

struct ShardedStore
	{
	flan_b200_sharded_pv desc{};
	bool summaries = false;
	~ShardedStore() { if( flan_b200_multi * m = engine().multi ) flan_b200_multi_free_pv( m, &desc ); }
	};

std::shared_ptr<ShardedStore> new_sharded_store() { return std::make_shared<ShardedStore>(); }
void * sharded_descriptor( ShardedStore & s ) { return &s.desc; }
void set_sharded_summaries( ShardedStore & s ) { s.summaries = true; }
bool sharded_summaries( const ShardedStore & s ) { return s.summaries; }

namespace {

void complain( flan_b200_ctx * ctx ) { std::cout << "flan_b200: " << flan_b200_last_error( ctx ) << std::endl; }

// ---- recycled host vectors -------------------------------------------------------------------------------------
constexpr size_t POOL_MIN_BYTES = size_t( 64 ) << 10;       // smaller vectors are cheaper to allocate than to look up
constexpr size_t POOL_MAX_ENTRY = size_t( 2 ) << 30;
constexpr size_t POOL_BUDGET    = size_t( 6 ) << 30;        // bytes parked in the pool at most (oldest leave first)
constexpr size_t PIN_MIN_BYTES  = size_t( 1 ) << 20;
constexpr int    PIN_AFTER_USES = 2;                        // page-lock a vector the second time it comes back

std::mutex g_pool_mutex;
size_t g_pool_bytes = 0;
uint64_t g_pool_clock = 0;
std::map<const void *, int> g_uses;                          // by storage address: how often a vector has been recycled

template<typename T> struct HostPool
	{
	struct Entry { std::vector<T> v; bool pinned; uint64_t stamp; };
	std::vector<Entry> entries;
	static HostPool & get() { static HostPool * p = new HostPool; return *p; }      // never destroyed: outlives the CUDA runtime's own teardown
	};

void unpin( const void * p )
	{
	if( flan_b200_ctx * ctx = context() ) flan_b200_host_unregister( ctx, const_cast<void *>( p ) );
	}

template<typename T> void evict_over_budget()      // g_pool_mutex held
	{
	auto & e = HostPool<T>::get().entries;
	while( g_pool_bytes > POOL_BUDGET && !e.empty() )
		{
		auto oldest = std::min_element( e.begin(), e.end(), []( const auto & a, const auto & b ) { return a.stamp < b.stamp; } );
		g_pool_bytes -= sizeof( T ) * oldest->v.size();
		if( oldest->pinned ) unpin( oldest->v.data() );
		g_uses.erase( oldest->v.data() );
		e.erase( oldest );
		}
	}

}

template<typename T> std::vector<T> pool_take( size_t count, bool zeroed, bool * pinned, bool only_if_pooled )
	{
	*pinned = false;
	const size_t bytes = sizeof( T ) * count;
	std::vector<T> v;
	int uses = 0;
	bool found = false;
	if( bytes >= POOL_MIN_BYTES )
		{
		std::lock_guard<std::mutex> lock( g_pool_mutex );
		auto & e = HostPool<T>::get().entries;
		for( size_t i = 0; i < e.size(); ++i )
			if( e[i].v.size() == count && ( !only_if_pooled || e[i].pinned || g_uses[e[i].v.data()] >= PIN_AFTER_USES ) )
				{
				v = std::move( e[i].v ); *pinned = e[i].pinned;
				e.erase( e.begin() + i );
				g_pool_bytes -= bytes;
				uses = g_uses[v.data()];
				found = true;
				break;
				}
		}
	if( !found )
		{
		if( only_if_pooled ) return v;
		return std::vector<T>( count );             // value-initialised, like the reference's buffers
		}
	if( !*pinned && uses >= PIN_AFTER_USES && bytes >= PIN_MIN_BYTES )
		if( flan_b200_ctx * ctx = context() )
			*pinned = flan_b200_host_register( ctx, v.data(), bytes ) == FLAN_B200_OK;
	if( zeroed ) std::memset( static_cast<void *>( v.data() ), 0, bytes );
	return v;
	}

template<typename T> void pool_give( std::vector<T> && v, bool pinned )
	{
	const size_t bytes = sizeof( T ) * v.size();
	if( bytes < POOL_MIN_BYTES || bytes > POOL_MAX_ENTRY )
		{
		if( pinned ) unpin( v.data() );
		return;
		}
	std::lock_guard<std::mutex> lock( g_pool_mutex );
	++g_uses[v.data()];
	HostPool<T>::get().entries.push_back( { std::move( v ), pinned, ++g_pool_clock } );
	g_pool_bytes += bytes;
	evict_over_budget<T>();
	}

// ---- Mirror ----------------------------------------------------------------------------------------------------
template<typename T>
struct Mirror<T>::DeviceMem
	{
	void * ptr = nullptr;
	~DeviceMem() { if( ptr && context() ) flan_b200_free( context(), ptr ); }      // back to the engine's block cache
	};

template<typename T>
Mirror<T>::Mirror( size_t count ) : count_( count )
	{
	host_ = pool_take<T>( count, true, &host_pinned_ );
	pinned_ptr_ = host_pinned_ ? host_.data() : nullptr;
	}

template<typename T>
void Mirror<T>::take( Mirror & o )
	{
	host_ = std::move( o.host_ ); count_ = o.count_; dev_ = std::move( o.dev_ ); shards_ = std::move( o.shards_ );
	host_valid_ = o.host_valid_.load(); device_valid_ = o.device_valid_.load();
	host_pinned_ = o.host_pinned_; pinned_ptr_ = o.pinned_ptr_;
	download_in_flight_ = o.download_in_flight_; upload_in_flight_ = o.upload_in_flight_;
	uploads_ = o.uploads_; nan_flag_ = o.nan_flag_; produced_on_device_ = o.produced_on_device_; o.produced_on_device_ = false;
	o.host_.clear(); o.count_ = 0; o.host_valid_ = true; o.device_valid_ = false;
	o.host_pinned_ = false; o.pinned_ptr_ = nullptr; o.download_in_flight_ = o.upload_in_flight_ = false; o.uploads_ = 0; o.nan_flag_ = nullptr;
	}

template<typename T>
void Mirror<T>::release()
	{
	flan_b200_ctx * ctx = nullptr;
	if( ( download_in_flight_ || upload_in_flight_ ) && dev_ && ( ctx = context() ) )
		flan_b200_wait_copies( ctx, dev_->ptr );          // no copy may still be touching host_ when it goes back to the pool
	download_in_flight_ = upload_in_flight_ = false;
	const bool still_pinned = host_pinned_ && host_.data() == pinned_ptr_;
	if( host_pinned_ && !still_pinned ) unpin( pinned_ptr_ );         // the user reallocated the vector: its old storage is gone
	if( !host_.empty() && host_.size() == count_ ) pool_give( std::move( host_ ), still_pinned );
	else if( still_pinned ) unpin( pinned_ptr_ );
	host_ = std::vector<T>();
	host_pinned_ = false; pinned_ptr_ = nullptr;
	dev_.reset();
	shards_.reset();
	count_ = 0; host_valid_ = true; device_valid_ = false; uploads_ = 0; nan_flag_ = nullptr; produced_on_device_ = false;
	}

template<typename T>
std::vector<T> & Mirror<T>::host_mut()
	{
	if( !host_valid_.load( std::memory_order_acquire ) ) sync_to_host();
	std::lock_guard<std::mutex> lock( lazy_ );
	if( upload_in_flight_ && dev_ )
		{
		// an asynchronous upload may still be reading the vector the caller is about to write
		if( flan_b200_ctx * ctx = context() ) flan_b200_wait_copies( ctx, dev_->ptr );
		upload_in_flight_ = false;
		}
	device_valid_ = false;
	shards_.reset();
	return host_;
	}

template<typename T>
void Mirror<T>::maybe_pin_host() const
	{
	if( host_pinned_ && host_.data() != pinned_ptr_ )       // reallocated by the user since
		{
		unpin( pinned_ptr_ );
		host_pinned_ = false; pinned_ptr_ = nullptr;
		}
	const size_t bytes = sizeof( T ) * count_;
	if( host_pinned_ || uploads_ < PIN_AFTER_USES || bytes < PIN_MIN_BYTES ) return;
	flan_b200_ctx * ctx = context();
	if( ctx && flan_b200_host_register( ctx, host_.data(), bytes ) == FLAN_B200_OK )
		{
		host_pinned_ = true;
		pinned_ptr_ = host_.data();
		}
	}

template<typename T>
const T * Mirror<T>::device_with( const std::function<int( const T * h, T * d )> * uploader, bool * uploaded ) const
	{
	if( uploaded ) *uploaded = false;
	flan_b200_ctx * ctx = context();
	if( !ctx ) return nullptr;
	std::lock_guard<std::mutex> lock( lazy_ );
	if( device_valid_ && dev_ ) return static_cast<const T *>( dev_->ptr );
	if( !dev_ )
		{
		auto mem = std::make_shared<DeviceMem>();
		if( flan_b200_malloc( ctx, sizeof( T ) * count_, &mem->ptr ) != FLAN_B200_OK ) { complain( ctx ); return nullptr; }
		dev_ = mem;
		}
	if( shards_ )
		{
		// a single-device consumer (a PV-domain method): the shards are gathered onto device 0, device to device
		flan_b200_multi * m = multi();
		if( !m || flan_b200_multi_gather_pv( m, &shards_->desc, nullptr, 0, static_cast<float *>( dev_->ptr ) ) != FLAN_B200_OK )
			{
			std::cout << "flan_b200: " << flan_b200_multi_last_error( m ) << std::endl;
			return nullptr;
			}
		shards_.reset();           // freed on their devices' streams, after the copies above
		device_valid_ = true;
		return static_cast<const T *>( dev_->ptr );
		}
	if( count_ )
		{
		if( host_.size() < count_ )
			{
			std::cout << "flan_b200: a buffer's host vector was shrunk below its format's size" << std::endl;
			return nullptr;
			}
		maybe_pin_host();
		++uploads_;
		T * d = static_cast<T *>( dev_->ptr );
		const int rc = uploader ? ( *uploader )( host_.data(), d ) : flan_b200_upload( ctx, d, host_.data(), sizeof( T ) * count_ );
		if( rc != FLAN_B200_OK ) { if( !uploader ) complain( ctx ); return nullptr; }      // an uploader's caller reports its own failure
		if( uploaded ) *uploaded = uploader != nullptr;
		upload_in_flight_ = true;      // asynchronous when host_ is page-locked; kernels on the block are ordered after it by the engine
		}
	device_valid_ = true;
	return static_cast<const T *>( dev_->ptr );
	}

template<typename T>
Mirror<T> Mirror<T>::device_result( size_t count, T ** d_out, T ** h_prefetch )
	{
	Mirror<T> m;
	*d_out = nullptr;
	if( h_prefetch ) *h_prefetch = nullptr;
	flan_b200_ctx * ctx = context();
	if( !ctx ) return m;
	auto mem = std::make_shared<DeviceMem>();
	if( flan_b200_malloc( ctx, sizeof( T ) * count, &mem->ptr ) != FLAN_B200_OK ) { complain( ctx ); return m; }
	m.dev_ = mem;
	m.count_ = count;
	m.host_valid_ = false;
	m.device_valid_ = true;
	m.produced_on_device_ = true;
	*d_out = static_cast<T *>( mem->ptr );
	if( h_prefetch && count )
		{
		// only a recycled, page-locked vector: the producer's copy into it is then asynchronous and costs the caller nothing
		bool pinned = false;
		std::vector<T> v = pool_take<T>( count, false, &pinned, true );
		if( v.size() == count && pinned )
			{
			m.host_ = std::move( v );
			m.host_pinned_ = true; m.pinned_ptr_ = m.host_.data();
			m.download_in_flight_ = true;
			*h_prefetch = m.host_.data();
			}
		else if( v.size() == count ) pool_give( std::move( v ), pinned );
		}
	return m;
	}

template<typename T>
Mirror<T> Mirror<T>::adopt_host( std::vector<T> && v, bool pinned )
	{
	Mirror<T> m;
	m.count_ = v.size();
	m.host_ = std::move( v );
	m.host_pinned_ = pinned; m.pinned_ptr_ = pinned ? m.host_.data() : nullptr;
	return m;
	}

template<typename T>
Mirror<T> Mirror<T>::from_shards( size_t count, std::shared_ptr<ShardedStore> shards )
	{
	Mirror<T> m;
	m.count_ = count;
	m.shards_ = std::move( shards );
	m.host_valid_ = false;
	m.device_valid_ = false;
	return m;
	}

template<typename T>
void Mirror<T>::sync_to_host() const
	{
	std::lock_guard<std::mutex> lock( lazy_ );
	if( host_valid_ ) return;
	flan_b200_ctx * ctx = context();
	if( shards_ && !device_valid_ )
		{
		// frame-range shards on several devices: every device copies its rows into the host vector
		if( host_.size() != count_ )
			{
			host_ = pool_take<T>( count_, false, &host_pinned_ );
			pinned_ptr_ = host_pinned_ ? host_.data() : nullptr;
			}
		flan_b200_multi * m = multi();
		if( !m || flan_b200_multi_gather_pv( m, &shards_->desc, reinterpret_cast<float *>( host_.data() ), 0, nullptr ) != FLAN_B200_OK )
			std::cout << "flan_b200: " << flan_b200_multi_last_error( m ) << std::endl;
		host_valid_.store( true, std::memory_order_release );
		return;
		}
	if( download_in_flight_ )
		{
		if( ctx && dev_ && flan_b200_wait_copies( ctx, dev_->ptr ) != FLAN_B200_OK ) complain( ctx );
		download_in_flight_ = false;
		}
	else
		{
		if( host_.size() != count_ )
			{
			host_ = pool_take<T>( count_, false, &host_pinned_ );
			pinned_ptr_ = host_pinned_ ? host_.data() : nullptr;
			}
		if( ctx && dev_ && count_ )
			{
			if( flan_b200_download( ctx, host_.data(), dev_->ptr, sizeof( T ) * count_ ) != FLAN_B200_OK
			 || flan_b200_wait_copies( ctx, dev_->ptr ) != FLAN_B200_OK )
				complain( ctx );
			}
		}
	if( nan_flag_ )
		{
		if( *nan_flag_ )       // AudioPV.cpp:88-89: warn and carry on
			std::cout << "flan::convert_to_audio recieved a nan or infinite value. This often happens when dividing by zero in an earlier algorithm.";
		nan_flag_ = nullptr;
		}
	host_valid_.store( true, std::memory_order_release );
	}

template<typename T>
Mirror<T> Mirror<T>::deep_copy() const
	{
	Mirror<T> m;
	const std::vector<T> & h = host();         // downloads if needed; plain host copy, device copy rebuilt on demand
	m.host_ = pool_take<T>( count_, false, &m.host_pinned_ );
	m.pinned_ptr_ = m.host_pinned_ ? m.host_.data() : nullptr;
	std::copy( h.begin(), h.begin() + std::min( h.size(), m.host_.size() ), m.host_.begin() );
	m.count_ = count_;
	return m;
	}

template class Mirror<float>;
template class Mirror<MF>;

}
